# TortoiseB200.jl -- Julia host side of libtortoise_b200.so (B200-native batched Monte-Carlo engine).
#
# Drop-in for the data-parallel hot path of RoboticExplorationLab/TortoiseSat.jl: every function
# below keeps the NAME and ARGUMENT MEANING of the reference function it replaces (file:line cited)
# and forwards to the C ABI declared in include/tortoise_b200.h through `ccall`.  Scalar calls are
# batch-of-1 (correctness path); the `*_batch` / `monte_carlo` entry points are the performance path.
#
# NOTE: this image has no Julia toolchain, so this file is NOT executed by the test-suite; the
# identical C ABI is exercised from Python ctypes (tortoisesat.jl_b200/host.py).  Array layout: Julia
# is column-major, the library is "row-major by sample" => a field table is passed as a 3 x rows
# Matrix{Float64}, a trajectory as 8 x N, so no transposition or copy is needed.
module TortoiseB200

using LinearAlgebra

const LIB = get(ENV, "TORTOISE_B200_LIB", joinpath(@__DIR__, "..", "tortoisesat.jl_b200", "libtortoise_b200.so"))

# ----------------------------------------------------------------------------- context
mutable struct Engine
    h::Ptr{Cvoid}
end
function Engine(device::Integer = 0)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:ts_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), r, device)
    rc == 0 || error("ts_create failed ($rc): no usable CUDA device (there is no CPU fallback)")
    e = Engine(r[])
    finalizer(x -> ccall((:ts_destroy, LIB), Cvoid, (Ptr{Cvoid},), x.h), e)
    e
end
const _default = Ref{Union{Nothing,Engine}}(nothing)
engine() = (_default[] === nothing && (_default[] = Engine(0)); _default[])
lasterr(e::Engine) = unsafe_string(ccall((:ts_last_error, LIB), Cstring, (Ptr{Cvoid},), e.h))
check(e::Engine, rc) = rc == 0 ? nothing : error("tortoise_b200 error $rc: $(lasterr(e))")

# ----------------------------------------------------------------------------- structs of the C ABI
struct FieldOpts            # ts_field_opts
    GM::Float64; mjd::Float64; igrf_date::Float64; field_radius_m::Float64; t0::Float64; tf::Float64; N::Int64
end
struct IlqrOpts             # ts_ilqr_opts
    max_outer::Int32; max_inner::Int32; max_linesearch::Int32; dJ_counter_limit::Int32; stage_cost_dt::Int32; goal_mask::Int32
    cost_tol::Float64; cost_tol_intermediate::Float64; grad_tol::Float64; grad_tol_intermediate::Float64; constraint_tol::Float64
    penalty_initial::Float64; penalty_scaling::Float64; penalty_max::Float64; dual_max::Float64
    ls_lower::Float64; ls_upper::Float64; bp_reg_increase::Float64; bp_reg_max::Float64; bp_reg_min::Float64; bp_reg_fp::Float64
    max_cost_value::Float64; max_state_value::Float64; max_control_value::Float64; u_max::Float64; u_min::Float64
    # SURVEY App. C assumption registry (0 = frozen default, 1 = the named alternative)
    a2_active_ge::Int32; a3_grad_over_N::Int32; a4_no_intermediate::Int32; a5_dual_active_only::Int32
    a6_penalty_conditional::Int32; a7_carry_cost::Int32; constraint_decrease_ratio::Float64
    # launch scheme of K3
    k3_suspend_after::Int32; k3_tail_share::Int32; k3_early_factor::Float64; k3_pair::Int32; k3_wide_occ::Int32
    quat_error::Int32; k3_generic_inertia::Int32     # 1: quaternion_error / quaternion_expansion variant (monte_carlo.jl:158,192)
end
struct TrialOutcome         # ts_trial_outcome (64 bytes)
    status::Int32; outer_iters::Int32; inner_iters::Int32; ls_rollouts::Int32; N::Int64
    J::Float64; c_max::Float64; t_final::Float64; slew_time::Float64; flops::Float64
end
struct AlState              # ts_al_state (104 bytes): exported AL-iLQR solver state of one trial (CS1-CS4, DESIGN.md section 4)
    mu::Float64; lam_goal::NTuple{8,Float64}; J::Float64; c_max::Float64
    status::Int32; outer_iters::Int32; inner_iters::Int32; ls_rollouts::Int32
end
struct TvlqrOpts            # ts_tvlqr_opts
    dt::Float64; t0::Float64; tf::Float64
    Qd::NTuple{6,Float64}; Qfd::NTuple{6,Float64}; Rd::NTuple{3,Float64}
    dt_squared::Int32; noise_mode::Int32; seed::UInt64
    w_limit::Float64; ang_limit::Float64; literal_postproc::Int32; pad_::Int32
end
struct McConfig             # ts_mc_config
    n_trials::Int64; shared_orbit::Int32; run_tvlqr::Int32; t0::Float64; tf::Float64; N_scope::Int64
    cutoff::Float64; dt::Float64; alpha::Float64; beta::Float64; eigen_axis_fix::Int32; keep_trajectories::Int32
    ilqr::IlqrOpts; tvlqr::TvlqrOpts
end
struct McStats              # ts_mc_stats
    n_trials::Int64; n_converged::Int64; n_no_cutoff::Int64; n_fail_slew::Int64
    sum_slew_time::Float64; sum_slew_time_sq::Float64; sum_t_final::Float64; sum_inner_iters::Float64
    sum_ls_rollouts::Float64; sum_knots::Float64; flops::Float64
    ms_field::Float64; ms_prep::Float64; ms_solve::Float64; ms_tvlqr::Float64
    n_status::NTuple{6,Int64}          # trials per TS_ST_* code
end
struct ReplayEnsembleOpts   # ts_replay_ensemble_opts
    n_real::Int64; r_first::Int64; q_noise_scale::Float64
end
function default_ilqr_opts()
    r = Ref{IlqrOpts}()
    ccall((:ts_ilqr_default_opts, LIB), Cvoid, (Ref{IlqrOpts},), r); r[]
end
function default_tvlqr_opts()
    r = Ref{TvlqrOpts}()
    ccall((:ts_tvlqr_default_opts, LIB), Cvoid, (Ref{TvlqrOpts},), r); r[]
end

# ----------------------------------------------------------------------------- L0 parameters
# struct params / input_parameters(type,Kep,MJD)            reference src/input_parameters.jl:4-16,24-66
struct params
    type::AbstractString; mass::Float64; J::Array{Float64}; BC::Float64; alt::Float64; Kep::Array{Float64}
    MJD::Float64; GM::Float64; R_E::Float64; T::Float64; ω_0::Float64
end
function input_parameters(type, Kep, MJD)
    GM = 3.986004418E14 * (1 / 1000)^3
    R_E = 6371.0
    if type == "1U"
        mass = .75; J = [0.00125 0 0; 0 0.00125 0; 0 0 0.00125]
    elseif type == "1P"
        mass = .25; J = [0.0001041667 0 0; 0 0.0001041667 0; 0 0 0.0001041667]
    elseif type == "3U"
        mass = 2.5; J = [0.020833 0 0; 0 0.020833 0; 0 0 0.0041666]
    else
        error("Type not recognized")
    end
    BC = mass / 2.2 / (J[1, 1] * J[2, 2])
    alt = 400                      # quirk Q10: forced (input_parameters.jl:58)
    T = 2 * pi * sqrt(Kep[2] .^ 3 / GM)
    ω_0 = sqrt(GM / Kep[2]^3)
    MJD = 58155.0                  # quirk Q10: forced (input_parameters.jl:63)
    params(type, mass, J, BC, alt, vec(collect(Float64, Kep)), MJD, GM, R_E, T, ω_0)
end

# ----------------------------------------------------------------------------- K1: IGRF
# igrf12(date, r, λ, Ω)                                     reference src/igrf.jl:67-274
function igrf12_batch(date::Real, r::Vector{Float64}, λ::Vector{Float64}, Ω::Vector{Float64}; e::Engine = engine())
    n = length(r)
    Bn = Vector{Float64}(undef, n); Be = similar(Bn); Bd = similar(Bn)
    rc = ccall((:ts_igrf12_batch, LIB), Cint,
               (Ptr{Cvoid}, Cdouble, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
               e.h, date, n, r, λ, Ω, Bn, Be, Bd, 0)
    check(e, rc)
    Bn, Be, Bd
end
function igrf12(date::Number, r::Number, λ::Number, Ω::Number; show_warns = true)
    show_warns && (date > 2020) &&
        @warn("The magnetic field computed with this IGRF version may be of reduced accuracy for years greater than 2020.")
    Bn, Be, Bd = igrf12_batch(date, [Float64(r)], [Float64(λ)], [Float64(Ω)])
    [Bn[1]; Be[1]; Bd[1]]
end
# igrf_data(altitude, year): the 1000 x 1000 x 3 map       reference src/magnetic_toolbox.jl:108-127
# Returned behind the reference's call shape mag_field(i,j,c) (monte_carlo.jl:90-96).  The reference wraps the array in
# a cubic B-spline interpolant with periodic extrapolation but evaluates it at integer nodes only, where an
# interpolating spline returns the data: node values + periodic index wrap; non-integer arguments are rejected.
struct MagFieldMap
    grid::Array{Float64,3}
end
function (m::MagFieldMap)(i, j, c)
    (isinteger(i) && isinteger(j) && isinteger(c)) || error("mag_field(i,j,c): only integer grid nodes are supported")
    n0, n1, n2 = size(m.grid)
    m.grid[mod(Int(i) - 1, n0) + 1, mod(Int(j) - 1, n1) + 1, mod(Int(c) - 1, n2) + 1]
end
Base.size(m::MagFieldMap) = size(m.grid)
Base.getindex(m::MagFieldMap, I...) = getindex(m.grid, I...)
function igrf_data(altitude, year::Int64)
    R_E = 6378; N = 1000
    lat = collect(range(-π / 2, length = N, π / 2)); long = collect(range(-π, length = N, π))
    LA = repeat(lat, inner = N); LO = repeat(long, outer = N)
    Bn, Be, Bd = igrf12_batch(year, fill((altitude + R_E) * 1000.0, N * N), LA, LO)
    mag_field = zeros(N, N, 3)
    for i = 1:N, j = 1:N
        k = (i - 1) * N + j
        mag_field[i, j, :] = [Bn[k], Be[k], Bd[k]] / 1.e9
    end
    MagFieldMap(mag_field)
end
# igrf_interpolant(altitude, year): the cubic B-spline of that map   reference src/magnetic_toolbox.jl:124-125
# extrapolate(interpolate(A, BSpline(Cubic(Reflect(OnCell())))), Periodic()) under rules FM1..FM4 (DESIGN.md section 4,
# K8): real i, j (periodic), integer c (period 3).  coefs is the 3 x (n1+2) x (n0+2) Julia array whose memory is the
# row-major (n0+2) x (n1+2) x 3 coefficient array of ts_field_map_prefilter.  Each call copies it to the GPU, so
# evaluate many points per field_map_eval call.
struct MagFieldInterpolant
    coefs::Array{Float64,3}
    n0::Int64
    n1::Int64
    e::Engine
end
function field_map_prefilter(grid::Array{Float64,3}; e::Engine = engine())
    n0, n1, _ = size(grid)
    g = permutedims(grid, (3, 2, 1))            # n0 x n1 x 3 (Julia) -> row-major n0 x n1 x 3 (C)
    C = Array{Float64}(undef, 3, n1 + 2, n0 + 2)
    rc = ccall((:ts_field_map_prefilter, LIB), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Cint),
               e.h, n0, n1, g, C, 0)
    check(e, rc)
    MagFieldInterpolant(C, n0, n1, e)
end
# the spline at the 1-based indices (i[p], j[p]) -> 3 x n (north, east, down)
function field_map_eval(m::MagFieldInterpolant, i::Vector{Float64}, j::Vector{Float64})
    n = length(i)
    length(j) == n || error("field_map_eval: i and j must have the same length")
    out = Matrix{Float64}(undef, 3, n)
    rc = ccall((:ts_field_map_eval_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
               m.e.h, m.n0, m.n1, m.coefs, n, i, j, out, 0)
    check(m.e, rc)
    out
end
function (m::MagFieldInterpolant)(i, j, c)
    isinteger(c) || error("mag_field(i,j,c): the component index c must be an integer")
    field_map_eval(m, [Float64(i)], [Float64(j)])[mod(Int(c) - 1, 3) + 1, 1]
end
igrf_interpolant(altitude, year::Int64; e::Engine = engine()) = field_map_prefilter(igrf_data(altitude, year).grid; e = e)

# ----------------------------------------------------------------------------- K2: orbit + field table
# magnetic_simulation(p,t0,tf,N,mag_field)                  reference src/magnetic_toolbox.jl:33-106
function magnetic_simulation(p::params, t0, tf, N, mag_field = nothing; alt = p.alt, igrf_date = 2019.0, e::Engine = engine())
    N = Int(N)
    fo = [FieldOpts(p.GM, p.MJD, igrf_date, (alt + p.R_E) * 1000.0, t0, tf, N)]
    offs = Int64[0, 2N]
    B = zeros(3, 2N); pos = zeros(3, 2N + 1); vel = zeros(3, 2N + 1)
    rc = ccall((:ts_magnetic_simulation_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{FieldOpts}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
               e.h, 1, p.Kep, fo, offs, C_NULL, B, pos, vel, 0)
    check(e, rc)
    Matrix(B'), pos, vel        # B_N_sim is (2N x 3) in the reference
end
# legacy 7-argument form used at src/monte_carlo.jl:134,149
magnetic_simulation(A::AbstractVector, t0, tf, N, mag_field, GM, MJD_0; alt = 400, R_E = 6371.0) =
    magnetic_simulation(params("", 0.0, zeros(3, 3), 0.0, alt, collect(Float64, A), MJD_0, GM, R_E, 0.0, 0.0), t0, tf, N, mag_field)

# magnetic_gramian(B_N,dt) -> 3 x 3 x rows                 reference src/magnetic_toolbox.jl:1-12
function magnetic_gramian(B_N, dt; e::Engine = engine())
    rows = size(B_N, 1)
    Bt = Matrix{Float64}(B_N'); G = zeros(3, 3, rows)
    rc = ccall((:ts_magnetic_gramian_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Cint),
               e.h, 1, Bt, Int64[0], Int64[rows], Float64[dt], G, 0)
    check(e, rc)
    G                               # symmetric 3x3 blocks: row/column-major agree
end
# condition_based_time(B_gram,cutoff)                       reference src/magnetic_toolbox.jl:14-31
function condition_based_time(B_gram, cutoff; e::Engine = engine())
    rows = size(B_gram, 3); idx = Int64[0]
    rc = ccall((:ts_condition_based_time_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Int64}, Cint),
               e.h, 1, B_gram, Int64[0], Int64[rows], Float64[cutoff], idx, 0)
    check(e, rc)
    Int(idx[1])
end

# ----------------------------------------------------------------------------- slew preparation
# eigen_axis_slew(x0,xf,t) -> (ω_guess (nt x 3), q_guess (nt x 4))    reference src/eigen_axis_slew.jl:1-38
function eigen_axis_slew(x0, xf, t; e::Engine = engine())
    nt = length(t); dt = t[2] - t[1]
    Qd = zeros(8); Qfd = zeros(8); Rd = zeros(3); wg = zeros(3, nt); qg = zeros(4, nt)
    rc = ccall((:ts_slew_weights_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cdouble, Cdouble, Cdouble, Cdouble, Cint,
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
               e.h, 1, [x0[1:7]; 0.0], [xf[1:7]; 0.0], vec(Matrix(1.0I, 3, 3)), Float64[t[end]], t[1], dt, 1.0, 1.0, 0,
               Qd, Qfd, Rd, Int64[0], wg, qg)      # 0: the literal qmult(q_f, q_0) of eigen_axis_slew.jl:16
    check(e, rc)
    Matrix(wg'), Matrix(qg')
end
# Bryson's-rule weights of src/TortoiseSat.jl:157-168 (α = 10) / src/monte_carlo.jl:165-176 (α = 0.1)
function bryson_weights(x0, xf, J, t_final; t0 = 0.0, dt = 0.2, α = 1.e1, β = 1.e3, e::Engine = engine())
    Qd = zeros(8); Qfd = zeros(8); Rd = zeros(3)
    rc = ccall((:ts_slew_weights_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cdouble, Cdouble, Cdouble, Cdouble, Cint,
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
               e.h, 1, collect(Float64, x0), collect(Float64, xf), vec(Matrix{Float64}(J')), Float64[t_final], t0, dt, α, β, 0,
               Qd, Qfd, Rd, C_NULL, C_NULL, C_NULL)
    check(e, rc)
    Matrix(Diagonal(Qd)), Matrix(Diagonal(Rd)), Matrix(Diagonal(Qfd))
end

# ----------------------------------------------------------------------------- K3: AL-iLQR
# Replaces the TrajectoryOptimization.jl block of src/TortoiseSat.jl:145-146,169,178-199:
#   model_d = rk3(Model(DerivFunction,8,3)); obj = LQRObjective(Q,R,Qf,xf,N); bnd = BoundConstraint(8,3,u_max=1,u_min=-1);
#   goal = goal_constraint(xf); sat = Problem(...); solver = AugmentedLagrangianSolver(sat,opts_al); solve!(sat,solver)
# B_ECI is the (rows x 3) field table the reference keeps in a global; N_field / tf_scope are the
# globals N and tf that DerivFunction reads (src/DerivFunction.jl:28,44).
function solve_slew(x0, xf, J, Q, R, Qf, B_ECI, N::Integer, dt; N_field = N, tf_scope = 5400.0, t0 = 0.0,
                    U0 = nothing, opts::IlqrOpts = default_ilqr_opts(), e::Engine = engine())
    Bt = Matrix{Float64}(B_ECI'); X = zeros(8, N); U = zeros(3, N); K = zeros(8, 3, N)
    out = Vector{TrialOutcome}(undef, 1)
    rc = ccall((:ts_alilqr_solve_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Cdouble, Ptr{Float64},
                Ref{IlqrOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{TrialOutcome}, Cint),
               e.h, 1, Int64[N], Int64[0], collect(Float64, x0), collect(Float64, xf), vec(Matrix{Float64}(J')), diag(Q), diag(Qf),
               diag(R), Bt, Int64[0], Int64[size(Bt, 2)], Float64[N_field], Float64[1 / (tf_scope - t0)], dt,
               U0 === nothing ? C_NULL : U0, Ref(opts), X, U, K, out, 0)
    check(e, rc)
    X, U[:, 1:N-1], permutedims(K, (2, 1, 3))[:, :, 1:N-1], out[1]
end
# solve_slew that also returns the solver state and the bound multipliers (6 x N, last column zero), and continues from
# them: pass `state`, `lam` and the X, U of an earlier call to run a slew that ended at max_outer on to opts.max_outer
# (CS2, CS3).  A slew that does not continue passes through unchanged (its K is then zero).
function solve_slew(x0, xf, J, Q, R, Qf, B_ECI, N::Integer, dt, state::Union{Nothing,AlState}; N_field = N, tf_scope = 5400.0,
                    t0 = 0.0, U0 = nothing, opts::IlqrOpts = default_ilqr_opts(), lam = nothing, X_in = nothing, U_in = nothing,
                    e::Engine = engine())
    Bt = Matrix{Float64}(B_ECI'); X = zeros(8, N); U = zeros(3, N); K = zeros(8, 3, N)
    if state !== nothing
        X .= X_in; U[:, 1:N-1] .= U_in
    end
    out = Vector{TrialOutcome}(undef, 1); st_out = Vector{AlState}(undef, 1); lam_out = zeros(6, N)
    rc = ccall((:ts_alilqr_solve_state_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Cdouble, Ptr{Float64},
                Ref{IlqrOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{TrialOutcome}, Cint,
                Ptr{AlState}, Ptr{Float64}, Ptr{AlState}, Ptr{Float64}),
               e.h, 1, Int64[N], Int64[0], collect(Float64, x0), collect(Float64, xf), vec(Matrix{Float64}(J')), diag(Q), diag(Qf),
               diag(R), Bt, Int64[0], Int64[size(Bt, 2)], Float64[N_field], Float64[1 / (tf_scope - t0)], dt,
               U0 === nothing ? C_NULL : U0, Ref(opts), X, U, K, out, 0,
               state === nothing ? C_NULL : AlState[state], state === nothing ? C_NULL : Matrix{Float64}(lam), st_out, lam_out)
    check(e, rc)
    X, U[:, 1:N-1], permutedims(K, (2, 1, 3))[:, :, 1:N-1], out[1], st_out[1], lam_out
end

# ----------------------------------------------------------------------------- K4: TVLQR replay
# attitude_simulation(f!,f_gains!,integration,X_lqr,U_lqr,dt_lqr,x0_lqr,t0,tf,Q_lqr,R_lqr,Qf_lqr) -> (X_sim,U_sim,dX,K)
#                                                           reference src/attitude_controller.jl:1-48
# f!, f_gains!, integration are accepted for signature compatibility: the library implements
# simulator / gain_simulator / :rk4 (src/simulator.jl, src/gain_simulator.jl, attitude_controller.jl:122-145).
function attitude_simulation(f!, f_gains!, integration, X_lqr::Matrix, U_lqr::Matrix, dt_lqr::Float64, x0_lqr::AbstractVector,
                             t0::Float64, tf::Float64, Q_lqr, R_lqr, Qf_lqr; B_ECI, J, N_field = size(X_lqr, 2), tf_scope = 5400.0,
                             noise_mode = 2, seed = 0, q_final = [1.0, 0, 0, 0], e::Engine = engine())
    N = size(X_lqr, 2)
    o = default_tvlqr_opts()
    o = TvlqrOpts(dt_lqr, t0, tf, Tuple(diag(Q_lqr)), Tuple(diag(Qf_lqr)), Tuple(diag(R_lqr)), o.dt_squared, noise_mode, seed,
                  o.w_limit, o.ang_limit, 0, 0)
    Up = zeros(3, N); Up[:, 1:size(U_lqr, 2)] = U_lqr
    Bt = Matrix{Float64}(B_ECI')
    X_sim = zeros(8, N); U_sim = zeros(3, N); dX = zeros(6, N); K = zeros(6, 3, N); nsim = Int64[0]; slew = Float64[0]
    rc = ccall((:ts_tvlqr_sim_batch, LIB), Cint,
               (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt32}, Ref{TvlqrOpts},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Cint),
               e.h, 1, Int64[N], Int64[0], X_lqr, Up, collect(Float64, x0_lqr), vec(Matrix{Float64}(J')), Bt, Int64[0],
               Int64[size(Bt, 2)], Float64[N_field], Float64[1 / (tf_scope - t0)], Float64[tf], collect(Float64, q_final), C_NULL,
               Ref(o), C_NULL, X_sim, U_sim, dX, K, nsim, slew, 0)
    check(e, rc)
    n = nsim[1]
    X_sim[:, 1:n], U_sim[:, 1:n], dX[:, 1:n], permutedims(K, (2, 1, 3))[:, :, 1:N-1]
end

# ----------------------------------------------------------------------------- fused Monte-Carlo
# The loop of src/monte_carlo.jl:118-262 (with the solver block of src/TortoiseSat.jl:178-199) for
# number_sims trials in ONE library call.  Returns the arrays the script leaves in globals
# (src/monte_carlo.jl:52-66,237-240): A, t_final, slew_time, fails + the per-trial outcome records.
function monte_carlo(; number_sims = 100, alt = 400, R_E = 6371.0, inclination = 96.6, MJD_0 = 58155.0, igrf_date = 2019.0,
                     t0 = 0.0, tf = 60 * 40, cutoff = 30, N = 5000, J = [0.00125 0 0; 0 0.00125 0; 0 0 0.00125],
                     q_0 = [1.0; 0; 0; 0], q_final = [sqrt(2) / 2; sqrt(2) / 2; 0; 0], α = 1.e-1, β = 1.e3, seed = 0, run_tvlqr = true,
                     ilqr::IlqrOpts = default_ilqr_opts(), sat_att = false, trajectories = true, resumable = false,
                     e::Engine = engine())
    # sat_att = true: the solver configuration of monte_carlo.jl:158,192 (quaternion_error / quaternion_expansion hooks)
    # resumable = true: keep_trajectories = 2, the solver state stays on `e` for continue_monte_carlo!
    if sat_att
        ilqr = IlqrOpts((f == :quat_error ? Int32(1) : getfield(ilqr, f) for f in fieldnames(IlqrOpts))...)
    end
    GM = 3.986004418E14 * (1 / 1000)^3
    A = zeros(6, number_sims)                       # column i = A[i,:] of the reference
    fo = Vector{FieldOpts}(undef, number_sims)
    x0 = zeros(8, number_sims); xf = zeros(8, number_sims); Jm = zeros(9, number_sims); qn = zeros(3, number_sims)
    for i in 1:number_sims
        A[:, i] = [0, alt + R_E, inclination, rand() * 360, 0, rand() * 360]      # monte_carlo.jl:122-127
        fo[i] = FieldOpts(GM, MJD_0, igrf_date, (alt + R_E) * 1000.0, 0.0, 0.0, 0)
        x0[4:7, i] = q_0 === nothing ? normalize(randn(4)) : q_0          # monte_carlo.jl:108-111 uses [1,0,0,0]
        xf[4:7, i] = q_final; xf[8, i] = 1
        Jm[:, i] = vec(Matrix{Float64}(J'))
        qn[:, i] = randn(3) * (1 * pi / 180)^2                                    # monte_carlo.jl:207
    end
    tv = default_tvlqr_opts()
    tv = TvlqrOpts(0.2, t0, 0.0, ntuple(_ -> 10.0, 6), ntuple(_ -> 1000.0, 6), ntuple(_ -> 0.5e3, 3), tv.dt_squared, 2, seed,
                   0.05, 0.08727, 0, 0)                                            # monte_carlo.jl:69-71,216-226
    cfg = McConfig(number_sims, 0, run_tvlqr ? 1 : 0, t0, tf, N, cutoff, 0.2, α, β, 0, resumable ? 2 : trajectories ? 1 : 0, ilqr, tv)
    out = Vector{TrialOutcome}(undef, number_sims); st = Ref{McStats}()
    rc = ccall((:ts_monte_carlo_run, LIB), Cint,
               (Ptr{Cvoid}, Ref{McConfig}, Ptr{Float64}, Ptr{FieldOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{UInt32}, Ptr{TrialOutcome}, Ref{McStats}),
               e.h, Ref(cfg), A, fo, x0, xf, Jm, qn, C_NULL, out, st)
    check(e, rc)
    t_final = [o.t_final for o in out]; slew_time = [o.slew_time for o in out]
    fails = [o.slew_time == o.t_final ? 1.0 : 0.0 for o in out]                  # monte_carlo.jl:257-261
    res = (A = Matrix(A'), t_final = t_final, slew_time = slew_time, fails = fails, outcomes = out, stats = st[])
    resumable && (res = merge(res, (ilqr = ilqr, run_tvlqr = run_tvlqr)))
    trajectories || return res
    # the per-trial arrays the script keeps (monte_carlo.jl:52-66,149,200-201,232-233), fetched from HBM
    ko = zeros(Int64, number_sims + 1); ro = zeros(Int64, number_sims + 1)
    check(e, ccall((:ts_mc_trajectory_layout, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}), e.h, number_sims, ko, ro))
    X = zeros(8, ko[end]); U = zeros(3, ko[end]); Xs = zeros(8, ko[end]); Us = zeros(3, ko[end]); B = zeros(3, ro[end])
    check(e, ccall((:ts_mc_fetch_trajectories, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   e.h, X, U, run_tvlqr ? Xs : C_NULL, run_tvlqr ? Us : C_NULL, B))
    rng(t) = (ko[t] + 1):ko[t + 1]
    merge(res, (states = [X[:, rng(t)] for t in 1:number_sims], control_inputs = [U[:, rng(t)[1:end-1]] for t in 1:number_sims],
                sim_states = [Xs[:, rng(t)] for t in 1:number_sims], sim_control_inputs = [Us[:, rng(t)] for t in 1:number_sims],
                B_ECI_total = [Matrix(B[:, (ro[t] + 1):(ro[t] + 2 * length(rng(t)))]') for t in 1:number_sims]))
end

# The kept solver state of the last monte_carlo(...; resumable = true) on `e` (ts_mc_fetch_state): one AlState per trial
# (NO_CUTOFF: zero record with status 5) and the multipliers, 6 x (sum N) ragged like the `states` arrays.
function mc_state(number_sims::Integer; e::Engine = engine())
    ko = zeros(Int64, number_sims + 1)
    check(e, ccall((:ts_mc_trajectory_layout, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}), e.h, number_sims, ko, C_NULL))
    st = Vector{AlState}(undef, number_sims); lam = zeros(6, ko[end])
    check(e, ccall((:ts_mc_fetch_state, LIB), Cint, (Ptr{Cvoid}, Ptr{AlState}, Ptr{Float64}), e.h, st, lam))
    return st, lam
end

# ts_mc_continue: the max-outer trials of the kept run continue to ilqr.max_outer (rules MC1-MC4, DESIGN.md section 4);
# returns the outcome records of the whole ensemble and the statistics of the call.
function mc_continue(number_sims::Integer, ilqr::IlqrOpts; e::Engine = engine())
    out = Vector{TrialOutcome}(undef, number_sims); st = Ref{McStats}()
    check(e, ccall((:ts_mc_continue, LIB), Cint, (Ptr{Cvoid}, Int64, Ref{IlqrOpts}, Ptr{TrialOutcome}, Ref{McStats}),
                   e.h, number_sims, Ref(ilqr), out, st))
    return out, st[]
end

# ts_mc_replay_ensemble: the kept run's slews (last monte_carlo with trajectories or resumable on `e`) replayed under
# n_real independent disturbance draws each, realisations r_first .. r_first + n_real - 1 (rules RE1-RE5, DESIGN.md
# section 4).  trials: 1-based indices (repeats allowed; nothing = all).  Returns slew_time (n_real x n_sel) and, with
# want_x_final, x_final (8 x n_real x n_sel); a NO_CUTOFF trial gets NaN columns.
function mc_replay_ensemble(number_sims::Integer, n_real::Integer; r_first::Integer = 0, trials = nothing,
                            q_noise_scale::Float64 = (pi / 180)^2, want_x_final::Bool = false, e::Engine = engine())
    sel = trials === nothing ? C_NULL : Int64[t - 1 for t in trials]
    ns = trials === nothing ? number_sims : length(trials)
    slew = zeros(n_real, ns); xf = want_x_final ? zeros(8, n_real, ns) : nothing
    o = ReplayEnsembleOpts(n_real, r_first, q_noise_scale)
    check(e, ccall((:ts_mc_replay_ensemble, LIB), Cint,
                   (Ptr{Cvoid}, Int64, Ref{ReplayEnsembleOpts}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
                   e.h, number_sims, Ref(o), ns, sel, slew, xf === nothing ? C_NULL : xf))
    return slew, xf
end

# The slew-time distribution of a monte_carlo result's optimised slews under the disturbances: slew_time (n_real x n_sel),
# fails (slew_time == t_final), fail_rate, slew_mean / slew_std over the non-failing draws, trials (1-based).
function replay_ensemble(res; n_real::Integer = 100, trials = nothing, r_first::Integer = 0, q_noise_scale::Float64 = (pi / 180)^2,
                         e::Engine = engine())
    n = length(res.outcomes)
    sel = trials === nothing ? collect(1:n) : collect(trials)
    slew, _ = mc_replay_ensemble(n, n_real; r_first = r_first, trials = sel, q_noise_scale = q_noise_scale, e = e)
    fails = slew .== reshape([res.outcomes[t].t_final for t in sel], 1, :)
    fail_rate = [all(isnan, slew[:, k]) ? NaN : sum(fails[:, k]) / count(!isnan, slew[:, k]) for k in eachindex(sel)]
    ok(k) = [slew[i, k] for i in 1:n_real if !isnan(slew[i, k]) && !fails[i, k]]
    mean_ = [isempty(ok(k)) ? NaN : sum(ok(k)) / length(ok(k)) for k in eachindex(sel)]
    std_ = [isempty(ok(k)) ? NaN : sqrt(sum((ok(k) .- mean_[k]) .^ 2) / length(ok(k))) for k in eachindex(sel)]
    return (slew_time = slew, fails = fails, fail_rate = fail_rate, slew_mean = mean_, slew_std = std_, trials = sel)
end

# Continues a monte_carlo(...; resumable = true) result `res` in place to max_outer outer iterations in all: outcomes,
# slew_time, fails (monte_carlo.jl:257-261) and the trajectory arrays of the continued trials.  Returns their indices.
function continue_monte_carlo!(res; max_outer = 30, ilqr::Union{Nothing,IlqrOpts} = nothing, e::Engine = engine())
    base = ilqr === nothing ? res.ilqr : ilqr
    o = IlqrOpts((f == :max_outer ? Int32(max_outer) : getfield(base, f) for f in fieldnames(IlqrOpts))...)
    n = length(res.outcomes)
    idx = [t for t in 1:n if res.outcomes[t].status == 1 && res.outcomes[t].outer_iters < max_outer]   # MC1
    out, _ = mc_continue(n, o; e = e)
    res.outcomes .= out
    res.slew_time .= [r.slew_time for r in out]
    res.fails .= [r.slew_time == r.t_final ? 1.0 : 0.0 for r in out]
    if !isempty(idx) && haskey(res, :states)
        ko = zeros(Int64, n + 1)
        check(e, ccall((:ts_mc_trajectory_layout, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}), e.h, n, ko, C_NULL))
        X = zeros(8, ko[end]); U = zeros(3, ko[end]); Xs = zeros(8, ko[end]); Us = zeros(3, ko[end])
        sim = res.run_tvlqr
        check(e, ccall((:ts_mc_fetch_trajectories, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                       e.h, X, U, sim ? Xs : C_NULL, sim ? Us : C_NULL, C_NULL))
        for t in idx
            r = (ko[t] + 1):ko[t + 1]
            res.states[t] = X[:, r]; res.control_inputs[t] = U[:, r[1:end-1]]
            if sim
                res.sim_states[t] = Xs[:, r]; res.sim_control_inputs[t] = Us[:, r]
            end
        end
    end
    return idx
end

# igrf12syn(isv,date,itype,alt,colat,elong) -> (x,y,z,f)      reference src/igrf.jl:335-534 (scalar call = batch of one)
function igrf12syn(isv::Integer, date::Number, itype::Integer, alt::Number, colat::Number, elong::Number; e::Engine = engine())
    x = zeros(1); y = zeros(1); z = zeros(1); f = zeros(1)
    check(e, ccall((:ts_igrf12syn_batch, LIB), Cint,
                   (Ptr{Cvoid}, Cint, Cdouble, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Cint), e.h, isv, date, itype, 1, Float64[alt], Float64[colat], Float64[elong], x, y, z, f, 0))
    x[1], y[1], z[1], f[1]
end

# attitude_dynamics_linear(x,u,x_linear,B_B,J)                  reference src/attitude_dynamics.jl:26-48
function attitude_dynamics_linear(x, u, x_linear, B_B, J; e::Engine = engine())
    dx = zeros(7)
    check(e, ccall((:ts_attitude_dynamics_linear_batch, LIB), Cint,
                   (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   e.h, 1, collect(Float64, x), collect(Float64, u), collect(Float64, x_linear), collect(Float64, B_B),
                   vec(Matrix{Float64}(J')), dx))
    dx
end

# The PD magnetic controller loop of comparison/psiaki2005.jl:116-164 (one trial; B_ECI is 3 x N as in the script)
function psiaki_pd_simulation(x0, w_guess, q_guess, B_ECI, J, dt; C_1 = 1e-6, C_2 = 1e-9, e::Engine = engine())
    N = size(B_ECI, 2)
    X = zeros(7, N); M = zeros(3, N); Qe = zeros(4, N)
    check(e, ccall((:ts_psiaki_pd_batch, LIB), Cint,
                   (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cdouble,
                    Cdouble, Cdouble, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   e.h, 1, Int64[N], Int64[0], collect(Float64, x0), Matrix{Float64}(w_guess), Matrix{Float64}(q_guess),
                   Matrix{Float64}(B_ECI), vec(Matrix{Float64}(J')), dt, C_1, C_2, X, M, Qe))
    X, M, Qe
end

# ----------------------------------------------------------------------------- element-wise building blocks
# kep_ECI(kep_elements,t0,GM) -> [r'; v'] (2 x 3)            reference src/kep_ECI.jl:1-35 (mutates kep_elements[6], :7-8)
function kep_ECI(kep_elements, t0, GM; e::Engine = engine())
    k = collect(Float64, vec(kep_elements)); rv = zeros(6)
    check(e, ccall((:ts_kep_eci_batch, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Cdouble, Ptr{Float64}),
                   e.h, 1, k, Float64[t0], GM, rv))
    kep_elements[6] = rem(kep_elements[6] + t0 * sqrt(GM ./ kep_elements[2] .^ 3), 360)
    [rv[1:3]'; rv[4:6]']
end
# OrbitPlotter(x,p,t) -> [v; a]                               reference src/OrbitPlotter.jl:1-52
function OrbitPlotter(x, p, t; e::Engine = engine())
    dx = zeros(6)
    check(e, ccall((:ts_orbit_rhs_batch, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}), e.h, 1, collect(Float64, x), dx))
    dx
end
# legendre(Val{:schmidt}, phi, n_max, false) / dlegendre(Val{:schmidt}, phi, P, false)   src/legendre.jl:254-292, src/dlegendre.jl:221-309
function legendre(::Type{Val{:schmidt}}, phi::Number, n_max::Number, ph_term::Bool = false; e::Engine = engine())
    ph_term && error("only ph_term = false is on the IGRF path (igrf.jl:124)")
    d = Int(n_max) + 1; P = zeros(d, d)
    check(e, ccall((:ts_legendre_schmidt_batch, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}),
                   e.h, 1, Float64[phi], n_max, P, C_NULL))
    Matrix(P')                      # the library is row-major
end
function dlegendre(::Type{Val{:schmidt}}, phi::Number, P::Matrix, ph_term::Bool = false; e::Engine = engine())
    ph_term && error("only ph_term = false is on the IGRF path (igrf.jl:125)")
    d = size(P, 1); Pb = zeros(d, d); dP = zeros(d, d)
    check(e, ccall((:ts_legendre_schmidt_batch, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}),
                   e.h, 1, Float64[phi], d - 1, Pb, dP))
    Matrix(dP')
end
# DerivFunction(dx,x,u) / gain_simulator(dx,x,u): in-place 8-state dynamics reading the reference's globals
# B_ECI (rows x 3), N, p.J, tf, t0                            reference src/DerivFunction.jl:1-48, src/gain_simulator.jl:1-53
function _dynamics!(mode, dx, x, u, B_ECI, N, J, tf, t0; e::Engine = engine())
    Bt = Matrix{Float64}(B_ECI'); o = zeros(8)
    check(e, ccall((:ts_dynamics_batch, LIB), Cint,
                   (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Cdouble, Cdouble, Ptr{Float64}, Ptr{Float64}),
                   e.h, mode, 1, collect(Float64, x), collect(Float64, u), Bt, size(Bt, 2), Float64(N), 1 / (tf - t0),
                   vec(Matrix{Float64}(J')), o))
    dx[1:8] = o
end
DerivFunction(dx, x, u) = _dynamics!(0, dx, x, u, Main.B_ECI, Main.N, Main.p.J, Main.tf, Main.t0)
gain_simulator(dx, x, u) = _dynamics!(1, dx, x, u, Main.B_ECI, Main.N, Main.p.J, Main.tf, Main.t0)
# attitude_dynamics(x,u,B_B,J) -> xdot (7)                      reference src/attitude_dynamics.jl:2-24
function attitude_dynamics(x, u, B_B, J; e::Engine = engine())
    o = zeros(7)
    check(e, ccall((:ts_dynamics_batch, LIB), Cint,
                   (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Cdouble, Cdouble, Ptr{Float64}, Ptr{Float64}),
                   e.h, 2, 1, collect(Float64, x), collect(Float64, u), collect(Float64, B_B), 1, 1.0, 0.0, vec(Matrix{Float64}(J')), o))
    o
end

# ----------------------------------------------------------------------------- small host-side helpers kept verbatim in meaning
qmult(q1, q2) = [q1[1] * q2[1] - q1[2:4]' * q2[2:4]; q1[1] * q2[2:4] + q2[1] * q1[2:4] + cross(q1[2:4], q2[2:4])]  # src/qmult.jl
qrot(q, r) = r + 2 * cross(q[2:4], cross(q[2:4], r) + q[1] * r)                                                      # src/qrot.jl
q_inv(q) = [q[1]; -q[2:4]]                                                              # src/attitude_controller.jl:164-166
hat(x) = [0 -x[3] x[2]; x[3] 0 -x[1]; -x[2] x[1] 0]                                     # src/magnetic_toolbox.jl:142-146

export Engine, params, input_parameters, igrf12, igrf12_batch, igrf_data, magnetic_simulation, magnetic_gramian, kep_ECI, OrbitPlotter,
       legendre, dlegendre, DerivFunction, gain_simulator, attitude_dynamics,
       condition_based_time, eigen_axis_slew, bryson_weights, solve_slew, attitude_simulation, monte_carlo, qmult, qrot, q_inv, hat,
       igrf12syn, attitude_dynamics_linear, psiaki_pd_simulation, igrf_interpolant, field_map_prefilter, field_map_eval, AlState,
       mc_state, mc_continue, continue_monte_carlo!, ReplayEnsembleOpts, mc_replay_ensemble, replay_ensemble

end # module
