# LoraineB200DD.jl -- `ccall` shims of the double-double LP path (include/loraine_b200_dd.h) for `Loraine.Optimizer{Float64x2}`
# on models WITHOUT semidefinite blocks (the shape of examples/k.jl:8-38).  Optional companion of LoraineB200.jl:
#
#     using Loraine, MultiFloats
#     include("LoraineB200.jl"); include("LoraineB200DD.jl"); LoraineB200.enable!("/path/to/libloraine_b200.so")
#     model = Model(Loraine.Optimizer{Float64x2}); ...; optimize!(model)
#
# The methods below are more specific than both the reference's (`MySolver{T}`) and LoraineB200.jl's rejection method
# (`solve(::MySolver{T}) where T<:AbstractFloat`), so a Float64x2 solver of an LP-only model runs on the GPU in double-double
# arithmetic; a Float64x2 model WITH PSD blocks is still rejected (ArgumentError), every other element type as before.
# A Float64x2 scalar crosses the boundary as its two limbs (`x._limbs`), a vector as two Float64 arrays (hi, lo).
#
# STATUS: UNTESTED UNDER JULIA (no Julia in the build image).  The executed mirror of this control flow is
# loraine.jl_b200/dd_lp.py (GPU tests tests/test_gpu_dd.py: examples/k.jl to 1e-24, phase parity against a 160-bit oracle).
module LoraineB200DD

using Loraine
using LinearAlgebra, Printf, SparseArrays
using MultiFloats
import ..LoraineB200: LIB, ENABLED, NGPUS
const S = Loraine.Solvers
const T2 = Float64x2

const HANDLES = IdDict{Any,Ptr{Cvoid}}()       # MySolver{Float64x2} => lrn_dd_handle_t

limbs(x::T2) = Float64[x._limbs[1], x._limbs[2]]
limbs(x::Real) = Float64[Float64(x), 0.0]
f64x2(v::Vector{Float64}) = T2(v[1]) + T2(v[2])
hi_lo(v) = (Float64[Float64(T2(x)._limbs[1]) for x in v], Float64[Float64(T2(x)._limbs[2]) for x in v])

dd(solver) = HANDLES[solver]
function ddcheck(solver, rc, what)
    rc < 0 && error("loraine_b200: $what failed ($rc): " * unsafe_string(ccall((:lrn_dd_last_error, LIB[]), Cstring, (Ptr{Cvoid},), dd(solver))))
    rc > 0 && throw(LinearAlgebra.PosDefException(rc))
    return rc
end

function S.setup_solver(solver::S.MySolver{T2}, halpha::S.Halpha)
    invoke(S.setup_solver, Tuple{S.MySolver,S.Halpha}, solver, halpha)      # reference body (src/Solvers.jl:363-446)
    ENABLED[] || return nothing
    md = solver.model
    md.nlmi == 0 || throw(ArgumentError("Loraine.Optimizer{Float64x2} on the B200 path: models without PSD blocks only (no fallback)"))
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    # enable!(...; ngpus) other than 1: one host thread drives several GPUs (Schur matrix sharded, NCCL inside the library)
    rc = if NGPUS[] == 1
        ccall((:lrn_dd_create, LIB[]), Int32, (Ref{Ptr{Cvoid}}, Int64, Int64, Int32), hr, md.n, md.nlin, -1)
    else
        ccall((:lrn_dd_create_multi, LIB[]), Int32, (Ref{Ptr{Cvoid}}, Int64, Int64, Int32, Ptr{Int32}), hr, md.n, md.nlin, NGPUS[], C_NULL)
    end
    rc == 0 || error("loraine_b200: lrn_dd_create / lrn_dd_create_multi failed ($rc); there is no CPU fallback")
    HANDLES[solver] = hr[]
    Cl = SparseMatrixCSC{Float64,Int64}(md.C_lin); d = Vector{Float64}(vec(md.d_lin)); b = Vector{Float64}(vec(md.b))
    GC.@preserve Cl d b begin        # model data are Float64 in the reference (src/model.jl:44, src/Solvers.jl:576)
        ddcheck(solver, ccall((:lrn_dd_set_lin, LIB[]), Int32,
                              (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                              dd(solver), Cl.colptr, Cl.rowval, Cl.nzval, C_NULL, d, C_NULL), "lrn_dd_set_lin")
        ddcheck(solver, ccall((:lrn_dd_set_b, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), dd(solver), b, C_NULL), "lrn_dd_set_b")
    end
    ddcheck(solver, ccall((:lrn_dd_finalize, LIB[]), Int32, (Ptr{Cvoid},), dd(solver)), "lrn_dd_finalize")
    return nothing
end

function S.initial_point(solver::S.MySolver{T2})
    invoke(S.initial_point, Tuple{Any}, solver)                            # src/initial_point.jl:1-81 (Float64 `ones` / `zeros`)
    ENABLED[] || return nothing
    yh, yl = hi_lo(vec(solver.y)); xh, xl = hi_lo(vec(solver.X_lin)); sh, sl = hi_lo(vec(solver.S_lin))
    ddcheck(solver, ccall((:lrn_dd_set_iterate, LIB[]), Int32,
                          (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                          dd(solver), yh, yl, xh, xl, sh, sl), "lrn_dd_set_iterate")
    return nothing
end

function S.find_mu(solver::S.MySolver{T2})                                 # src/Solvers.jl:480-494
    ENABLED[] || return invoke(S.find_mu, Tuple{Any}, solver)
    mu = zeros(2)
    ddcheck(solver, ccall((:lrn_dd_find_mu, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), dd(solver), mu), "lrn_dd_find_mu")
    solver.mu = f64x2(mu)
end

function S.prepare_W(solver::S.MySolver{T2})                               # src/prepare_W.jl:86 (LP part only)
    ENABLED[] || return invoke(S.prepare_W, Tuple{S.MySolver}, solver)
    ddcheck(solver, ccall((:lrn_dd_prepare_W, LIB[]), Int32, (Ptr{Cvoid},), dd(solver)), "lrn_dd_prepare_W")
end

function S.find_step(solver::S.MySolver{T2})                               # src/predictor_corrector.jl:329-364
    ENABLED[] || return invoke(S.find_step, Tuple{S.MySolver}, solver)
    a = zeros(2); b = zeros(2)
    ddcheck(solver, ccall((:lrn_dd_find_step, LIB[]), Int32,
                          (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Float64}, Ptr{Float64}),
                          dd(solver), solver.predict ? 1 : 0, limbs(solver.sigma), limbs(solver.mu), Float64(solver.tau), a, b), "lrn_dd_find_step")
    solver.alpha_lin = f64x2(a); solver.beta_lin = f64x2(b)
    solver.alpha = T2[]; solver.beta = T2[]
end

function S.predictor(solver::S.MySolver{T2}, halpha::S.Halpha)             # src/predictor_corrector.jl:5-146, kit = 0 branch
    ENABLED[] || return invoke(S.predictor, Tuple{S.MySolver,S.Halpha}, solver, halpha)
    solver.predict = true
    h = dd(solver)
    ddcheck(solver, ccall((:lrn_dd_residuals, LIB[]), Int32, (Ptr{Cvoid},), h), "lrn_dd_residuals")
    ddcheck(solver, ccall((:lrn_dd_schur_assemble, LIB[]), Int32, (Ptr{Cvoid},), h), "lrn_dd_schur_assemble")
    ddcheck(solver, ccall((:lrn_dd_rhs_predictor, LIB[]), Int32, (Ptr{Cvoid},), h), "lrn_dd_rhs_predictor")
    which = Int32(3)
    rc = ccall((:lrn_dd_schur_factor, LIB[]), Int32, (Ptr{Cvoid},), h)
    rc < 0 && ddcheck(solver, rc, "lrn_dd_schur_factor")
    if rc > 0                                                              # :60-88
        solver.verb > 0 && println("Matrix H not positive definite, trying to regularize")
        icount = 0
        solver.regcount += 1
        if solver.regcount > 5
            solver.verb > 0 && println("WARNING: too many regularizations of H, giving up")
            solver.status = 3
            return
        end
        while true
            ddcheck(solver, ccall((:lrn_dd_schur_shift, LIB[]), Int32, (Ptr{Cvoid}, Float64), h, 1e-4), "lrn_dd_schur_shift")
            icount += 1
            rc = ccall((:lrn_dd_schur_factor, LIB[]), Int32, (Ptr{Cvoid},), h)
            rc < 0 && ddcheck(solver, rc, "lrn_dd_schur_factor")
            rc == 0 && break
            if icount > 1000
                solver.verb > 0 && println("WARNING: H cannot be made positive definite, giving up")
                solver.status = 3
                return
            end
        end
        which = Int32(6)                                                   # `cholesky(BBBB)` object: H^-1 H^-1 h (:85-90)
    end
    solver.cholBBBB = which                                                # the corrector solves with the same factor (:199)
    ddcheck(solver, ccall((:lrn_dd_schur_solve, LIB[]), Int32, (Ptr{Cvoid}, Int32), h, which), "lrn_dd_schur_solve")
    S.find_step(solver)
end

function S.sigma_update(solver::S.MySolver{T2})                            # src/predictor_corrector.jl:148-179
    ENABLED[] || return invoke(S.sigma_update, Tuple{S.MySolver}, solver)
    step_pred = min(solver.alpha_lin, solver.beta_lin)
    if solver.mu > 1e-6
        expon_used = step_pred < 1 / sqrt(3) ? 1.0 : max(solver.expon, T2(3) * step_pred^2)
    else
        expon_used = max(1, min(solver.expon, T2(3) * step_pred^2))
    end
    dl = zeros(2)
    ddcheck(solver, ccall((:lrn_dd_sigma_trace, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), dd(solver), dl), "lrn_dd_sigma_trace")
    tmp12 = convert(Float64, f64x2(dl) / (0 + solver.model.nlin))          # the reference rounds to Float64 here (:173-175)
    solver.sigma = min(1.0, (tmp12 / Float64(solver.mu))^Float64(expon_used))
    return solver.sigma
end

function S.corrector(solver::S.MySolver{T2}, halpha)                       # src/predictor_corrector.jl:181-246, kit = 0 branch
    ENABLED[] || return invoke(S.corrector, Tuple{Any,Any}, solver, halpha)
    solver.predict = false
    ddcheck(solver, ccall((:lrn_dd_rhs_corrector, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), dd(solver),
                          limbs(solver.sigma), limbs(solver.mu)), "lrn_dd_rhs_corrector")
    ddcheck(solver, ccall((:lrn_dd_schur_solve, LIB[]), Int32, (Ptr{Cvoid}, Int32), dd(solver), Int32(solver.cholBBBB)), "lrn_dd_schur_solve")
    S.find_step(solver)
end

function S.myIPstep(solver::S.MySolver{T2}, halpha::S.Halpha)              # src/Solvers.jl:448-478
    ENABLED[] || return invoke(S.myIPstep, Tuple{S.MySolver,S.Halpha}, solver, halpha)
    solver.iter += 1
    if solver.iter > solver.maxit
        solver.status = 4
        solver.verb > 0 && println("WARNING: Stopped by iteration limit (stopping status = 4)")
    end
    solver.cg_iter_pre = 0
    solver.cg_iter_cor = 0
    S.find_mu(solver)
    S.prepare_W(solver)
    S.predictor(solver, halpha)
    solver.status == 3 && return
    S.sigma_update(solver)
    S.corrector(solver, halpha)
end

function S.check_convergence(solver::S.MySolver{T2})                       # src/Solvers.jl:496-568 for nlmi = 0
    ENABLED[] || return invoke(S.check_convergence, Tuple{Any}, solver)
    md = solver.model
    err = zeros(12); by = zeros(2); dx = zeros(2)
    ddcheck(solver, ccall((:lrn_dd_dimacs, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), dd(solver), err, by, dx), "lrn_dd_dimacs")
    e = [f64x2(err[2k-1:2k]) for k in 1:6]
    solver.err1, solver.err2, solver.err3, solver.err4, solver.err5, solver.err6 = e
    DIMACS_error = e[2] + e[3] + e[4] + abs(e[5]) + e[6]                   # nlmi = 0: err1 is left out (:521)
    solver.DIMACS_error = DIMACS_error
    byv = f64x2(by); dxv = f64x2(dx)
    if solver.verb > 0 && solver.status == 0
        @printf("%3.0d %16.8e %9.2e %8.2f\n", solver.iter, Float64(-byv + md.b_const), Float64(DIMACS_error), solver.itertime)
    end
    if DIMACS_error < solver.eDIMACS
        solver.status = 1
        if solver.verb > 0
            println("Primal objective: ", -byv + md.b_const)
            println("Dual objective:   ", -dxv)
        end
    end
    if DIMACS_error > 1e55
        solver.status = 2
    elseif abs(byv) > 1e55
        solver.status = 3
    end
end

function S.solve(solver::S.MySolver{T2}, halpha::S.Halpha)                 # src/Solvers.jl:304-361
    ENABLED[] || return invoke(S.solve, Tuple{S.MySolver,S.Halpha}, solver, halpha)
    invoke(S.solve, Tuple{S.MySolver,S.Halpha}, solver, halpha)            # the reference loop; the calls inside dispatch to the methods above
    md = solver.model
    yh = zeros(md.n); yl = zeros(md.n); xh = zeros(md.nlin); xl = zeros(md.nlin); sh = zeros(md.nlin); sl = zeros(md.nlin)
    ddcheck(solver, ccall((:lrn_dd_get_solution, LIB[]), Int32,
                          (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                          dd(solver), yh, yl, xh, xl, sh, sl), "lrn_dd_get_solution")
    solver.y = T2.(yh) .+ T2.(yl); solver.X_lin = T2.(xh) .+ T2.(xl); solver.S_lin = T2.(sh) .+ T2.(sl)
    ccall((:lrn_dd_destroy, LIB[]), Int32, (Ptr{Cvoid},), dd(solver)); delete!(HANDLES, solver)
    return nothing
end

end # module
