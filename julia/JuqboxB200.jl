# JuqboxB200.jl — the reference-side binding of libjuqbox_b200.so (include/juqbox_b200.h).
#
# NOT EXECUTED IN THIS REPO'S CI: the build image has no `julia`.  It is the ~150 lines a Juqbox maintainer adds
# (e.g. as src/b200.jl, `include`d from src/Juqbox.jl after evalobjgrad.jl and ipopt_interface.jl) so that
# setup scripts, `setup_ipopt_problem` and `run_optimizer` run unchanged while every objective/gradient
# evaluation goes to the GPU.  The Python mirror juqbox_b200/api.py is this file's tested twin.
#
# What it replaces in the reference:
#   Working_Arrays(params, nCoeff)                      src/evalobjgrad.jl:405      -> Working_Arrays_B200
#   traceobjgrad(pcof0, params, wa, verbose, evaladjoint)  src/evalobjgrad.jl:504   -> new method on Working_Arrays_B200
#   eval_f_g_grad!(pcof, params, wa, nodes, weights, ..)   src/ipopt_interface.jl:24 -> new method: ONE batched ccall
#                                                                                     instead of the nquad loop
# eval_f_par / eval_grad_f_par / eval_g_par / eval_jac_g_par take `wa` untyped (src/ipopt_interface.jl:77-179); the methods at
# the end of this file specialise them on Working_Arrays_B200 so that each Ipopt callback is ONE ccall (jq_eval_f_grad: cache
# test, sample loop, weighted sums and Tikhonov behind the ABI).  Without those four methods the generic ones still work:
# they dispatch to eval_f_g_grad! below through `wa`.
#
# Layout pin: tests/c_abi_harness.c (gcc) asserts sizeof(jq_problem) == 208, sizeof(jq_operator) == 40 and the field offsets
# the two structs below produce; at run time compare with jq_abi_info (jq_check_layout()).

const libjq = get(ENV, "JUQBOX_B200_LIB", "libjuqbox_b200.so")

struct JqOperator            # == jq_operator
    format::Int32
    nnz::Int64
    colptr::Ptr{Int64}
    rowval::Ptr{Int64}
    nzval::Ptr{Float64}
end

struct JqProblem             # == jq_problem
    n::Int32; m::Int32; ncoupled::Int32; nfreq::Int32
    neumann_terms::Int32; obj_func_type::Int32; pfid_type::Int32; linear_solver::Int32
    nsteps::Int64
    T::Float64
    uinit::Ptr{Float64}; vtarget_r::Ptr{Float64}; vtarget_i::Ptr{Float64}; wdiag::Ptr{Float64}; cfreq::Ptr{Float64}
    h0::JqOperator
    hsym::Ptr{JqOperator}
    hanti::Ptr{JqOperator}
    solver_tol::Float64
    global_phase::Float64                    # params.globalPhase (pFidType 1 and 4)
    wmat_real::Ptr{Float64}                  # dense Ntot x Ntot weights (use_custom_forbidden) or C_NULL
    wmat_imag::Ptr{Float64}
    nuncoupled::Int32; reserved0::Int32
    hunc::Ptr{JqOperator}
    unc_is_symm::Ptr{Int32}
    unc_rfreq::Ptr{Float64}
end

function jq_check_layout()
    info(k) = ccall((:jq_abi_info, libjq), Int64, (Int32,), k)
    (info(1) == sizeof(JqProblem) && info(2) == sizeof(JqOperator) && info(3) == fieldoffset(JqProblem, 9) &&
     info(6) == fieldoffset(JqProblem, 16) && info(8) == fieldoffset(JqProblem, 19)) ||
        error("juqbox_b200: struct layout of JuqboxB200.jl does not match the library (ABI version ", info(0), ")")
end

jq_error() = unsafe_string(ccall((:jq_last_error, libjq), Cstring, ()))
jq_check(rc) = rc == 0 ? nothing : error("juqbox_b200: ", jq_error())     # non-zero -> Julia error(), as the reference does

mutable struct Working_Arrays_B200
    handle::Ptr{Cvoid}
    nCoeff::Int64
    keep::Vector{Any}        # arrays referenced by the descriptor while jq_create runs
end

# dense Array{Float64,2} is already column-major; SparseMatrixCSC is CSC with 1-based indices -> shift to 0-based
function jq_operator(A::Array{Float64,2}, keep)
    push!(keep, A)
    JqOperator(0, length(A), C_NULL, C_NULL, pointer(A))
end
function jq_operator(A::SparseMatrixCSC{Float64,Int64}, keep)
    cp = A.colptr .- 1; rv = A.rowval .- 1; nz = copy(A.nzval)
    append!(keep, (cp, rv, nz))
    JqOperator(1, length(nz), pointer(cp), pointer(rv), pointer(nz))
end

function Working_Arrays_B200(params::objparams, nCoeff::Int64; device::Int = 0)
    @assert params.linear_solver.solver_id in (NEUMANN_SOLVER, JACOBI_SOLVER) "Neumann and Jacobi solvers are built for B200"
    @assert params.Integrator_id == Stormer_Verlet
    jq_check_layout()
    keep = Any[]
    Ntot = params.N + params.Nguard
    Nctrl = params.Ncoupled + params.Nunc
    Cf = Array{Float64,2}(params.Cfreq[1:Nctrl, :])
    wd = Vector{Float64}(diag(params.wmat_real))
    dense_w = !isa(params.wmat_real, Diagonal)                     # use_custom_forbidden (src/evalobjgrad.jl:214-232)
    wr = dense_w ? Array{Float64,2}(params.wmat_real) : zeros(0, 0)
    wi = dense_w ? Array{Float64,2}(params.wmat_imag) : zeros(0, 0)
    hs = [jq_operator(h, keep) for h in params.Hsym_ops]
    ha = [jq_operator(h, keep) for h in params.Hanti_ops]
    hu = [jq_operator(h, keep) for h in params.Hunc_ops]           # two splines per uncoupled control, as KS! reads them (:2372-2387)
    sy = Int32[s ? 1 : 0 for s in params.isSymm]
    rf = Vector{Float64}(params.Rfreq[1:params.Nunc])
    append!(keep, (Cf, wd, wr, wi, hs, ha, hu, sy, rf, params.Uinit, params.Utarget_r, params.Utarget_i))
    pb = JqProblem(Ntot, params.N, params.Ncoupled, params.Nfreq, params.linear_solver.max_iter, params.objFuncType,
                   params.pFidType, params.linear_solver.solver_id, params.nsteps, params.T, pointer(params.Uinit), pointer(params.Utarget_r),
                   pointer(params.Utarget_i), pointer(wd), pointer(Cf), jq_operator(params.Hconst, keep),
                   params.Ncoupled > 0 ? pointer(hs) : Ptr{JqOperator}(C_NULL), params.Ncoupled > 0 ? pointer(ha) : Ptr{JqOperator}(C_NULL),
                   params.linear_solver.tol, params.globalPhase, dense_w ? pointer(wr) : Ptr{Float64}(C_NULL),
                   dense_w ? pointer(wi) : Ptr{Float64}(C_NULL), Int32(params.Nunc), Int32(0),
                   params.Nunc > 0 ? pointer(hu) : Ptr{JqOperator}(C_NULL), params.Nunc > 0 ? pointer(sy) : Ptr{Int32}(C_NULL),
                   params.Nunc > 0 ? pointer(rf) : Ptr{Float64}(C_NULL))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve keep pb jq_check(ccall((:jq_create, libjq), Cint, (Ref{JqProblem}, Cint, Ref{Ptr{Cvoid}}), pb, device, h))
    wa = Working_Arrays_B200(h[], nCoeff, Any[])
    finalizer(w -> ccall((:jq_destroy, libjq), Cint, (Ptr{Cvoid},), w.handle), wa)
    return wa
end

# change_target! (src/evalobjgrad.jl:1492) must be followed by this to refresh the device copy
update_target!(wa::Working_Arrays_B200, params::objparams) =
    jq_check(ccall((:jq_update_target, libjq), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), wa.handle, params.Utarget_r, params.Utarget_i))

# Batched core: pcof is Npar x nbatch (one candidate per column), shifts is n x nsamples (one diagonal per column).
function traceobjgrad_batch(pcof::Array{Float64,2}, params::objparams, wa::Working_Arrays_B200;
                            shifts::Union{Nothing,Array{Float64,2}} = nothing, weights::Union{Nothing,Vector{Float64}} = nothing,
                            evaladjoint::Bool = true)
    Npar, nbatch = size(pcof)
    nsamples = shifts === nothing ? 1 : size(shifts, 2)
    nout = weights === nothing ? nbatch * nsamples : nbatch
    infid = zeros(nout); leak = zeros(nout); tinf = zeros(nout)
    two = params.objFuncType != 1                        # objFuncType 1: infidelgrad aliases totalgrad (src/evalobjgrad.jl:951),
    grad = zeros(Npar, nout)                             # so only one gradient is fetched from the device
    igrad = two ? zeros(Npar, nout) : grad
    lgrad = two ? zeros(Npar, nout) : zeros(Npar, 0)
    jq_check(ccall((:jq_traceobjgrad_batch, libjq), Cint,
                   (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Int32,
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   wa.handle, nbatch, pcof, Npar, nsamples, shifts === nothing ? C_NULL : shifts,
                   weights === nothing ? C_NULL : weights, evaladjoint, infid, leak, tinf, grad,
                   two ? pointer(igrad) : Ptr{Float64}(C_NULL), two ? pointer(lgrad) : Ptr{Float64}(C_NULL)))
    return infid, leak, tinf, grad, igrad, lgrad
end

# Drop-in method: same return tuples as src/evalobjgrad.jl:1032-1035.  verbose=true is not offered on the GPU
# (state history + forward-sensitivity check, SURVEY.md row 14): keep a CPU Working_Arrays for plot_results.
function traceobjgrad(pcof0::Array{Float64,1}, params::objparams, wa::Working_Arrays_B200, verbose::Bool = false, evaladjoint::Bool = true)
    verbose && error("verbose=true: call traceobjgrad with a CPU Working_Arrays")
    infid, leak, tinf, grad, igrad, lgrad = traceobjgrad_batch(reshape(pcof0, :, 1), params, wa; evaladjoint = evaladjoint)
    objfv = infid[1] + leak[1]
    evaladjoint || return objfv, infid[1], leak[1]
    totalgrad = grad[:, 1]
    if params.objFuncType != 1
        return objfv, totalgrad, infid[1], leak[1], tinf[1], igrad[:, 1], lgrad[:, 1]
    else
        return objfv, totalgrad, infid[1], leak[1], tinf[1], totalgrad, zeros(0)
    end
end

# The risk-neutral sample loop (src/ipopt_interface.jl:38-65) as one call: no mutate/restore of params.Hconst.
function eval_f_g_grad!(pcof::Vector{Float64}, params::objparams, wa::Working_Arrays_B200,
                        nodes::AbstractArray = [0.0], weights::AbstractArray = [1.0], compute_adjoint::Bool = true)
    n = params.N + params.Nguard
    shifts = zeros(n, length(nodes))
    for i in 1:length(nodes), j in 2:n
        shifts[j, i] = 0.01 * nodes[i] * (10.0^(j - 2))          # src/ipopt_interface.jl:43
    end
    infid, leak, _, _, igrad, lgrad = traceobjgrad_batch(reshape(pcof, :, 1), params, wa; shifts = shifts,
                                                         weights = Vector{Float64}(weights), evaladjoint = compute_adjoint)
    params.last_pcof .= pcof
    params.last_infidelity = infid[1]
    params.last_leak = leak[1]
    if compute_adjoint
        params.last_infidelity_grad .= igrad[:, 1]                 # == total gradient when objFuncType == 1 (:951)
        params.objFuncType != 1 && (params.last_leak_grad .= lgrad[:, 1])
    end
    params.lastTraceInfidelity = params.last_infidelity
    params.lastLeakIntegral = params.last_leak
end

# evalctrl (src/plotstatectrl.jl:246-276) on the GPU handle: control `jFunc` (1-based) on the grid `td`, rad/ns.
function evalctrl(params::objparams, pcof0::Array{Float64,1}, td::Array{Float64,1}, jFunc::Int64, wa::Working_Arrays_B200)
    nt = length(td)
    p = zeros(nt, params.Ncoupled); q = zeros(nt, params.Ncoupled)       # column c = control c  ==  ABI [ncoupled][ntimes]
    jq_check(ccall((:jq_eval_controls, libjq), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   wa.handle, pcof0, length(pcof0), nt, td, p, q))
    return p[:, jFunc], q[:, jFunc]
end

# eval_forward(U0, pcof, params; saveEndOnly=false, saveEvery) (src/evalobjgrad.jl:2727-2873) with U0 = params.Uinit:
# returns the Ntot x N x nsave complex state history.
function eval_forward(pcof0::Array{Float64,1}, params::objparams, wa::Working_Arrays_B200; saveEvery::Int64 = 1)
    Ntot = params.N + params.Nguard
    nsave = div(params.nsteps, saveEvery) + 1
    hr = zeros(Ntot, params.N, nsave); hi = zeros(Ntot, params.N, nsave)
    jq_check(ccall((:jq_eval_forward, libjq), Cint,
                   (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Int32, Ptr{Float64}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   wa.handle, 1, pcof0, length(pcof0), 1, C_NULL, saveEvery, hr, hi, C_NULL, C_NULL))
    return hr .+ im .* hi
end

# Forward sensitivities (the forward-sensitivity check of traceobjgrad(pcof, params, wa, true, true), src/evalobjgrad.jl:724-745,768-784,
# for ndir directions in one launch): dirs is Npar x ndir, one direction per column (dirs = I: the whole forward-mode gradient;
# dirs = e_kpar: the reference's component kpar).  Without weights: infid, leak [nsamples] and dinfid, dleak ndir x nsamples;
# with weights: the weighted sums over the nodes, infid, leak [1] and dinfid, dleak [ndir].  The column-major arrays are the ABI's
# row-major views, nothing is transposed.
function forward_sensitivity(pcof::Vector{Float64}, params::objparams, wa::Working_Arrays_B200, dirs::Array{Float64,2};
                             nodes::AbstractArray = [0.0], weights::Union{Nothing,AbstractArray} = nothing)
    Npar, ndir = size(dirs)
    Npar == length(pcof) || error("forward_sensitivity: dirs must be Npar x ndir with Npar = length(pcof)")
    shifts = jq_shifts(params, nodes)
    nsamples = length(nodes)
    w = weights === nothing ? nothing : Vector{Float64}(weights)
    nout = w === nothing ? nsamples : 1
    infid = zeros(nout); leak = zeros(nout)
    dinfid = zeros(ndir, nout); dleak = zeros(ndir, nout)
    jq_check(ccall((:jq_forward_sensitivity, libjq), Cint,
                   (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                   wa.handle, 1, pcof, Npar, nsamples, shifts, w === nothing ? C_NULL : w, ndir, dirs,
                   infid, leak, dinfid, dleak, C_NULL, C_NULL))
    return w === nothing ? (infid, leak, dinfid, dleak) : (infid, leak, vec(dinfid), vec(dleak))
end


# ---- the four Ipopt callbacks as ONE ccall each (src/ipopt_interface.jl:77-179): jq_eval_f_grad keeps the last-pcof cache, runs
# eval_f_g_grad!'s sample loop as one launch and adds the Tikhonov terms on the device.  params.last_* scalars are kept for
# intermediate_par (:212-228).
function jq_shifts(params::objparams, nodes::AbstractArray)
    n = params.N + params.Nguard
    shifts = zeros(n, length(nodes))
    for i in 1:length(nodes), j in 2:n
        shifts[j, i] = 0.01 * nodes[i] * (10.0^(j - 2))          # src/ipopt_interface.jl:43
    end
    return shifts
end

function jq_eval_f_grad(pcof::Vector{Float64}, params::objparams, wa::Working_Arrays_B200, nodes::AbstractArray, weights::AbstractArray)
    Npar = length(pcof)
    shifts = jq_shifts(params, nodes)
    w = Vector{Float64}(weights)
    f = Ref{Float64}(0.0); infid = Ref{Float64}(0.0); leak = Ref{Float64}(0.0); ev = Ref{Int32}(0)
    grad = zeros(Npar)
    lgrad = params.objFuncType != 1 ? zeros(Npar) : zeros(0)
    prior = params.usingPriorCoeffs ? Vector{Float64}(params.priorCoeffs) : zeros(0)
    jq_check(ccall((:jq_eval_f_grad, libjq), Cint,
                   (Ptr{Cvoid}, Ptr{Float64}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Float64},
                    Ref{Float64}, Ptr{Float64}, Ref{Float64}, Ref{Float64}, Ptr{Float64}, Ref{Int32}),
                   wa.handle, pcof, Npar, length(nodes), shifts, w, params.tik0,
                   params.usingPriorCoeffs ? pointer(prior) : Ptr{Float64}(C_NULL), f, grad, infid, leak,
                   params.objFuncType != 1 ? pointer(lgrad) : Ptr{Float64}(C_NULL), ev))
    params.last_pcof .= pcof
    params.last_infidelity = infid[]; params.last_leak = leak[]
    params.lastTraceInfidelity = infid[]; params.lastLeakIntegral = leak[]
    return f[], grad, leak[], lgrad, ev[] != 0
end

eval_f_par(pcof::Vector{Float64}, params::objparams, wa::Working_Arrays_B200, nodes::AbstractArray = [0.0], weights::AbstractArray = [1.0]) =
    jq_eval_f_grad(pcof, params, wa, nodes, weights)[1]

function eval_grad_f_par(pcof::Vector{Float64}, grad_f::Vector{Float64}, params::objparams, wa::Working_Arrays_B200,
                         nodes::AbstractArray = [0.0], weights::AbstractArray = [1.0])
    grad_f .= jq_eval_f_grad(pcof, params, wa, nodes, weights)[2]
    params.save_pcof_hist && push!(params.pcof_hist, copy(pcof))
end

function eval_g_par(pcof::Vector{Float64}, g::Vector{Float64}, params::objparams, wa::Working_Arrays_B200,
                    nodes::AbstractArray = [0.0], weights::AbstractArray = [1.0])
    g[1] = jq_eval_f_grad(pcof, params, wa, nodes, weights)[3]
    return g[1]
end

function eval_jac_g_par(pcof::Vector{Float64}, rows::Vector{Int32}, cols::Vector{Int32}, jac_g::Union{Nothing,Vector{Float64}},
                        params::objparams, wa::Working_Arrays_B200, nodes::AbstractArray = [0.0], weights::AbstractArray = [1.0])
    if jac_g === nothing
        for i in 1:(length(rows) > 0 ? length(pcof) : 0)
            rows[i] = 1; cols[i] = i
        end
        return
    end
    _, _, _, lgrad, evaluated = jq_eval_f_grad(pcof, params, wa, nodes, weights)
    evaluated && return            # the reference returns without filling jac_g when it had to re-evaluate (:169-173)
    jac_g .= lgrad
    return
end

# ---- kernel selection and multi-GPU switches (optional: automatic mode serves one pcof per callback with the time-parallel path) ----
# kernel: 0 automatic … 7 time-parallel evaluation; nseg: number of time segments of kernel 7 (0 = automatic)
set_kernel!(wa::Working_Arrays_B200, kernel::Integer) = jq_check(ccall((:jq_set_kernel, libjq), Cint, (Ptr{Cvoid}, Int32), wa.handle, kernel))
set_time_segments!(wa::Working_Arrays_B200, nseg::Integer) = jq_check(ccall((:jq_set_time_segments, libjq), Cint, (Ptr{Cvoid}, Int32), wa.handle, nseg))
# one Julia process per GPU: rank 0 creates the id, every rank attaches (section 5 of INTEGRATION.md)
comm_unique_id() = (id = zeros(UInt8, 128); jq_check(ccall((:jq_comm_unique_id, libjq), Cint, (Ptr{UInt8},), id)); id)
comm_init!(wa::Working_Arrays_B200, rank::Integer, nranks::Integer, id::Vector{UInt8}) =
    jq_check(ccall((:jq_comm_init, libjq), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}), wa.handle, rank, nranks, id))
# every rank passes the same pcof: the ranks share out ONE evaluation (time segments of kernel 7), bit-identical result everywhere
comm_set_cooperative!(wa::Working_Arrays_B200, on::Bool = true) =
    jq_check(ccall((:jq_comm_set_cooperative, libjq), Cint, (Ptr{Cvoid}, Int32), wa.handle, on ? 1 : 0))
