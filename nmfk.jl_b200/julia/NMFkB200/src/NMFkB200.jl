# NMFkB200.jl - drop-in for the factorization hot path of NMFk.jl on B200 GPUs.
#
# Same signatures and return shapes as the reference for this path
#   NMFk.NMFmultiplicative   (NMFk.jl/src/NMFkMultiplicative.jl:24, :129 for the distributed method's stop rule)
#   NMFk.execute_singlerun   (NMFk.jl/src/NMFkExecute.jl:714,729)   method=:simple and method=:nmf, algorithm=:multdiv / :multmse
#   NMFk.execute_run         (NMFk.jl/src/NMFkExecute.jl:483)
#   NMFk.execute             (NMFk.jl/src/NMFkExecute.jl:178, 236)  including the JLD result cache (load / save / loadonly)
#   NMFk.robustkmeans        (NMFk.jl/src/NMFkCluster.jl:138, 172)
# and nothing else.  All numerics happen in libnmfk_b200.so (hand-written CUDA for sm_100a) through the C ABI declared in
# include/nmfk_b200.h; this file only marshals arguments with `ccall`.
# Random initial factors are drawn HERE with Julia's RNG in the reference's order (W = rand(n,k) only if Winit is empty, then
# H = rand(k,m) only if Hinit is empty; restart i seeded seed+i), so a run with a given `seed` starts from exactly the factors
# the reference would start from.
#
# STATUS: EXPERIMENTAL.  No Julia runtime exists in the build / test environment of this repository, so this file has never
# been executed there; every call below is mirrored 1:1 by the Python ctypes host (nmfk.jl_b200/python/nmfk_b200/api.py,
# cache.py, dist.py), which is what the parity tests drive.  INTEGRATION.md lists what a first run under Julia should check.
module NMFkB200

import Random
import Libdl
import Statistics

const libnmfk = get(ENV, "NMFK_B200_LIB", joinpath(@__DIR__, "..", "..", "..", "lib", "libnmfk_b200.so"))

const NMFK_F32 = Cint(0)
const NMFK_F64 = Cint(1)

# mirrors `struct nmfk_params` (include/nmfk_b200.h, ABI version 2)
struct Params
	tol::Cdouble
	tolOF::Cdouble
	eps_clamp::Cdouble
	weight::Cdouble
	maxiter::Cint
	maxbaditers::Cint
	maxreattempts::Cint
	stopconv::Cint
	check_every::Cint
	Wfixed::Cint
	Hfixed::Cint
	normalize::Cint
	iter_limit::Cint
	engine::Cint
	clusterWmatrix::Cint
	stop_rule::Cint
	variant::Cint
	reserved::Cint
end

"Keyword arguments of the reference -> nmfk_params; unknown keywords are tolerated like the `kw...` sink of NMFkMultiplicative.jl:24"
function makeparams(; tol=1e-19, tolOF=1e-3, weight=1, maxiter=10000, maxbaditers=10, maxreattempts=2, stopconv=1000, Wfixed=false, Hfixed=false, normalize=1, engine=0, clusterWmatrix=false, stop_rule=0, method::Symbol=:simple, algorithm::Symbol=:multdiv, kw...)
	variant = 0
	if method == :nmf
		# the reference swaps the names (NMFkExecute.jl:765-768): :multdiv = MultUpdate(obj=:mse), :multmse = MultUpdate(obj=:div)
		algorithm in (:multdiv, :multmse) || error("NMFkB200: method=:nmf covers algorithm=:multdiv and :multmse (NMF.MultUpdate) only")
		variant = algorithm == :multdiv ? 1 : 3
	elseif method == :sparsity
		variant = 2 # NMFsparsity (NMFkSparsity.jl); its own options travel through setsparsity! (called by the entry points)
	elseif method != :simple
		error("NMFkB200 covers method=:simple, :sparsity and :nmf with algorithm=:multdiv or :multmse; use NMFk for $(method)")
	end
	w = typeof(weight) <: Number ? weight : 1 # array weights are installed on the context (setweight!)
	return Params(tol, tolOF, eps(Float64), w, maxiter, maxbaditers, maxreattempts, stopconv, 10, Wfixed, Hfixed, normalize, 0, engine, clusterWmatrix, stop_rule, variant, 0)
end

dtypecode(::Type{Float32}) = NMFK_F32
dtypecode(::Type{Float64}) = NMFK_F64

function check(status::Integer, ctx::Ptr{Cvoid}=C_NULL)
	status == 0 && return nothing
	msg = unsafe_string(ccall((:nmfk_last_error, libnmfk), Cstring, (Ptr{Cvoid},), ctx))
	if status == -2
		throw(ErrorException("All matrix entries must be nonnegative!")) # NMFkMultiplicative.jl:4-7
	elseif status == -7
		error("Input array has a zero dimension!") # NMFkExecute.jl:242-244
	end
	error("nmfk_b200 status $(status): $(msg)")
end

mutable struct Context
	h::Ptr{Cvoid}
	function Context(device::Integer=0)
		r = Ref{Ptr{Cvoid}}(C_NULL)
		check(ccall((:nmfk_ctx_create, libnmfk), Cint, (Cint, Ref{Ptr{Cvoid}}), device, r))
		c = new(r[])
		finalizer(x->(x.h != C_NULL && ccall((:nmfk_ctx_destroy, libnmfk), Cint, (Ptr{Cvoid},), x.h); x.h = C_NULL), c)
		return c
	end
end

"NMFpreprocessing! (NMFkMultiplicative.jl:3-22) + normalizevector (:27-31); the caller's X is not modified"
function setX!(c::Context, X::AbstractMatrix{T}; lambda::Number=1e-32, normalizevector::AbstractVector=Vector{T}(undef, 0)) where {T <: Union{Float32,Float64}}
	Xd = Matrix{T}(X) # dense, column-major
	nv = C_NULL
	nvd = Vector{T}(undef, 0)
	if length(normalizevector) == size(Xd, 1)
		nvd = Vector{T}(normalizevector)
		nv = pointer(nvd)
	elseif length(normalizevector) != 0
		error("Length of normalizing vector does not match: $(length(normalizevector)) vs $(size(Xd, 1))") # :30
	end
	GC.@preserve nvd check(ccall((:nmfk_set_X, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Cint, Cdouble, Ptr{Cvoid}, Cint), c.h, Xd, size(Xd, 1), size(Xd, 2), dtypecode(T), lambda, nv, 0), c.h)
	return nothing
end

"The `weight` keyword when it is an array (NMFkExecute.jl:484): vector of length n, 1 x m, or n x m; a scalar clears it"
function setweight!(c::Context, ::Type{T}, weight) where {T}
	if typeof(weight) <: Number
		check(ccall((:nmfk_set_weight, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64), c.h, C_NULL, 0, 0), c.h)
	else
		w = Matrix{T}(reshape(weight, size(weight, 1), size(weight, 2)))
		check(ccall((:nmfk_set_weight, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64), c.h, w, size(w, 1), size(w, 2)), c.h)
	end
	return nothing
end

"Options of NMFsparsity (NMFkSparsity.jl:1): cost_function / beta_divergence, sparsity, lambda"
function setsparsity!(c::Context; cost_function::Symbol=:ed, beta_divergence::Number=-1, sparsity::Number=1, lambda::Number=1e-9, kw...)
	beta = beta_divergence == -1 ? (cost_function == :kl ? 1 : (cost_function == :is ? 0 : 2)) : beta_divergence # :5-22
	check(ccall((:nmfk_set_sparsity_options, libnmfk), Cint, (Ptr{Cvoid}, Cdouble, Cdouble, Cdouble), c.h, beta, sparsity, lambda), c.h)
end

"NMFk.NMFsparsity(X, k; ...) -> (W, H, objvalue)  (NMFkSparsity.jl:1-113)"
function NMFsparsity(X::AbstractMatrix{T}, k::Int; maxiter::Int=100000, tol::Number=1e-19, seed::Number=-1, Winit::AbstractMatrix{T}=Matrix{T}(undef, 0, 0), Hinit::AbstractMatrix{T}=Matrix{T}(undef, 0, 0), ctx::Context=Context(), kw...) where {T <: Union{Float32,Float64}}
	n, m = size(X)
	setX!(ctx, X)
	setsparsity!(ctx; kw...)
	seed != -1 && Random.seed!(seed)
	Wi, Hi = drawinits(T, n, m, k, 1; Winit=Winit, Hinit=Hinit)
	p = makeparams(; maxiter=maxiter, tol=tol, normalize=0, method=:sparsity)
	W = Matrix{T}(undef, n, k); H = Matrix{T}(undef, k, m)
	ssq = Ref{Cdouble}(0); nrm = Ref{Cdouble}(0); it = Ref{Cint}(0); sr = Ref{Cint}(0)
	check(ccall((:nmfk_run_batch, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Params}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Cdouble}, Ref{Cdouble}, Ref{Cint}, Ref{Cint}), ctx.h, k, 1, Wi, Hi, p, W, H, ssq, nrm, it, sr), ctx.h)
	return W, H, ssq[]
end

"Initial factors for nNMF restarts drawn like the reference: W = rand(n,k) only if Winit is empty, then H = rand(k,m) only if Hinit is empty (NMFkMultiplicative.jl:37-55), restart i seeded seed+i (NMFkExecute.jl:536)"
function drawinits(::Type{T}, n::Integer, m::Integer, k::Integer, nNMF::Integer; seed::Integer=-1, Winit::AbstractMatrix=Matrix{T}(undef, 0, 0), Hinit::AbstractMatrix=Matrix{T}(undef, 0, 0), kw...) where {T}
	W = Array{T,3}(undef, n, k, nNMF)
	H = Array{T,3}(undef, k, m, nNMF)
	for i = 1:nNMF
		seed >= 0 && Random.seed!(seed + i)
		if sizeof(Winit) == 0
			W[:, :, i] = rand(n, k)
		else
			@assert size(Winit) == (n, k)
			sum(isnan.(Winit)) > 0 && error("Initial values for the W matrix entries include NaNs!")
			W[:, :, i] = Winit
		end
		if sizeof(Hinit) == 0
			H[:, :, i] = rand(k, m)
		else
			@assert size(Hinit) == (k, m)
			sum(isnan.(Hinit)) > 0 && error("Initial values for the H matrix entries include NaNs!")
			H[:, :, i] = Hinit
		end
	end
	return W, H
end

# ---- batches of restarts (nmfk_batch_*) -------------------------------------------------------------------------------
mutable struct Batch
	h::Ptr{Cvoid}
	ctx::Context
	k::Int
	R::Int
	function Batch(c::Context, k::Integer, R::Integer)
		r = Ref{Ptr{Cvoid}}(C_NULL)
		check(ccall((:nmfk_batch_create, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ref{Ptr{Cvoid}}), c.h, k, R, r), c.h)
		b = new(r[], c, k, R)
		finalizer(x->(x.h != C_NULL && x.ctx.h != C_NULL && ccall((:nmfk_batch_destroy, libnmfk), Cint, (Ptr{Cvoid},), x.h); x.h = C_NULL), b)
		return b
	end
end

function setinit!(b::Batch, W::Array{T,3}, H::Array{T,3}) where {T}
	check(ccall((:nmfk_batch_set_init, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), b.h, W, H), b.ctx.h)
end

function solve!(c::Context, bs::Vector{Batch}, p::Params)
	hs = [b.h for b in bs]
	check(ccall((:nmfk_solve, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Ptr{Cvoid}}, Cint, Ref{Params}), c.h, hs, length(hs), p), c.h)
end

function getbatch(b::Batch, ::Type{T}, n::Integer, m::Integer) where {T}
	W = Array{T,3}(undef, n, b.k, b.R); H = Array{T,3}(undef, b.k, m, b.R)
	ssq = Vector{Cdouble}(undef, b.R); nrm = Vector{Cdouble}(undef, b.R); it = Vector{Cint}(undef, b.R); sr = Vector{Cint}(undef, b.R)
	check(ccall((:nmfk_batch_get, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ptr{Cint}), b.h, W, H, ssq, nrm, it, sr), b.ctx.h)
	return W, H, ssq, nrm, it, sr
end

"NMFk.NMFmultiplicative(X, k; ...) -> (W, H, objvalue)  (NMFkMultiplicative.jl:24-127)"
function NMFmultiplicative(X::AbstractMatrix{T}, k::Int; seed::Int=-1, lambda::Number=1e-32, maxiter::Int=1000000, weight=1, Winit::AbstractMatrix{T}=Matrix{T}(undef, 0, 0), Hinit::AbstractMatrix{T}=Matrix{T}(undef, 0, 0), normalizevector::AbstractVector{T}=Vector{T}(undef, 0), ctx::Context=Context(), kw...) where {T <: Union{Float32,Float64}}
	n, m = size(X)
	setX!(ctx, X; lambda=lambda, normalizevector=normalizevector)
	setweight!(ctx, T, weight)
	seed >= 0 && Random.seed!(seed)
	Wi, Hi = drawinits(T, n, m, k, 1; Winit=Winit, Hinit=Hinit)
	p = makeparams(; maxiter=maxiter, normalize=0, weight=weight, kw...)
	W = Matrix{T}(undef, n, k); H = Matrix{T}(undef, k, m)
	ssq = Ref{Cdouble}(0); nrm = Ref{Cdouble}(0); it = Ref{Cint}(0); sr = Ref{Cint}(0)
	check(ccall((:nmfk_run_batch, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Params}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Cdouble}, Ref{Cdouble}, Ref{Cint}, Ref{Cint}), ctx.h, k, 1, Wi, Hi, p, W, H, ssq, nrm, it, sr), ctx.h)
	return W, H, ssq[]
end

"NMFk.NMFmultiplicative(X::DArray, k; ...) (NMFkMultiplicative.jl:129-197): the distributed method's own stop rule (no tolOF / baditers / reattempts, no weight, stopconv=10000) on one GPU; rows of X over several GPUs: nmfk_ctx_comm_init + the same flag"
NMFmultiplicative_darray(X::AbstractMatrix, k::Int; stopconv::Int=10000, kw...) = NMFmultiplicative(X, k; stop_rule=1, stopconv=stopconv, filter(p->p.first != :weight, kw)...)

"NMFk.execute_singlerun(X, nk; ...) -> (W, H, objvalue)  (NMFkExecute.jl:729-807)"
function execute_singlerun(X::AbstractMatrix{T}, nk::Int; seed::Int=-1, clusterWmatrix::Bool=false, modifymatrices::Bool=true, weight=1, normalizevector::AbstractVector{T}=Vector{T}(undef, 0), ctx::Context=Context(), kw...) where {T <: Union{Float32,Float64}}
	n, m = size(X)
	setX!(ctx, X; normalizevector=normalizevector)
	setweight!(ctx, T, weight)
	seed >= 0 && Random.seed!(seed)
	Wi, Hi = drawinits(T, n, m, nk, 1; kw...)
	p = makeparams(; normalize=(modifymatrices ? (clusterWmatrix ? 2 : 1) : 0), weight=weight, kw...) # :795-805
	W = Matrix{T}(undef, n, nk); H = Matrix{T}(undef, nk, m)
	ssq = Ref{Cdouble}(0); nrm = Ref{Cdouble}(0); it = Ref{Cint}(0); sr = Ref{Cint}(0)
	check(ccall((:nmfk_run_batch, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Params}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Cdouble}, Ref{Cdouble}, Ref{Cint}, Ref{Cint}), ctx.h, nk, 1, Wi, Hi, p, W, H, ssq, nrm, it, sr), ctx.h)
	return W, H, convert(T, nrm[])
end

"NMFk.execute_run(X, nk, nNMF; ...) -> (Wa, Ha, phi_final, minsilhouette, aic)  (NMFkExecute.jl:483-711)"
function execute_run(X::AbstractMatrix{T}, nk::Int, nNMF::Int; clusterWmatrix::Bool=false, acceptratio::Number=1, acceptfactor::Number=Inf, best::Bool=true, nanaction::Symbol=:zeroed, seed::Int=-1, weight=1, normalizevector::AbstractVector{T}=Vector{T}(undef, 0), ctx::Context=Context(), kw...) where {T <: Union{Float32,Float64}}
	n, m = size(X)
	setX!(ctx, X; normalizevector=normalizevector)
	setweight!(ctx, T, weight)
	get(kw, :method, :simple) == :sparsity && setsparsity!(ctx; kw...)
	modifymatrices = !(haskey(kw, :Wfixed) || haskey(kw, :Hfixed)) # NMFkExecute.jl:486-489
	Wi, Hi = drawinits(T, n, m, nk, nNMF; seed=seed, kw...)
	# clusterWmatrix is consumed here and NOT forwarded to the restarts (:516-540): they keep the H-row normalisation
	p = makeparams(; normalize=(modifymatrices ? 1 : 0), clusterWmatrix=clusterWmatrix, weight=weight, kw...)
	if acceptratio == 1 && acceptfactor == Inf && best && nanaction == :zeroed
		Wa = Matrix{T}(undef, n, nk); Ha = Matrix{T}(undef, nk, m)
		phi = Ref{Cdouble}(0); rob = Ref{Cdouble}(0); aic = Ref{Cdouble}(0); tot = Ref{Int64}(0)
		check(ccall((:nmfk_execute_run, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ref{Params}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Cdouble}, Ref{Cdouble}, Ref{Cdouble}, Ref{Int64}), ctx.h, nk, nNMF, Wi, Hi, 0, p, Wa, Ha, phi, rob, aic, tot), ctx.h)
		return Wa, Ha, convert(T, phi[]), (nk > 1 ? convert(T, rob[]) : 1), aic[]
	end
	# any other keyword combination: the same device calls composed here (like api.py::execute_run)
	b = Batch(ctx, nk, nNMF)
	setinit!(b, Wi, Hi)
	solve!(ctx, [b], p)
	Wpre, Hpre, _, objpre, _, _ = getbatch(b, T, n, m) # Wbest / Hbest are copied before the NaN pass (:549-550)
	order = Vector{Cint}(undef, nNMF); nkept = Ref{Cint}(0)
	check(ccall((:nmfk_batch_select, libnmfk), Cint, (Ptr{Cvoid}, Cdouble, Cdouble, Cint, Ptr{Cint}, Ref{Cint}), b.h, acceptratio, acceptfactor, (nanaction == :removed ? 1 : 0), order, nkept), ctx.h)
	nkept[] > 0 || error("NMF solutions removed based on various criteria: none remain")
	R = Int(nkept[])
	labels = Matrix{Cint}(undef, nk, R); sil = Matrix{Cdouble}(undef, nk, R); csil = Vector{Cdouble}(undef, nk); rob = Ref{Cdouble}(1)
	ord = Vector{Cint}(undef, nNMF); ccols = Ref{Cint}(0)
	check(ccall((:nmfk_batch_cluster, libnmfk), Cint, (Ptr{Cvoid}, Cint, Ptr{Cint}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ptr{Cvoid}, Ref{Cint}), b.h, clusterWmatrix, ord, labels, sil, csil, rob, C_NULL, ccols), ctx.h)
	Wall, Hall, _, _, _, _ = getbatch(b, T, n, m)
	bi = sortperm(convert.(T, objpre))[1]
	Wbest = Wpre[:, :, bi]; Hbest = Hpre[:, :, bi]
	minsilhouette = 1
	if nk > 1
		ci = labels[:, 1]
		Wbest = Wall[:, ci, bi]; Hbest = Hall[ci, :, bi] # :631-635 reads the stored (NaN-zeroed, possibly centroid-overwritten) best
		Wm = Matrix{T}(undef, n, nk); Hm = Matrix{T}(undef, nk, m); Wv = Matrix{T}(undef, n, nk); Hv = Matrix{T}(undef, nk, m)
		check(ccall((:nmfk_batch_cluster_means, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cint}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), b.h, ord, labels, Wm, Hm, Wv, Hv), ctx.h)
		minsilhouette = convert(T, rob[])
		Wa, Ha = Wm, Hm
	else
		order_full = sortperm(convert.(T, objpre))
		first = minimum(findall(in(order[1:R] .+ 1), order_full)) # idxsol is a positional mask applied to WBig itself (:646-650)
		Wa = Wall[:, :, first]; Ha = Hall[:, :, first]
	end
	if best
		Wa, Ha = Wbest, Hbest
	end
	phi = Ref{Cdouble}(0)
	check(ccall((:nmfk_fit, libnmfk), Cint, (Ptr{Cvoid}, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Cdouble}), ctx.h, nk, Wa, Ha, phi), ctx.h)
	numobservations = sum(.!isnan.(X))
	aic = 2 * (length(Wa) + length(Ha)) + numobservations * log(phi[] / numobservations) # :697-708
	return Wa, Ha, convert(T, phi[]), minsilhouette, aic
end

"signalorder (NMFkPostprocess.jl:148-158)"
function signalorder(W::AbstractMatrix, H::AbstractMatrix)
	k = size(W, 2)
	return sortperm([sum(W[:, i:i] * H[i:i, :]) for i = 1:k]; rev=true)
end

normnan(A) = sqrt(sum(A[.!isnan.(A)] .^ 2))

"NMFk.execute(X, nk::Integer, nNMF; ...) -> (W[:,so], H[so,:], fitquality, robustness, aic)  (NMFkExecute.jl:236-329) with the JLD result cache: same file names and keys as the reference, so existing result directories load unchanged"
function execute(X::AbstractMatrix{T}, nk::Integer, nNMF::Integer=10; resultdir::AbstractString=".", casefilename::AbstractString="nmfk", loadonly::Bool=false, load::Bool=true, save::Bool=true, ordersignals::Bool=true, kw...) where {T <: Union{Float32,Float64}}
	.*(size(X)...) == 0 && error("Input array has a zero dimension! Array size=$(size(X))")
	runflag = true
	if loadonly
		load = true; save = false; runflag = false
	end
	JLD = (load || save) ? Base.require(Base.PkgId(Base.UUID("4138dd39-2aa7-5051-a626-17a0bb65d9c8"), "JLD")) : nothing
	local W, H, fitquality, robustness, aic
	execute_ordersignals = true
	if load
		filename = joinpath(resultdir, "$(casefilename)_$(size(X,1))_$(size(X,2))_$(nk)_$(nNMF).jld")
		if !isfile(filename)
			filename = joinpath(resultdir, "$(casefilename)-$(nk)-$(nNMF).jld") # old filename convention (:266-269)
		end
		if isfile(filename)
			W, H, fitquality, robustness, aic = JLD.load(filename, "W", "H", "fit", "robustness", "aic")
			if size(W) == (size(X, 1), nk) && size(H) == (nk, size(X, 2))
				fit = normnan(X .- W * H)
				if abs(fit - fitquality) > eps(Float16)
					fitquality = fit; save = true
				else
					save = false
				end
				runflag = false
			end
		elseif loadonly
			W = Matrix{T}(undef, 0, 0); H = Matrix{T}(undef, 0, 0); fitquality = Inf; robustness = -1; aic = -Inf
			execute_ordersignals = false
		end
	end
	if haskey(kw, :Wfixed) || haskey(kw, :Hfixed)
		ordersignals = false # :305-307
	end
	if runflag
		W, H, fitquality, robustness, aic = execute_run(X, Int(nk), Int(nNMF); kw...)
	end
	so = execute_ordersignals ? (ordersignals ? signalorder(W, H) : collect(axes(W, 2))) : Int64[]
	if save
		mkpath(resultdir)
		JLD.save(joinpath(resultdir, "$(casefilename)_$(size(X,1))_$(size(X,2))_$(nk)_$(nNMF).jld"), "W", W[:, so], "H", H[so, :], "fit", fitquality, "robustness", robustness, "aic", aic)
	end
	return W[:, so], H[so, :], fitquality, robustness, aic
end

"getk (NMFkPostprocess.jl:7-41) through the C ABI"
function getk(nkrange, robustness::AbstractVector, cutoff::Number=0.5; strict::Bool=true)
	ks = collect(Cint, nkrange); rb = collect(Cdouble, robustness)
	r = ccall((:nmfk_getk, libnmfk), Cint, (Ptr{Cint}, Ptr{Cdouble}, Cint, Cdouble, Cint), ks, rb, length(ks), cutoff, strict)
	return r < 0 ? nothing : Int(r)
end

"NMFk.execute(X, nkrange, nNMF; cutoff=0.5, ...) -> (W, H, fitquality, robustness, aic, kopt)  (NMFkExecute.jl:178-233).  Without the cache (load=false, save=false) all k are solved concurrently on the GPU by one call; with it, k by k like the reference"
function execute(X::AbstractMatrix{T}, nkrange::Union{Vector{Int},AbstractUnitRange{Int}}, nNMF::Integer=10; cutoff::Number=0.5, clusterWmatrix::Bool=false, load::Bool=true, save::Bool=true, seed::Int=-1, weight=1, normalizevector::AbstractVector{T}=Vector{T}(undef, 0), ctx::Context=Context(), kw...) where {T <: Union{Float32,Float64}}
	.*(size(X)...) == 0 && error("Input array has a zero dimension! Array size=$(size(X))")
	n, m = size(X)
	ks = collect(Cint, nkrange)
	nks = length(ks)
	maxk = maximum(ks)
	W = Vector{Matrix{T}}(undef, maxk); H = Vector{Matrix{T}}(undef, maxk)
	fitquality = zeros(T, maxk); robustness = zeros(T, maxk); aic = zeros(T, maxk)
	fitquality[1] = Inf; robustness[1] = -1 # NMFkExecute.jl:200-201
	if load || save
		for k in ks
			W[k], H[k], fitquality[k], robustness[k], aic[k] = execute(X, Int(k), nNMF; clusterWmatrix=clusterWmatrix, load=load, save=save, seed=seed, weight=weight, normalizevector=normalizevector, ctx=ctx, kw...)
		end
		if all(isinf.(fitquality[ks]))
			return W, H, fitquality, robustness, aic, 0
		end
		for k in ks
			fitquality[k] = normnan(X .- W[k] * H[k]) # :211-222
		end
		return W, H, fitquality, robustness, aic, getk(ks, robustness[ks], cutoff)
	end
	setX!(ctx, X; normalizevector=normalizevector)
	setweight!(ctx, T, weight)
	modifymatrices = !(haskey(kw, :Wfixed) || haskey(kw, :Hfixed))
	p = makeparams(; normalize=(modifymatrices ? 1 : 0), clusterWmatrix=clusterWmatrix, weight=weight, kw...)
	inits = [drawinits(T, n, m, Int(k), nNMF; seed=seed, kw...) for k in ks]
	Wo = [Matrix{T}(undef, n, Int(k)) for k in ks]
	Ho = [Matrix{T}(undef, Int(k), m) for k in ks]
	fit = Vector{Cdouble}(undef, nks); rob = Vector{Cdouble}(undef, nks); aicv = Vector{Cdouble}(undef, nks)
	kopt = Ref{Cint}(0); tot = Ref{Int64}(0)
	GC.@preserve inits Wo Ho begin
		Wip = [pointer(i[1]) for i in inits]; Hip = [pointer(i[2]) for i in inits]
		Wop = [pointer(w) for w in Wo]; Hop = [pointer(h) for h in Ho]
		check(ccall((:nmfk_execute, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cint}, Cint, Cint, Ptr{Ptr{T}}, Ptr{Ptr{T}}, UInt64, Ref{Params}, Cdouble, Ptr{Ptr{T}}, Ptr{Ptr{T}}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cint}, Ref{Int64}), ctx.h, ks, nks, nNMF, Wip, Hip, 0, p, cutoff, Wop, Hop, fit, rob, aicv, kopt, tot), ctx.h)
	end
	for (i, k) in enumerate(ks)
		W[k] = Wo[i]; H[k] = Ho[i]
		fitquality[k] = fit[i]; robustness[k] = (k > 1 ? rob[i] : 1); aic[k] = aicv[i]
	end
	ko = kopt[] < 0 ? nothing : Int(kopt[]) # getk returns `nothing` when no k passes the cutoff
	return W, H, fitquality, robustness, aic, ko
end

# ---- restart-sharded sweep over several GPUs (the reference's pmap over restarts, NMFkExecute.jl:511-526) ------------------
"128-byte NCCL id: make it on one worker and send it to the others (e.g. with remotecall_fetch)"
function comm_unique_id()
	id = Vector{UInt8}(undef, 128)
	check(ccall((:nmfk_comm_unique_id, libnmfk), Cint, (Ptr{UInt8},), id))
	return id
end

"One Julia worker per GPU: every worker calls this with its rank, then execute_sharded with the same arguments"
sweep_comm_init!(c::Context, nranks::Integer, rank::Integer, id::Vector{UInt8}) = check(ccall((:nmfk_ctx_sweep_comm_init, libnmfk), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{UInt8}), c.h, nranks, rank, id), c.h)

"execute(X, nkrange, nNMF = nranks * R_local) with the restarts sharded over the workers (nmfk_sweep); every worker returns the full result"
function execute_sharded(c::Context, X::AbstractMatrix{T}, nkrange, R_local::Integer; rank::Integer, seed::Integer=0, cutoff::Number=0.5, kw...) where {T <: Union{Float32,Float64}}
	n, m = size(X)
	setX!(c, X)
	ks = collect(Cint, nkrange); nks = length(ks)
	p = makeparams(; kw...)
	# this worker's restarts rank*R_local+1 .. (rank+1)*R_local of every k, drawn with Julia's RNG seeded like the reference
	inits = [begin
		W = Array{T,3}(undef, n, Int(k), R_local); H = Array{T,3}(undef, Int(k), m, R_local)
		for i = 1:R_local
			Random.seed!(seed + rank * R_local + i); W[:, :, i] = rand(n, Int(k)); H[:, :, i] = rand(Int(k), m)
		end
		(W, H)
	end for k in ks]
	Wo = [Matrix{T}(undef, n, Int(k)) for k in ks]; Ho = [Matrix{T}(undef, Int(k), m) for k in ks]
	fit = Vector{Cdouble}(undef, nks); rob = Vector{Cdouble}(undef, nks); aicv = Vector{Cdouble}(undef, nks)
	kopt = Ref{Cint}(0); tot = Ref{Int64}(0); totl = Ref{Int64}(0)
	GC.@preserve inits Wo Ho begin
		Wip = [pointer(i[1]) for i in inits]; Hip = [pointer(i[2]) for i in inits]
		Wop = [pointer(w) for w in Wo]; Hop = [pointer(h) for h in Ho]
		check(ccall((:nmfk_sweep, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cint}, Cint, Cint, Ptr{Ptr{T}}, Ptr{Ptr{T}}, UInt64, Ref{Params}, Cdouble, Ptr{Ptr{T}}, Ptr{Ptr{T}}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cint}, Ref{Int64}, Ref{Int64}), c.h, ks, nks, R_local, Wip, Hip, 0, p, cutoff, Wop, Hop, fit, rob, aicv, kopt, tot, totl), c.h)
	end
	return Dict(Int(k)=>Wo[i] for (i, k) in enumerate(ks)), Dict(Int(k)=>Ho[i] for (i, k) in enumerate(ks)), fit, rob, aicv, (kopt[] < 0 ? nothing : Int(kopt[]))
end

# ---- robustkmeans (NMFkCluster.jl:138-246) ---------------------------------------------------------------------------------
struct KmeansResult
	centers::Matrix{Float64}
	assignments::Vector{Int}
	costs::Vector{Float64}
	counts::Vector{Int}
	totalcost::Float64
	iterations::Int
	converged::Bool
end

"k-means++ seeding like Clustering.kmeans' default (squared Euclidean costs), drawn from Julia's RNG; 0-based indices"
function kmpp_seeds(X::AbstractMatrix, k::Integer)
	n = size(X, 2)
	seeds = Vector{Cint}(undef, k)
	seeds[1] = rand(1:n) - 1
	cost = vec(sum((X .- X[:, seeds[1]+1]) .^ 2; dims=1))
	for q = 2:k
		r = rand() * sum(cost); acc = 0.0; j = n
		for i = 1:n
			acc += cost[i]
			if acc >= r
				j = i; break
			end
		end
		seeds[q] = j - 1
		cost = min.(cost, vec(sum((X .- X[:, j]) .^ 2; dims=1)))
	end
	return seeds
end

"NMFk.robustkmeans(X, k, repeats; ...) (NMFkCluster.jl:172-246): all repeats run concurrently on the GPU"
function robustkmeans(X::AbstractMatrix, k::Integer, repeats::Integer=1000; maxiter::Integer=1000, tol::Number=1e-32, compute_silhouettes_flag::Bool=false, ctx::Context=Context(), kw...)
	Xd = Matrix{Float64}(X)
	d, N = size(Xd)
	seeds = hcat([kmpp_seeds(Xd, k) for _ = 1:repeats]...)
	assign = Vector{Cint}(undef, N); centers = Matrix{Cdouble}(undef, d, k); costs = Vector{Cdouble}(undef, N); counts = Vector{Cint}(undef, k)
	sil = zeros(Cdouble, N); tc = Ref{Cdouble}(0); it = Ref{Cint}(0); cv = Ref{Cint}(0); best = Ref{Cint}(0); nempty = Ref{Cint}(0)
	check(ccall((:nmfk_robustkmeans, libnmfk), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cint, Cint, Cint, Cint, Ptr{Cint}, Cint, Cdouble, Cint, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ref{Cdouble}, Ref{Cint}, Ref{Cint}, Ptr{Cdouble}, Ref{Cint}, Ref{Cint}), ctx.h, Xd, d, N, k, repeats, seeds, maxiter, tol, compute_silhouettes_flag, assign, centers, costs, counts, tc, it, cv, sil, best, nempty), ctx.h)
	nc = length(unique(assign))
	nc < k && @warn("Robust k-means analysis could not find $k clusters! Only $(nc) clusters were found.")
	sc = KmeansResult(centers[:, 1:nc], Int.(assign), costs, Int.(counts[1:nc]), tc[], it[], cv[] != 0)
	return compute_silhouettes_flag ? (sc, sil) : sc
end

"NMFk.robustkmeans(X, krange, repeats; best_method=:worst_cliff) (NMFkCluster.jl:138-170)"
function robustkmeans(X::AbstractMatrix, krange::Union{AbstractUnitRange{Int},AbstractVector{Int64}}, repeats::Int=1000; best_method::Symbol=:worst_cliff, kw...)
	krange[1] >= size(X, 2) && return nothing
	cresult = Vector{Any}(undef, length(krange)); worst_silhouette = Vector{Float64}(undef, length(krange)); cluster_silhouettes = Vector{Any}(undef, length(krange))
	for (i, k) in enumerate(krange)
		k >= size(X, 2) && continue
		cresult[i], silhouettes = robustkmeans(X, k, repeats; kw..., compute_silhouettes_flag=true)
		cluster_silhouettes[i] = map(j->Statistics.mean(silhouettes[cresult[i].assignments .== j]), unique(cresult[i].assignments))
		worst_silhouette[i] = minimum(silhouettes)
	end
	if best_method == :worst_cliff
		ki = last(findmax(map(i->worst_silhouette[i] - worst_silhouette[i+1], eachindex(krange)[begin:end-1]))) + 1
	elseif best_method == :worst_cluster_cliff
		ki = last(findmax(map(i->minimum(cluster_silhouettes[i]) - minimum(cluster_silhouettes[i+1]), eachindex(krange)[begin:end-1]))) + 1
	else
		error("Unknown method: best_method must be :worst_cliff or :worst_cluster_cliff")
	end
	return cresult[ki]
end

end
