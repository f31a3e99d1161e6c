# NnSdpB200.jl -- Julia host side of libnnsdp_b200.so (C ABI: include/nnsdp_b200.h).
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: Julia is not installed in the build image.  The file is kept
# deliberately thin (ccall + array reshapes) so that a reviewer can vouch for it against the header;
# the same ABI is exercised by the ctypes binding (nn-sdp_b200/nnsdp_b200/_lib.py) in tests/.
#
# It plugs into the reference at its three dispatch points without touching solveQuery / runQuery:
#   * makeIntervalsInfo(x1min, x1max, ffnet, ::IntervalsB200)      src/Intervals/Intervals.jl:38-49
#   * makeZin / makeZac / makeZout for numeric gamma                src/Qc/input.jl:19, activ.jl:30, output.jl:52,64
#   * makeCliques (index sets), assembleCliqueBlocks (batched)      src/Methods/chordal_cliques.jl:13-59
# Usage from the reference's module tree:   include("NnSdpB200.jl"); using .NnSdpB200
module NnSdpB200

using LinearAlgebra
using SparseArrays
using ..MyMath
using ..MyNeuralNetwork
using ..Intervals
using ..Qc
using ..Methods

const LIB = get(ENV, "NNSDP_B200_LIB", joinpath(@__DIR__, "..", "lib", "libnnsdp_b200.so"))

const OUT_SAFETY, OUT_HPLANE, OUT_CIRCLE, OUT_ELLIPSOID = Int32(0), Int32(1), Int32(2), Int32(3)

# mirrors `nnsdp_sizes` (14 x int64)
struct Sizes
  K::Int64; Zdim::Int64; acdim::Int64; xtot::Int64; lamdim::Int64; secdim::Int64
  n_in::Int64; n_out::Int64; sdim::Int64; ncliques::Int64; sum_ck::Int64; sum_ck_sq::Int64
  sum_dk::Int64; max_ck::Int64
end

# mirrors `nnsdp_query_inputs` (13 (pointer, stride) pairs; out_kind/reserved after the 9th)
struct QueryInputs
  x1min::Ptr{Float64}; x1min_stride::Int64
  x1max::Ptr{Float64}; x1max_stride::Int64
  ymin::Ptr{Float64}; ymin_stride::Int64
  ymax::Ptr{Float64}; ymax_stride::Int64
  smin::Ptr{Float64}; smin_stride::Int64
  smax::Ptr{Float64}; smax_stride::Int64
  gamma_in::Ptr{Float64}; gamma_in_stride::Int64
  gamma_bnd::Ptr{Float64}; gamma_bnd_stride::Int64
  gamma_sec::Ptr{Float64}; gamma_sec_stride::Int64
  out_kind::Int32; reserved::Int32
  out_S::Ptr{Float64}; out_S_stride::Int64
  out_vec::Ptr{Float64}; out_vec_stride::Int64
  out_invP::Ptr{Float64}; out_invP_stride::Int64
  gamma_out::Ptr{Float64}; gamma_out_stride::Int64
end

# mirrors `nnsdp_packed_cell`
struct PackedCell
  kind::Int32; blk::Int32
  row0::Int64; col0::Int64; nrows::Int64; ncols::Int64; offset::Int64
  always::Int32; reserved::Int32
end
const CELL_WINDOW, CELL_DIAG, CELL_BAND, CELL_RECT = Int32(1), Int32(2), Int32(3), Int32(4)
const FORMAT_BLOCKS, FORMAT_DENSE_Z, FORMAT_PACKED = Int32(0), Int32(1), Int32(2)

# the hand-mirrored structs must have the layout of the C header (include/nnsdp_b200.h); checked when the module loads
function __init__()
  @assert sizeof(Sizes) == 14 * 8 "nnsdp_sizes layout drifted"
  @assert sizeof(QueryInputs) == 13 * 16 + 8 "nnsdp_query_inputs layout drifted"
  @assert fieldoffset(QueryInputs, 19) == 9 * 16 "nnsdp_query_inputs.out_kind offset drifted"   # out_kind is field 19
  @assert sizeof(PackedCell) == 56 "nnsdp_packed_cell layout drifted"
  @assert ccall((:nnsdp_version, LIB), Int32, ()) >= 100
end

lasterror() = unsafe_string(ccall((:nnsdp_last_error, LIB), Cstring, ()))
check(status::Int32) = status == 0 ? nothing : error("nnsdp_b200 error $(status): $(lasterror())")

# ---- handles --------------------------------------------------------------------------------------
mutable struct Context
  h::Ptr{Cvoid}
  function Context(devices::Vector{Int} = [0])
    out = Ref{Ptr{Cvoid}}(C_NULL)
    ids = Int32.(devices)
    check(ccall((:nnsdp_ctx_create, LIB), Int32, (Int32, Ptr{Int32}, Ptr{Ptr{Cvoid}}), length(ids), ids, out))
    ctx = new(out[])
    finalizer(c -> ccall((:nnsdp_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), c.h), ctx)
  end
end

mutable struct DeviceNet
  h::Ptr{Cvoid}
  ctx::Context
  ffnet::FeedFwdNet
  function DeviceNet(ctx::Context, ffnet::FeedFwdNet)
    # Ms[k] is a dense column-major Matrix{Float64} [W_k b_k]: passed as-is (MyNeuralNetwork.jl:12-27)
    Ms = [Matrix{Float64}(M) for M in ffnet.Ms]
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve Ms begin
      ptrs = [pointer(M) for M in Ms]
      check(ccall((:nnsdp_net_upload, LIB), Int32,
                  (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Ptr{Float64}}, Ptr{Ptr{Cvoid}}),
                  ctx.h, ffnet.K, Int64.(ffnet.xdims), ptrs, out))
    end
    net = new(out[], ctx, ffnet)
    finalizer(n -> ccall((:nnsdp_net_destroy, LIB), Int32, (Ptr{Cvoid},), n.h), net)
  end
end

function sizes(net::DeviceNet, β::Int)
  s = Ref{Sizes}()
  check(ccall((:nnsdp_query_sizes, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{Sizes}), net.h, β, s))
  return s[]
end

# ---- dispatch point 1: interval bounds -----------------------------------------------------------
struct IntervalsB200 <: IntervalsMethod
  net::DeviceNet
end

# Same return type as intervalsWorstCase (src/Intervals/intervals_easy.jl:2-37)
function Intervals.makeIntervalsInfo(x1min::VecReal, x1max::VecReal, ffnet::FeedFwdNet, method::IntervalsB200)
  sz = sizes(method.net, 0)
  lo, hi = Vector{Float64}(x1min), Vector{Float64}(x1max)
  xmin, xmax = zeros(sz.xtot), zeros(sz.xtot)
  amin, amax = zeros(sz.acdim), zeros(sz.acdim)
  check(ccall((:nnsdp_bounds_ibp, LIB), Int32,
              (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
              method.net.ctx.h, method.net.h, 1, lo, hi, xmin, xmax, amin, amax))
  xoff = cumsum([0; ffnet.xdims])
  aoff = cumsum([0; ffnet.xdims[2:end-1]])
  x_intvs = [(xmin[xoff[k]+1:xoff[k+1]], xmax[xoff[k]+1:xoff[k+1]]) for k in 1:(ffnet.K+1)]
  acx_intvs = [(amin[aoff[k]+1:aoff[k+1]], amax[aoff[k]+1:aoff[k+1]]) for k in 1:(ffnet.K-1)]
  return IntervalsInfo(ffnet=ffnet, x_intvs=x_intvs, acx_intvs=acx_intvs)
end

# CROWN bounds: the reference's default method (IntervalsAutoLirpa -> intervalsAutoLirpaSliced,
# src/Intervals/intervals_auto_lirpa.jl:44-63) without the K ONNX / Python round trips, FP64 on the device.
struct IntervalsCrownB200 <: IntervalsMethod
  net::DeviceNet
end

function Intervals.makeIntervalsInfo(x1min::VecReal, x1max::VecReal, ffnet::FeedFwdNet, method::IntervalsCrownB200)
  sz = sizes(method.net, 0)
  lo, hi = Vector{Float64}(x1min), Vector{Float64}(x1max)
  xmin, xmax = zeros(sz.xtot), zeros(sz.xtot)
  amin, amax = zeros(sz.acdim), zeros(sz.acdim)
  check(ccall((:nnsdp_bounds_crown, LIB), Int32,
              (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
              method.net.ctx.h, method.net.h, 1, lo, hi, xmin, xmax, amin, amax))
  xoff = cumsum([0; ffnet.xdims])
  aoff = cumsum([0; ffnet.xdims[2:end-1]])
  x_intvs = [(xmin[xoff[k]+1:xoff[k+1]], xmax[xoff[k]+1:xoff[k+1]]) for k in 1:(ffnet.K+1)]
  acx_intvs = [(amin[aoff[k]+1:aoff[k+1]], amax[aoff[k]+1:aoff[k+1]]) for k in 1:(ffnet.K-1)]
  return IntervalsInfo(ffnet=ffnet, x_intvs=x_intvs, acx_intvs=acx_intvs)
end

# ---- clique index sets (bit-exact with makeCliques, src/Methods/chordal_cliques.jl:13-59) ---------
function makeCliquesB200(net::DeviceNet, β::Int)
  sz = sizes(net, β)
  ck_off, ck_idx = zeros(Int64, sz.ncliques + 1), zeros(Int64, sz.sum_ck)
  ck1_len, d_off, d_idx = zeros(Int64, sz.ncliques), zeros(Int64, 2 * sz.ncliques + 1), zeros(Int64, sz.sum_dk)
  check(ccall((:nnsdp_cliques, LIB), Int32,
              (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}),
              net.h, β, ck_off, ck_idx, ck1_len, d_off, d_idx))
  cliques = Vector{Tuple{VecInt, Vector{VecInt}, Vector{VecInt}}}()
  for k in 1:sz.ncliques
    Ck = ck_idx[ck_off[k]+1:ck_off[k+1]]
    parts = ck1_len[k] < length(Ck) ? [Ck[1:ck1_len[k]], Ck[ck1_len[k]+1:end]] : [Ck]
    D1 = d_idx[d_off[2k-1]+1:d_off[2k]]
    D2 = d_idx[d_off[2k]+1:d_off[2k+1]]
    push!(cliques, (Ck, parts, isempty(D2) ? [D1] : [D1, D2]))
  end
  return cliques
end

# ---- dispatch point 2/3: numeric-gamma assembly --------------------------------------------------
# One query = what SafetyQuery / ReachQuery hold (src/Methods/Methods.jl:19-41) plus numeric multipliers.
# `γacs = [γbounded, γsector]` in the order makeQcActivsIntvs returns the QCs (src/Qc/activ.jl:64).
function query_inputs(qc_input::QcInputBox, qc_out, qc_bounded::QcActivBounded, qc_sector::QcActivSector,
                      γin::Vector{Float64}, γacs::Vector{Vector{Float64}}, γout::Vector{Float64}, keep::Vector{Any})
  p(v) = (push!(keep, v); pointer(v))
  kind, S, vec, invP = OUT_SAFETY, Float64[], Float64[], Float64[]
  if qc_out isa QcSafety
    S = vec_colmajor(Matrix{Float64}(qc_out.S))
  elseif qc_out isa QcReachHplane
    kind, vec = OUT_HPLANE, Vector{Float64}(qc_out.normal)
  elseif qc_out isa QcReachCircle
    kind, vec = OUT_CIRCLE, Vector{Float64}(qc_out.yc)
  elseif qc_out isa QcReachEllipsoid
    kind, vec, invP = OUT_ELLIPSOID, Vector{Float64}(qc_out.yc), vec_colmajor(Matrix{Float64}(qc_out.invP))
  else
    error("unrecognized qc: $(qc_out)")   # src/Qc/output.jl:95
  end
  n(v) = length(v)
  return QueryInputs(
    p(Vector{Float64}(qc_input.x1min)), n(qc_input.x1min), p(Vector{Float64}(qc_input.x1max)), n(qc_input.x1max),
    p(Vector{Float64}(qc_bounded.acymin)), qc_bounded.acydim, p(Vector{Float64}(qc_bounded.acymax)), qc_bounded.acydim,
    p(Vector{Float64}(qc_sector.smin)), qc_sector.acxdim, p(Vector{Float64}(qc_sector.smax)), qc_sector.acxdim,
    p(γin), n(γin), p(γacs[1]), n(γacs[1]), p(γacs[2]), n(γacs[2]),
    kind, Int32(0),
    isempty(S) ? Ptr{Float64}(C_NULL) : p(S), n(S), isempty(vec) ? Ptr{Float64}(C_NULL) : p(vec), n(vec),
    isempty(invP) ? Ptr{Float64}(C_NULL) : p(invP), n(invP), isempty(γout) ? Ptr{Float64}(C_NULL) : p(γout), n(γout))
end
vec_colmajor(M::Matrix{Float64}) = vec(copy(M))

# Z[C_k, C_k] for every clique (dense Matrix{Float64}), i.e. Ec(Ck) * (Zin + Zout + sum(Zacs)) * Ec(Ck)'
# with the numeric multipliers of scripts/test_acas.jl:81-85.
function assembleCliqueBlocks(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector,
                              γin, γacs, γout = Float64[])
  sz = sizes(net, β)
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  out = Vector{Float64}(undef, sz.sum_ck_sq)
  GC.@preserve keep check(ccall((:nnsdp_assemble_blocks, LIB), Int32,
              (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{QueryInputs}, Ptr{Float64}), net.ctx.h, net.h, β, 1, qi, out))
  cliques = makeCliquesB200(net, β)
  blocks, o = Vector{Matrix{Float64}}(), 0
  for (Ck, _, _) in cliques
    n = length(Ck)
    push!(blocks, reshape(out[o+1:o+n*n], n, n))   # column-major on the wire == Julia layout
    o += n * n
  end
  return cliques, blocks
end

# The dense Z = Zin + Zout + sum(Zacs) (src/Methods/chordal_sdp.jl:114,145) for numeric multipliers.
function assembleZ(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector, γin, γacs, γout = Float64[])
  sz = sizes(net, β)
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  Z = Matrix{Float64}(undef, sz.Zdim, sz.Zdim)
  GC.@preserve keep check(ccall((:nnsdp_assemble_dense, LIB), Int32,
              (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{QueryInputs}, Ptr{Float64}), net.ctx.h, net.h, β, 1, qi, Z))
  return Z
end

# ---- packed records: the block-sparse upper triangle of Z (NNSDP_FORMAT_PACKED) --------------------------------
# One record holds every region of Z that can be non-zero once; Z[C_k, C_k] of any clique is a set of sub-rectangles of
# its cells.  cellView gives a cell as a zero-copy matrix; cliqueBlocks expands a record into the dense blocks the
# reference's setupZksum! scatters (src/Methods/chordal_sdp.jl:60-93) through the library's own nnsdp_packed_unpack.
function packedLayout(ffnet::FeedFwdNet, β::Int)
  n, rec, alw = Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0)
  xd = Int64.(ffnet.xdims)
  check(ccall((:nnsdp_packed_layout, LIB), Int32,
              (Int64, Ptr{Int64}, Int64, Int64, Ptr{PackedCell}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}),
              ffnet.K, xd, β, 0, C_NULL, n, rec, alw))
  cells = Vector{PackedCell}(undef, n[])
  check(ccall((:nnsdp_packed_layout, LIB), Int32,
              (Int64, Ptr{Int64}, Int64, Int64, Ptr{PackedCell}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}),
              ffnet.K, xd, β, n[], cells, n, rec, alw))
  return cells, rec[], alw[]
end

cellView(record::AbstractVector{Float64}, c::PackedCell) =
  reshape(view(record, (c.offset + 1):(c.offset + c.nrows * c.ncols)), Int(c.nrows), Int(c.ncols))

function assemblePacked(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector, γin, γacs, γout = Float64[])
  cells, rec, _ = packedLayout(net.ffnet, β)
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  record, present = zeros(rec), zeros(UInt8, length(cells))
  GC.@preserve keep check(ccall((:nnsdp_assemble_packed, LIB), Int32,
              (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{QueryInputs}, Ptr{Float64}, Ptr{UInt8}),
              net.ctx.h, net.h, β, 1, qi, record, present))
  return cells, record, present
end

function cliqueBlocks(ffnet::FeedFwdNet, β::Int, cliques, record::Vector{Float64}, present::Vector{UInt8})
  out = Vector{Float64}(undef, sum(length(Ck)^2 for (Ck, _, _) in cliques))
  check(ccall((:nnsdp_packed_unpack, LIB), Int32,
              (Int64, Ptr{Int64}, Int64, Ptr{Float64}, Ptr{UInt8}, Int32, Ptr{Float64}),
              ffnet.K, Int64.(ffnet.xdims), β, record, present, FORMAT_BLOCKS, out))
  blocks, o = Vector{Matrix{Float64}}(), 0
  for (Ck, _, _) in cliques
    n = length(Ck)
    push!(blocks, reshape(out[o+1:o+n*n], n, n))
    o += n * n
  end
  return blocks
end

# ---- certificate check: eigmax(Z) without forming Z (src/Methods/Methods.jl:116-117, experiments/acas.jl:71-79) ----
# λmax of Z(γ) for numeric multipliers, matrix-free Lanczos on the device (nnsdp_batch_lambda_max_ex).  Returns
# (λ, residual, converged): the Ritz value λ is a LOWER bound of λmax; it certifies eigmax(Z) <= 1e-4 only when
# `converged` is true (an eigenvalue of Z then lies within `residual` of λ).
function eigmaxZ(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector, γin, γacs, γout = Float64[];
                 max_iters::Int = 300, tol::Float64 = 1e-10)
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  h = Ref{Ptr{Cvoid}}(C_NULL)
  check(ccall((:nnsdp_batch_create, LIB), Int32,
              (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Int64, Int64, Int64, Int32, Ptr{Ptr{Cvoid}}),
              net.ctx.h, 0, net.h, β, 1, 1, 0, h))
  lam, its, resid, conv = zeros(1), zeros(Int32, 1), zeros(1), zeros(Int32, 1)
  try
    GC.@preserve keep check(ccall((:nnsdp_batch_set_inputs, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{QueryInputs}), h[], 1, qi))
    check(ccall((:nnsdp_batch_prepare, LIB), Int32, (Ptr{Cvoid},), h[]))
    st = ccall((:nnsdp_batch_lambda_max_ex, LIB), Int32,
               (Ptr{Cvoid}, Int32, Float64, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}),
               h[], max_iters, tol, lam, its, resid, conv)
    st == Int32(-6) || check(st)          # NNSDP_ERR_NOCONV: the outputs are written, converged = 0
  finally
    ccall((:nnsdp_batch_destroy, LIB), Int32, (Ptr{Cvoid},), h[])
  end
  return lam[1], resid[1], conv[1] == 1
end

# Sound form of the same acceptance test (nnsdp_batch_certify): a Cholesky factorisation of τ'I - Z(γ) along the
# cliques with a margin for its rounding error.  Returns (certified, bound, lower): certified == true PROVES
# eigmax(Z) <= bound <= τ for the FP64 Z the library assembles; false proves eigmax(Z) >= lower instead (from the
# failed factorisation, nnsdp_batch_certify_ex; lower = -Inf when certified).  of_gamma = true makes both statements
# about the exact Z(γ) of the same inputs instead (nnsdp_batch_certify_gamma: the factorisation at τ minus a bound on
# the assembly's rounding error, see assemblyErrorB200).
function eigmaxLeB200(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector, γin, γacs, γout = Float64[];
                      τ::Float64 = 1e-4, of_gamma::Bool = false)
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  h = Ref{Ptr{Cvoid}}(C_NULL)
  check(ccall((:nnsdp_batch_create, LIB), Int32,
              (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Int64, Int64, Int64, Int32, Ptr{Ptr{Cvoid}}),
              net.ctx.h, 0, net.h, β, 1, 1, 0, h))
  tau, cert, bound, fidx, lower, err = [τ], zeros(Int32, 1), zeros(1), zeros(Int64, 1), zeros(1), zeros(1)
  try
    GC.@preserve keep check(ccall((:nnsdp_batch_set_inputs, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{QueryInputs}), h[], 1, qi))
    check(ccall((:nnsdp_batch_prepare, LIB), Int32, (Ptr{Cvoid},), h[]))
    if of_gamma
      check(ccall((:nnsdp_batch_certify_gamma, LIB), Int32,
                  (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64},
                   Ptr{Float64}),
                  h[], tau, 0, cert, bound, fidx, C_NULL, lower, err))
    else
      check(ccall((:nnsdp_batch_certify_ex, LIB), Int32,
                  (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
                  h[], tau, 0, cert, bound, fidx, C_NULL, lower))
    end
  finally
    ccall((:nnsdp_batch_destroy, LIB), Int32, (Ptr{Cvoid},), h[])
  end
  return cert[1] == 1, bound[1], lower[1]
end

# e ≥ ‖Z_dev - Z(γ)‖∞ (nnsdp_batch_assembly_error): how far the FP64 Z the library assembles can be from the exact
# Z(γ) of the same inputs, QC bounds as computed by the library; so eigmax(Z(γ)) lies within e of eigmax(Z_dev).
function assemblyErrorB200(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector, γin, γacs, γout = Float64[])
  keep = Any[]
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, Vector{Float64}(γin),
                        [Vector{Float64}(g) for g in γacs], Vector{Float64}(γout), keep))
  h = Ref{Ptr{Cvoid}}(C_NULL)
  check(ccall((:nnsdp_batch_create, LIB), Int32,
              (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Int64, Int64, Int64, Int32, Ptr{Ptr{Cvoid}}),
              net.ctx.h, 0, net.h, β, 1, 1, 0, h))
  err = zeros(1)
  try
    GC.@preserve keep check(ccall((:nnsdp_batch_set_inputs, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{QueryInputs}), h[], 1, qi))
    check(ccall((:nnsdp_batch_prepare, LIB), Int32, (Ptr{Cvoid},), h[]))
    check(ccall((:nnsdp_batch_assembly_error, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), h[], err, C_NULL))
  finally
    ccall((:nnsdp_batch_destroy, LIB), Int32, (Ptr{Cvoid},), h[])
  end
  return err[1]
end

# ---- vnnlib property -> batched safety queries (experiments/vnnlib_utils.jl:18-56) -------------------
# Returns what loadVnnlibCnf returns -- a Vector of disjunctive clauses, each a Vector of
# (QcInputBox, QcSafety) -- but parsed and flattened by the library in one call; x1min / x1max / S come back
# as Q-column arrays that assembleCliqueBlocks can take as one batch.
function loadVnnlibCnfB200(spec_file::String, ffnet)
  n_in, n_out = ffnet.xdims[1], ffnet.xdims[end]
  nq, nc = Ref{Int64}(0), Ref{Int64}(0)
  check(ccall((:nnsdp_vnnlib_read, LIB), Int32,
              (Cstring, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
              spec_file, n_in, n_out, 0, nq, nc, C_NULL, C_NULL, C_NULL, C_NULL))
  sdim = n_in + n_out + 1
  x1min, x1max = zeros(n_in, nq[]), zeros(n_in, nq[])
  S = zeros(sdim, sdim, nq[])
  clause = zeros(Int64, nq[])
  check(ccall((:nnsdp_vnnlib_read, LIB), Int32,
              (Cstring, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
              spec_file, n_in, n_out, nq[], nq, nc, x1min, x1max, S, clause))
  cnf = [Vector{Tuple{Any, Any}}() for _ in 1:nc[]]
  for q in 1:nq[]
    push!(cnf[clause[q] + 1], (QcInputBox(x1min=x1min[:, q], x1max=x1max[:, q]),
                               QcSafety(S=Symmetric(S[:, :, q]))))
  end
  return cnf, x1min, x1max, S, clause
end

# ---- dispatch point 3: the symbolic hand-off -----------------------------------------------------
# Z(γ) = Z0 + Σ_v γ_v Z_v over the upper triangle of the clique cover, as a sparse matrix A (nent × nvar)
# and a constant vector z0: what `Z = Zin + Zout + sum(Zacs)` holds entry by entry as AffExpr
# (src/Methods/chordal_sdp.jl:114,145) without ever forming the AffExpr matrices.
struct AffineSizes
  nvar::Int64; nent::Int64; nnz::Int64
  var_in::Int64; var_out::Int64; var_bnd::Int64; var_sec::Int64
end

function affineForm(net::DeviceNet, β::Int, qc_input, qc_out, qc_bounded, qc_sector; max_nnz::Int = 0)
  keep = Any[]
  nsec = qc_sector.vardim
  qi = Ref(query_inputs(qc_input, qc_out, qc_bounded, qc_sector, zeros(length(qc_input.x1min)),
                        [zeros(qc_bounded.acydim), zeros(nsec)], qc_out isa QcSafety ? Float64[] : [0.0], keep))
  h, sz = Ref{Ptr{Cvoid}}(C_NULL), Ref{AffineSizes}()
  GC.@preserve keep check(ccall((:nnsdp_affine_create, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{QueryInputs}, Int64, Ptr{Ptr{Cvoid}}, Ptr{AffineSizes}),
      net.ctx.h, net.h, β, qi, max_nnz, h, sz))
  s = sz[]
  ent_row, ent_col, z0 = zeros(Int64, s.nent), zeros(Int64, s.nent), zeros(s.nent)
  coo_ent, coo_var, coo_val = zeros(Int64, s.nnz), zeros(Int64, s.nnz), zeros(s.nnz)
  try
    check(ccall((:nnsdp_affine_get, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
        h[], ent_row, ent_col, z0, coo_ent, coo_var, coo_val))
  finally
    ccall((:nnsdp_affine_destroy, LIB), Int32, (Ptr{Cvoid},), h[])
  end
  A = sparse(coo_ent, coo_var, coo_val, s.nent, s.nvar)   # duplicates are summed
  return s, ent_row, ent_col, z0, A
end

# The affine forms of several queries in one call (nnsdp_affine_create_batch): the directions of a reach polytope
# (src/NnSdp.jl:73-95) or the members of a vnnlib property (experiments/vnnlib_utils.jl:58-74).  The queries share one
# output-QC type; their boxes, QC bounds and output data are packed as Q-column arrays.  Queries with the same box and
# QC bounds share one coefficient matrix, built once on the device as canonical CSC (no sort, no duplicate sum here):
# `A` is then the same SparseMatrixCSC object for every member of the group.  Returns one
# (sizes, ent_row, ent_col, z0, A) per query, as affineForm does for one.
struct AffineBatchSizes
  Q::Int64; ngroups::Int64
  nvar::Int64; nent::Int64
  var_in::Int64; var_out::Int64; var_bnd::Int64; var_sec::Int64
  nnz_total::Int64; nnz_max::Int64
end

function affineFormBatch(net::DeviceNet, β::Int, queries; max_nnz::Int = 0)
  Q = length(queries)
  Q >= 1 || error("affineFormBatch needs at least one query")
  outs = [q isa Methods.SafetyQuery ? q.qc_safety : q.qc_reach for q in queries]
  all(o -> typeof(o) == typeof(outs[1]), outs) || error("affineFormBatch: the queries must share one output-QC type")
  cols(f) = reduce(hcat, [Vector{Float64}(f(i)) for i in 1:Q])   # n x Q: column q belongs to query q
  x1min, x1max = cols(i -> queries[i].qc_input.x1min), cols(i -> queries[i].qc_input.x1max)
  ymin, ymax = cols(i -> queries[i].qc_activs[1].acymin), cols(i -> queries[i].qc_activs[1].acymax)
  smin, smax = cols(i -> queries[i].qc_activs[2].smin), cols(i -> queries[i].qc_activs[2].smax)
  kind, S, vec, invP = OUT_SAFETY, zeros(0, 0), zeros(0, 0), zeros(0, 0)
  o1 = outs[1]
  if o1 isa QcSafety
    S = cols(i -> vec_colmajor(Matrix{Float64}(outs[i].S)))
  elseif o1 isa QcReachHplane
    kind, vec = OUT_HPLANE, cols(i -> outs[i].normal)
  elseif o1 isa QcReachCircle
    kind, vec = OUT_CIRCLE, cols(i -> outs[i].yc)
  elseif o1 isa QcReachEllipsoid
    kind, vec = OUT_ELLIPSOID, cols(i -> outs[i].yc)
    invP = cols(i -> vec_colmajor(Matrix{Float64}(outs[i].invP)))
  else
    error("unrecognized qc: $(o1)")   # src/Qc/output.jl:95
  end
  zin, zbnd, zsec, zout = zeros(size(x1min, 1)), zeros(size(ymin, 1)), zeros(queries[1].qc_activs[2].vardim), [0.0]
  p(a) = isempty(a) ? Ptr{Float64}(C_NULL) : pointer(a)
  ld(a) = Int64(size(a, 1))
  keep = Any[x1min, x1max, ymin, ymax, smin, smax, S, vec, invP, zin, zbnd, zsec, zout]
  qi = Ref(QueryInputs(p(x1min), ld(x1min), p(x1max), ld(x1max), p(ymin), ld(ymin), p(ymax), ld(ymax),
                       p(smin), ld(smin), p(smax), ld(smax), p(zin), 0, p(zbnd), 0, p(zsec), 0, kind, Int32(0),
                       p(S), ld(S), p(vec), ld(vec), p(invP), ld(invP),
                       kind == OUT_SAFETY ? Ptr{Float64}(C_NULL) : p(zout), 0))
  h, sz = Ref{Ptr{Cvoid}}(C_NULL), Ref{AffineBatchSizes}()
  GC.@preserve keep check(ccall((:nnsdp_affine_create_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{QueryInputs}, Int64, Ptr{Ptr{Cvoid}}, Ptr{AffineBatchSizes}),
      net.ctx.h, net.h, β, Q, qi, max_nnz, h, sz))
  s = sz[]
  ent_row, ent_col, z0 = zeros(Int64, s.nent), zeros(Int64, s.nent), zeros(s.nent, Q)
  group_of, group_nnz, group_first = zeros(Int64, Q), zeros(Int64, s.ngroups), zeros(Int64, s.ngroups)
  mats = Vector{SparseMatrixCSC{Float64, Int64}}(undef, s.ngroups)
  try
    check(ccall((:nnsdp_affine_batch_get, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
                h[], ent_row, ent_col, z0))
    check(ccall((:nnsdp_affine_batch_groups, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}),
                h[], group_of, group_nnz, group_first))
    for g in 1:s.ngroups
      var_ptr, ent_idx, val = zeros(Int64, s.nvar + 1), zeros(Int64, group_nnz[g]), zeros(group_nnz[g])
      check(ccall((:nnsdp_affine_batch_get_group, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
                  h[], g - 1, var_ptr, ent_idx, val))
      mats[g] = SparseMatrixCSC(s.nent, s.nvar, var_ptr, ent_idx, val)   # canonical: no sort, no duplicate sum
    end
  finally
    ccall((:nnsdp_affine_batch_destroy, LIB), Int32, (Ptr{Cvoid},), h[])
  end
  sizes_of(A) = AffineSizes(s.nvar, s.nent, nnz(A), s.var_in, s.var_out, s.var_bnd, s.var_sec)
  return [(sizes_of(mats[group_of[q] + 1]), ent_row, ent_col, z0[:, q], mats[group_of[q] + 1]) for q in 1:Q]
end

# Options type that selects the GPU-assembled constraints in runQuery (src/Methods/Methods.jl:97-103);
# same five fields as ChordalSdpOptions (src/Methods/chordal_sdp.jl:10-16) plus the device network.
# `forms`: query => affineForm result, e.g. from affineFormBatch for a polytope or a vnnlib property; setupB200! then
# uses that entry instead of calling affineForm.
Base.@kwdef struct ChordalB200Options <: Methods.QueryOptions
  include_default_mosek_opts::Bool = true
  mosek_opts::Dict{String, Any} = Dict()
  decomp_mode::Methods.DecompMode = Methods.SingleDecomp()
  use_dual::Bool = false
  verbose::Bool = false
  net::DeviceNet
  forms::Union{Nothing, IdDict} = nothing
end

# Common part of setupSafety!/setupReach! (src/Methods/chordal_sdp.jl:96-153): variables in the reference's
# creation order, clique PSD variables through the reference's own setupZs!, and the equality
# Z[r,c](γ) == Zksum[r,c] on the upper triangle of the cover (both sides are symmetric and identically zero
# outside the cover, so this is the same feasible set as the reference's Zdim^2 scalar equalities).
function setupB200!(model, query, qc_out, opts::ChordalB200Options)
  ffnet = query.ffnet
  qc_bounded, qc_sector = query.qc_activs[1], query.qc_activs[2]   # order of makeQcActivsIntvs (activ.jl:64)
  β = qc_sector.β
  s, ent_row, ent_col, z0, A = (opts.forms !== nothing && haskey(opts.forms, query)) ? opts.forms[query] :
                                affineForm(opts.net, β, query.qc_input, qc_out, qc_bounded, qc_sector)
  vars = Dict()
  γin = Methods.JuMP.@variable(model, [1:query.qc_input.vardim])
  Methods.JuMP.@constraint(model, γin .>= 0)
  vars[:γin] = γin
  γ = Vector{Methods.JuMP.VariableRef}(γin)
  if !(qc_out isa QcSafety)
    γout = Methods.JuMP.@variable(model, [1:qc_out.vardim])
    Methods.JuMP.@constraint(model, γout .>= 0)
    vars[:γout] = γout
    append!(γ, γout)
  end
  for (i, qc) in enumerate(query.qc_activs)
    γac = Methods.JuMP.@variable(model, [1:qc.vardim])
    Methods.JuMP.@constraint(model, γac .>= 0)
    vars[Symbol(:γac, i)] = γac
    append!(γ, γac)
  end
  @assert length(γ) == s.nvar
  Zvec = A * γ .+ z0                                   # nent affine expressions, built by one sparse product
  # Zksum on the same entries: sum of the clique variables that contain (r, c)
  cliques = Methods.makeCliques(query.qcs, ffnet)
  ref_opts = Methods.ChordalSdpOptions(decomp_mode = opts.decomp_mode)
  Zs, _ = Methods.setupZs!(model, cliques, query, ref_opts)
  entry_of = Dict{Tuple{Int64, Int64}, Int64}()         # (row, column) of the cover's upper triangle -> entry number
  for e in 1:s.nent; entry_of[(ent_row[e], ent_col[e])] = e end
  @assert length(entry_of) == s.nent
  entry(r, c) = entry_of[(r, c)]                        # KeyError if a clique reaches outside the cover
  Zksum = [zero(Methods.JuMP.AffExpr) for _ in 1:s.nent]   # distinct objects: add_to_expression! mutates in place
  for (k, (Ck, _, _)) in enumerate(cliques)
    for j in 1:length(Ck), i in 1:j
      Methods.JuMP.add_to_expression!(Zksum[entry(Ck[i], Ck[j])], Zs[k][i, j])
    end
  end
  Methods.JuMP.@constraint(model, Zvec .== Zksum)
  # Z(γ) as the reference's consumers index it (soln.values[:Z], Methods.jl:116): symmetric, backed by its upper triangle
  vars[:Z] = Symmetric(sparse(ent_row, ent_col, Zvec, sum(ffnet.zdims), sum(ffnet.zdims)), :U)
  return vars
end

function Methods.setupSafety!(model, query::Methods.SafetyQuery, opts::ChordalB200Options)
  vars = setupB200!(model, query, query.qc_safety, opts)
  γacs = [vars[Symbol(:γac, i)] for i in 1:length(query.qc_activs)]
  Methods.JuMP.@objective(model, Min, sum(vars[:γin]) + sum(sum(γac) for γac in γacs))   # chordal_sdp.jl:111
  return model, vars
end

function Methods.setupReach!(model, query::Methods.ReachQuery, opts::ChordalB200Options)
  vars = setupB200!(model, query, query.qc_reach, opts)
  Methods.JuMP.@objective(model, Min, query.obj_func(vars[:γout]))                        # chordal_sdp.jl:136
  return model, vars
end

export Context, DeviceNet, IntervalsB200, IntervalsCrownB200, makeCliquesB200, assembleCliqueBlocks, assembleZ
export affineForm, affineFormBatch, ChordalB200Options, eigmaxZ, packedLayout, cellView, assemblePacked, cliqueBlocks

end # module
