# bpots_b200.jl -- OPTIONAL addition after src/decoders/bpots_decoder.jl (which stays as it is) and
# julia/belief_propagation_b200.jl (for the ccall helpers).
#
# UNEXECUTED IN THE BUILD ENVIRONMENT (no julia binary in the image); mirrored by ldpcdecoders.jl_b200/decoder.py: BPOTSDecoder.
#
# decode!(::BPOTSDecoder, syndrome) (bpots_decoder.jl:226-340) keeps running in Julia for a single syndrome; this file adds the
# batch method: every column of `syndromes` through ldpcb200_bpots_decode_batch (csrc/bpots.cuh: one CTA per syndrome, Float64
# LLR-domain tanh/atanh updates, oscillation counting, best-so-far tracking, bias -C every T iterations), instead of the
# generic column loop of abstract_decoder.jl:31-42.  The GPU handle (the device-resident Tanner graph of decoder.sparse_H) is
# created on first use and cached per decoder.  tanh / atanh / log are CUDA's on the device and Julia's on the host, so the two
# agree except where a last-bit difference of those functions is amplified (DESIGN.md section 3.7).
const _B200_OTS_HANDLES = IdDict{BPOTSDecoder,Ptr{Cvoid}}()

function _b200_ots_handle(decoder::BPOTSDecoder)
    get!(_B200_OTS_HANDLES, decoder) do
        out = Ref{Ptr{Cvoid}}(C_NULL)
        H = decoder.sparse_H
        colptr, rowval = Vector{Int64}(H.colptr), Vector{Int64}(H.rowval)
        GC.@preserve colptr rowval _b200_check(ccall((:ldpcb200_create, LDPCB200_LIB), Cint,
            (Int64, Int64, Ptr{Int64}, Ptr{Int64}, Int32, Float64, Int32, Int32, Ptr{Int32}, Int32, Ptr{Ptr{Cvoid}}),
            decoder.s, decoder.n, colptr, rowval, 1, decoder.per, decoder.max_iters, 0, C_NULL, 0, out))
        out[]
    end
end

function batchdecode!(decoder::BPOTSDecoder, syndromes::AbstractMatrix, errors::AbstractMatrix, converged::AbstractVector{Bool})
    @assert size(syndromes, 2) == size(errors, 2)
    @assert size(syndromes, 2) == length(converged)
    h = _b200_ots_handle(decoder)
    B = size(syndromes, 2)
    syn = syndromes isa _B200_IN ? syndromes : Matrix{Int64}(syndromes)
    err = errors isa _B200_OUT ? errors : Matrix{Int64}(undef, decoder.n, B)
    conv = converged isa Vector{Bool} ? converged : Vector{Bool}(undef, B)
    GC.@preserve syn err conv begin
        _b200_check(ccall((:ldpcb200_bpots_decode_batch, LDPCB200_LIB), Cint,
                          (Ptr{Cvoid}, Int64, Ptr{Cvoid}, Int32, Int64, Ptr{Cvoid}, Int32, Int64, Ptr{UInt8}, Ptr{Int32}, Int32, Float64),
                          h, B, _b200_ptr(syn), _b200_fmt(syn), decoder.s, _b200_ptr(err), _b200_fmt(err), decoder.n,
                          pointer(conv), C_NULL, Int32(decoder.T), decoder.C))
    end
    err === errors || (errors .= err)
    conv === converged || (converged .= conv)
    return errors, converged
end

"""
    sample_decode_score(decoder::BPOTSDecoder, shots; first=0, seed=12345, per_channel=decoder.per) -> NamedTuple

The sampling + scoring harness of `sample_decode_score(::BeliefPropagationDecoder, ...)` with BP-OTS as the decoder
(ldpcb200_sample_bpots_score): errors drawn, decoded with the decoder's per, max_iters, T and C, and scored on the GPUs.
`iterations` counts BP-OTS iterations; `osd_processed` is 0.
"""
function sample_decode_score(decoder::BPOTSDecoder, shots::Integer; first::Integer=0, seed::Integer=12345,
                             per_channel::Float64=decoder.per)
    h = _b200_ots_handle(decoder)
    out = zeros(Int64, 8)
    GC.@preserve out _b200_check(ccall((:ldpcb200_sample_bpots_score, LDPCB200_LIB), Cint,
                                       (Ptr{Cvoid}, Int64, Int64, UInt64, Float64, Int32, Float64, Ptr{Int64}),
                                       h, shots, first, UInt64(seed), per_channel, Int32(decoder.T), decoder.C, out))
    return (shots=out[1], converged=out[2], iterations=out[3], exact_matches=out[4], syndrome_satisfied=out[5],
            failures=out[6], residual_weight=out[7], osd_processed=out[8])
end
