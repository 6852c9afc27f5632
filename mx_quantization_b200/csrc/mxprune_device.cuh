// Device-side building blocks shared by every kernel of libmxprune.
//
// Arithmetic contract (SURVEY.md section 8a; reference citations relative to the
// d9bjo0522/mx_quantization checkout):
//   A1 bf16 pre-rounding, half away from zero   microxscaling/mx/elemwise_ops.py:201-216, :64-65
//   A2 MXINT8 block quantizer                   microxscaling/mx/mx_ops.py:49-99, 180-306
//                                               microxscaling/mx/elemwise_ops.py:92-180
// All of it is integer / exactly-rounded fp32 work, so results are bit-identical to the
// reference's CPU fp32 path by construction, not by tolerance.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mxp {

constexpr unsigned FULL = 0xffffffffu;
constexpr int WARPS = 8;
constexpr int THREADS = WARPS * 32;
constexpr int ZERO_BLOCK_EXP = -126;   // floor(log2(2^-126)), mx_ops.py:83-87

struct View {   // (B,H,N,hd) view, element strides, innermost stride 1
    const float* p;  // fp32 elements, or the 16-bit elements of a kernel instantiated for DT_BF16 / DT_F16
    int64_t sB, sH, sN;
};

// Element types of the activation views and of the attention output (MXP_DT_* of include/mxprune.h).  A kernel that
// touches activations takes its element type as a template parameter; loads widen 16-bit values to their fp32 bit
// pattern (exact), so everything after the load is the fp32 arithmetic, and only the final output store narrows.
constexpr int DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2;

// eight 16-bit elements (one 16-byte chunk) -> their exact fp32 bit patterns
template <int DT>
__device__ __forceinline__ void widen8(const uint4 v, uint32_t* x) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (DT == DT_BF16) {
            x[2 * i] = w[i] << 16;
            x[2 * i + 1] = w[i] & 0xffff0000u;
        } else {
            float lo, hi;
            asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}"
                : "=f"(lo), "=f"(hi) : "r"(w[i]));
            x[2 * i] = __float_as_uint(lo);
            x[2 * i + 1] = __float_as_uint(hi);
        }
    }
}
template <int DT>
__device__ __forceinline__ uint32_t widen1(uint16_t h) {
    if (DT == DT_BF16) return (uint32_t)h << 16;
    float f;
    asm("cvt.f32.f16 %0, %1;" : "=f"(f) : "h"(h));
    return __float_as_uint(f);
}

// One 32-element block of a row from global memory as fp32 bit patterns (elements >= nd are 0): eight 16-byte loads of
// fp32, four of 16-bit values.  src is 16-byte aligned.
template <int DT>
__device__ __forceinline__ void load_block_bits(const float* src, int nd, bool ok, uint32_t (&xv)[32]) {
    if constexpr (DT == DT_F32) {
#pragma unroll
        for (int s = 0; s < 8; ++s) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (ok && 4 * s < nd) v = __ldg(reinterpret_cast<const uint4*>(src) + s);
            xv[4 * s] = v.x; xv[4 * s + 1] = v.y; xv[4 * s + 2] = v.z; xv[4 * s + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (ok && 8 * s < nd) v = __ldg(reinterpret_cast<const uint4*>(src) + s);
            widen8<DT>(v, &xv[8 * s]);
        }
    }
}
// element pointer of a view row (element offsets, in the view's element type)
template <int DT>
__device__ __forceinline__ const float* view_elem(const float* p, int64_t off) {
    if constexpr (DT == DT_F32) return p + off;
    else return reinterpret_cast<const float*>(reinterpret_cast<const uint16_t*>(p) + off);
}
// fp32 bit pattern of one element at element offset off
template <int DT>
__device__ __forceinline__ uint32_t load_elem_bits(const float* p, int64_t off) {
    if constexpr (DT == DT_F32) return __float_as_uint(__ldg(p + off));
    else return widen1<DT>(__ldg(reinterpret_cast<const unsigned short*>(p) + off));
}
// output element at element offset off of an fp32 (out16 false) or 16-bit output
__device__ __forceinline__ float* out_elem(float* p, int64_t off, bool out16) {
    return out16 ? reinterpret_cast<float*>(reinterpret_cast<uint16_t*>(p) + off) : p + off;
}
// four fp32 output values (bit patterns) -> the output type, round to nearest even; dst 16- (fp32) or 8-byte aligned
template <int DT>
__device__ __forceinline__ void store_out4(float* dst, int64_t off, const uint4 v) {
    if constexpr (DT == DT_F32) {
        *reinterpret_cast<uint4*>(dst + off) = v;
    } else {
        const uint32_t in[4] = {v.x, v.y, v.z, v.w};
        uint32_t o[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            uint32_t r;
            if (DT == DT_BF16)
                asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(in[2 * i + 1])), "f"(__uint_as_float(in[2 * i])));
            else
                asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(in[2 * i + 1])), "f"(__uint_as_float(in[2 * i])));
            o[i] = r;
        }
        *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(dst) + off) = make_uint2(o[0], o[1]);
    }
}

struct PredParams {
    View q, k;
    int B, H, Nq, Nk, hd, top_k, bf16, flush;
    uint32_t* mask;
    int32_t* idx;
    int8_t *q_codes, *q_exps, *k_codes, *k_exps;
    unsigned char *q_op, *k_op;   // MMA-ready bf16 operands for the exact-attention kernel (may be null)
    float* scores;   // dense debug output (k_predict_scores only)
    const float* key_bias;       // optional additive bias per (batch, key), added to the predicted scores (fp32)
    int64_t kb_sB;               //   key_bias[b * kb_sB + j]; rows then take the generic fp32 path
    const uint8_t* row_filter;   // k_predict_topk_long only: [heads][Nq], process rows with a non-zero flag (null = all)
    void* long_ws;               // host side: workspace of the long-sequence tensor-core path (may be null)
    size_t long_ws_bytes;
    int pred_mode;               // 0 exponent-sign (default), 1 partial_Q, 2 partial_K, 3 exact scores, 4 MXINT4, 5 two-step, 6 true_ex, 7 ELSA (mxprune_predict_wide.cuh)
    float score_scale;           // pred_mode 3: the attention scale the true scores are ranked with
    const float* elsa_proj;      // pred_mode 7 (ELSA): the hd x hd projection matrix, fp32 row-major (hash j = sign(x . P[j]))
    float elsa_cap;              // pred_mode 7: hash dot products above this value tie (the reference's angle clamp)
    int dt;                      // element type of q / k (DT_*; host side: selects the kernel instantiation)
};

// 2^e as fp32 for e in [-149, 127] (subnormal below -126).
__device__ __forceinline__ float exp2i(int e) {
    return __uint_as_float(e >= -126 ? (uint32_t)(e + 127) << 23 : 1u << (e + 149));
}

// A1: round-half-away to bf16 on the fp32 bit pattern (sign preserved).
// Adding half a bf16 ulp to the magnitude never carries into the sign bit for finite values and
// infinities, so the sign needs no separate handling (NaN is outside the path's contract).
__device__ __forceinline__ uint32_t bf16_half_away(uint32_t b) {
    return (b + 0x8000u) & 0xffff0000u;
}
__device__ __forceinline__ float bf16_half_away(float x) {
    return __uint_as_float(bf16_half_away(__float_as_uint(x)));
}

// Shared exponent of a block from the bit pattern of its max magnitude.
// The reference evaluates floor(log2(max)) in fp32 (mx_ops.py:93-97): when max is within
// jmax(n) ulps below 2^n the fp32 logarithm rounds up to n.  jmax depends only on the binade
// of n: floor(ln2 * 2^floor(log2 a)), a = n-1 (n>0) or -n (n<0)  ->  {0,1,2,5,11,22,44,88}.
// zero block -> -126; subnormal max -> -127 (the scale_bits=8 floor, mx_ops.py:289-291).
__device__ __forceinline__ int mx_shared_exp(uint32_t maxbits) {
    const int E = (int)(maxbits >> 23);
    const uint32_t m = maxbits & 0x7fffffu;
    if (E == 0) return m == 0 ? ZERO_BLOCK_EXP : -127;
    int e = E - 127;
    const int n = e + 1;
    const int a = n > 0 ? n - 1 : -n;
    int jm = 0;
    if (a > 0) jm = (int)((0x582C160B05020100ull >> (8 * (31 - __clz(a)))) & 0xffull);
    if ((int)(0x800000u - m) <= jm) e += 1;
    return min(e, 127);
}

// Element code given the (possibly bf16-rounded) bit pattern and the block exponent:
// sign * min(127, floor(|x| / 2^e * 64 + 0.5)), the +0.5 being an fp32 add exactly as in
// elemwise_ops.py:64-65 (so that 0.5 - 2^-25 rounds the way the reference rounds it).
__device__ __forceinline__ int mx_code(uint32_t bits, int e, bool dead) {
    const float t = __uint_as_float(bits & 0x7fffffffu) * exp2i(-e) * 64.0f;
    const float r = floorf(t + 0.5f);
    int c = (int)fminf(r, 127.0f);
    if (dead) c = 0;
    return (bits >> 31) ? -c : c;
}

// One warp quantizes one 32-wide block held one element per lane (padding lanes pass 0).
// Returns the lane's code; e_out = block exponent (A2), ep_out = predictor exponent (A3:
// floor(log2(max|MX|)) == e for every non-zero in-contract block, -126 for a zero block).
__device__ __forceinline__ int quantize_block_warp(float x, bool bf16, bool flush,
                                                   int& e_out, int& ep_out) {
    uint32_t b = __float_as_uint(x);
    if (bf16) b = bf16_half_away(b);
    const uint32_t mx = __reduce_max_sync(FULL, b & 0x7fffffffu);
    const int e = mx_shared_exp(mx);
    const bool dead = flush && e <= -127;           // mx_ops.py:282-283
    e_out = e;
    ep_out = dead ? ZERO_BLOCK_EXP : e;
    return mx_code(b, e, dead);
}

// float -> u32 key whose unsigned order equals the float order (-0 canonicalised to +0 first).
// Negative values map to 0x80000000 - magnitude (not to ~bits): a subtraction keeps the trailing
// zero bits that these scores have (small integers times a power of two), so the radix select
// only has to resolve the few bit positions that really differ between keys.
__device__ __forceinline__ uint32_t ordered_key(float s) {
    const uint32_t b = __float_as_uint(s + 0.0f);
    return (b & 0x80000000u) ? 0x80000000u - (b & 0x7fffffffu) : b | 0x80000000u;
}

// n_b - 2*p as an exact float without an int->float conversion:
// (2^23 + p) * -2 + (2^24 + n_b), one FFMA, exact because n_b is even.
__device__ __forceinline__ float signed_count(int popc, float two24_plus_nb) {
    return fmaf(__uint_as_float(0x4B000000u | (uint32_t)popc), -2.0f, two24_plus_nb);
}

// Keep only the m lowest set bits of x.
__device__ __forceinline__ uint32_t keep_lowest_bits(uint32_t x, int m) {
    uint32_t y = 0;
    for (int t = 0; t < m; ++t) {
        const uint32_t low = x & (0u - x);
        y |= low;
        x ^= low;
    }
    return y;
}

// exp(x) for x <= 0, branch-free (the softmax epilogue evaluates it for every key position of a
// row under a per-thread predicate, so divergence would serialise it).  x*log2(e) is split into
// n = rint(.) and a remainder f in [-0.5, 0.5] carried in two FMAs (hi/lo parts of log2 e), so the
// argument error does not grow with |x|; 2^f comes from MUFU.EX2 (<= 2 ulp), 2^n is added into the
// exponent field.  x is clamped at -87 (exp(-87) ~ 1.6e-38, the last normal binade).
__device__ __forceinline__ float exp_nonpos(float x) {
    x = fmaxf(x, -87.0f);
    const float t = fmaf(x, 1.4426950216293335f, 12582912.0f);         // 1.5 * 2^23 + rint(x * log2e)
    const float n = t - 12582912.0f;
    float f = fmaf(x, 1.4426950216293335f, -n);
    f = fmaf(x, 1.9259629911266175e-8f, f);
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(f));
    return __uint_as_float(__float_as_uint(r) + (__float_as_uint(t) << 23));
}

// exp(x), x <= 0, for the streamed long-sequence kernel: MUFU.EX2 on fl(x * log2 e).  Relative error <= 2 ulp (MUFU) +
// 0.9e-7 |x| (the rounded product; -inf and anything below -87.3 give +0).  The second term only grows where exp(x) no longer
// matters: a key 10 below the row maximum carries 4.5e-5 of its weight and 9e-7 of relative error, and can change an MXINT8
// code of P only in a 32-key window whose every key is that small (one step there is < 1e-6 of the row's largest p).
__device__ __forceinline__ float exp_fast_nonpos(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fmul_rn(x, 1.4426950408889634f)));
    return r;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

}  // namespace mxp
