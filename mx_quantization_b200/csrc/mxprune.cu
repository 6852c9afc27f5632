// libmxprune: MXINT8 exponent-sign pruned attention for sm_100a behind the C ABI of
// include/mxprune.h.  See DESIGN.md for the data layout and the roofline of each kernel.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "mxprune.h"
#include "mxprune_host.cuh"
#include "mxprune_device.cuh"
#include "mxprune_predict.cuh"
#include "mxprune_attend.cuh"
#include "mxprune_attend_long.cuh"
#include "mxprune_predict_tc.cuh"
#include "mxprune_predict_long_tc.cuh"
#include "mxprune_predict_wide.cuh"
#include "mxprune_linear.cuh"

using namespace mxp;

namespace {

constexpr int MAX_HD = 128;
constexpr int MAX_KEYS = 8192;        // mxp_limits(): the most keys the attention entry points accept
constexpr int MAX_KEYS_FUSED = 256;   // keys held in registers, 8 per lane

int check_view(const char* name, const void* p, int64_t sB, int64_t sH, int64_t sN, int hd, int dt = DT_F32) {
    if (!p) return fail(MXP_E_BADARG, "%s: null pointer", name);
    const int64_t m = dt == DT_F32 ? 3 : 7;                 // 16 bytes of elements - 1
    if (((uintptr_t)p & 15) || (sB & m) || (sH & m) || (sN & m))
        return fail(MXP_E_BADARG, "%s: base pointer and strides must be 16-byte aligned (strides multiples of %d elements)",
                    name, (int)m + 1);
    if (sN < hd) return fail(MXP_E_BADARG, "%s: row stride %lld < head_dim %d", name, (long long)sN, hd);
    return MXP_OK;
}

int check_shape(int B, int H, int Nq, int Nk, int hd, int bfloat_bits) {
    if (B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0) return fail(MXP_E_BADARG, "empty shape B=%d H=%d Nq=%d Nk=%d", B, H, Nq, Nk);
    if (hd < 4 || hd > MAX_HD || (hd & 3)) return fail(MXP_E_UNSUPPORTED, "head_dim %d: need a multiple of 4 in [4,%d]", hd, MAX_HD);
    if (bfloat_bits != 16 && bfloat_bits != 32) return fail(MXP_E_UNSUPPORTED, "bfloat=%d: only 16 or 32 are on the path", bfloat_bits);
    if ((int64_t)B * H > 0x7fffffffLL) return fail(MXP_E_UNSUPPORTED, "B*H too large");
    return MXP_OK;
}

// the entry points that take keys check their count up front, before any launch; the quantizer takes any row count
int check_keys(int Nk) {
    if (Nk > MAX_KEYS) return fail(MXP_E_UNSUPPORTED, "Nk=%d: at most %d keys (mxp_limits)", Nk, MAX_KEYS);
    return MXP_OK;
}

int check_dtype(const char* name, int dt) {
    if (dt != DT_F32 && dt != DT_BF16 && dt != DT_F16)
        return fail(MXP_E_BADARG, "%s: element type %d is not MXP_DT_F32, MXP_DT_BF16 or MXP_DT_F16", name, dt);
    return MXP_OK;
}

// the scope of 16-bit activations (include/mxprune.h): the tensor-core kernels, head_dim a multiple of 8 in [32, 128]
int check_half_scope(int dt, int hd) {
    if (dt == DT_F32) return MXP_OK;
    if (g_attn_path != 0 || g_predict_path != 0)
        return fail(MXP_E_UNSUPPORTED, "16-bit inputs need the tensor-core predictor and attention paths (the default)");
    if (hd < 32 || (hd & 7))
        return fail(MXP_E_UNSUPPORTED, "head_dim %d: 16-bit inputs need a multiple of 8 in [32, 128]", hd);
    return MXP_OK;
}

inline int row_splits(int heads, int Nq) {
    // enough CTAs for ~4 per SM when B*H is small; 1 when the grid is already large
    const int want = 148 * 4;
    int s = (want + heads - 1) / heads;
    const int max_s = (Nq + WARPS * 4 - 1) / (WARPS * 4);   // >= 4 rows per warp: staging is per CTA
    if (s > max_s) s = max_s;
    return s < 1 ? 1 : s;
}

// ------------------------------------------------------------------------------------
// K0a: standalone exponent-sign approximation (+-2^e per element, mxp_exp_sign_approx), one warp per row
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS)
k_quantize(View x, int rows_per_bh, int H, int64_t total_rows, int hd, int bf16, int flush,
           float* __restrict__ approx) {
    const int lane = threadIdx.x & 31;
    const int nb = (hd + 31) >> 5;
    for (int64_t row = (int64_t)blockIdx.x * WARPS + (threadIdx.x >> 5); row < total_rows;
         row += (int64_t)gridDim.x * WARPS) {
        const int64_t bh = row / rows_per_bh;
        const int n = (int)(row - bh * rows_per_bh);
        const float* xr = x.p + (bh / H) * x.sB + (bh % H) * x.sH + (int64_t)n * x.sN;
        for (int b = 0; b < nb; ++b) {
            const int d = b * 32 + lane;
            const float v = d < hd ? __ldg(xr + d) : 0.f;
            int e, ep;
            const int c = quantize_block_warp(v, bf16, flush, e, ep);
            if (d < hd) approx[row * hd + d] = c < 0 ? -exp2i(ep) : exp2i(ep);
        }
    }
}

// ------------------------------------------------------------------------------------
// K0b: the stand-alone quantizer proper (codes / exps / sign words): ONE THREAD PER MX BLOCK with the F2I-free block
// arithmetic of the fused kernels (quantize_block_thread, mxprune_predict_tc.cuh).  Consecutive threads take
// consecutive blocks of a row, so a warp reads 4 KB of contiguous fp32 with eight independent 128-bit loads per
// thread and writes 1 KB of contiguous codes.  Replaces the reference's quantize_mx_innermost / _by_tile CUDA
// kernels (microxscaling/mx/cpp/mx.cuh:57-158) on this path: tools/bench_quant.py times them side by side.
// ------------------------------------------------------------------------------------
template <bool SIGNS, int DT = DT_F32>
__global__ void __launch_bounds__(256)
k_quantize_blocks(View x, int rows_per_bh, int H, int64_t total_rows, int hd, int nb, int bf16, int flush,
                  int8_t* __restrict__ codes, int8_t* __restrict__ exps, uint32_t* __restrict__ signs) {
    const int64_t total = total_rows * nb;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = t / nb;
        const int b = (int)(t - row * nb);
        const int64_t bh = row / rows_per_bh;
        const int n = (int)(row - bh * rows_per_bh);
        const float* src = view_elem<DT>(x.p, (bh / H) * x.sB + (bh % H) * x.sH + (int64_t)n * x.sN + 32 * b);
        const int nd = min(32, hd - 32 * b);
        uint32_t xv[32];
        load_block_bits<DT>(src, nd, true, xv);
        BlockQ r;
        quantize_block_thread<true, false>(xv, nd, bf16 != 0, flush != 0, r);
        exps[row * nb + b] = (int8_t)r.e;
        uint32_t* dst = reinterpret_cast<uint32_t*>(codes + row * hd + 32 * b);
        // two 16-byte stores only for a full block with 16-byte aligned rows: a partial last block (hd % 32 == 16)
        // writes its own nd bytes, not the first codes of the next row
        if ((hd & 15) == 0 && nd == 32) {
            reinterpret_cast<uint4*>(dst)[0] = make_uint4(r.cw[0], r.cw[1], r.cw[2], r.cw[3]);
            reinterpret_cast<uint4*>(dst)[1] = make_uint4(r.cw[4], r.cw[5], r.cw[6], r.cw[7]);
        } else {
#pragma unroll
            for (int v = 0; v < 8; ++v)
                if (4 * v < nd) dst[v] = r.cw[v];
        }
        if (SIGNS) {
            // sign word in natural element order: bit d = (code d < 0); four code bytes -> four bits per multiply
            uint32_t sw = 0u;
#pragma unroll
            for (int v = 0; v < 8; ++v)
                sw |= (((((r.cw[v] >> 7) & 0x01010101u) * 0x01020408u) >> 24) & 0xfu) << (4 * v);
            signs[row * nb + b] = sw;
        }
    }
}

// ------------------------------------------------------------------------------------
// Predictor parameters
// ------------------------------------------------------------------------------------
// Quantize the Nk key rows of one head into shared memory: sign words + 2^e weights.
// All warps of the CTA cooperate, one row per warp per step.
template <int NB>
__device__ __forceinline__ void stage_keys(const PredParams& p, int head, int nkp,
                                           uint32_t* s_ksign, float* s_kw) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bb = head / p.H, hh = head % p.H;
    const float* kb = p.k.p + bb * p.k.sB + hh * p.k.sH;
    for (int j = warp; j < nkp; j += WARPS) {
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const int d = b * 32 + lane;
            const float x = (j < p.Nk && d < p.hd) ? __ldg(kb + (int64_t)j * p.k.sN + d) : 0.f;
            int e, ep;
            const int c = quantize_block_warp(x, p.bf16, p.flush, e, ep);
            const uint32_t sw = __ballot_sync(FULL, c < 0);
            if (lane == 0) {
                s_ksign[b * nkp + j] = sw;
                s_kw[b * nkp + j] = j < p.Nk ? exp2i(ep) : 0.f;
            }
        }
    }
}

// Quantize one query row held by a warp: warp-uniform sign words and 2^e weights.
template <int NB>
__device__ __forceinline__ void quantize_query_row(const PredParams& p, const float* qrow,
                                                   uint32_t (&sq)[NB], float (&wq)[NB]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int d = b * 32 + lane;
        const float x = d < p.hd ? __ldg(qrow + d) : 0.f;
        int e, ep;
        const int c = quantize_block_warp(x, p.bf16, p.flush, e, ep);
        sq[b] = __ballot_sync(FULL, c < 0);
        wq[b] = exp2i(ep);
    }
}

template <int NB>
__device__ __forceinline__ float block_width_const(int b, int hd) {
    // 2^24 + n_b  (n_b = real dims in block b), exactly representable since n_b is even
    const int nb_w = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
    return 16777216.0f + (float)nb_w;
}

// score = sum_b 2^(eq_b + ek_b) * (n_b - 2 popc(sq_b ^ sk_b)), accumulated over b ascending in
// fp32 (every product is exact; the sum is exact inside a 24-bit window - SURVEY 8a note ii).
template <int NB>
__device__ __forceinline__ float pred_score(const uint32_t (&sk)[NB], const float (&wk)[NB],
                                            const uint32_t (&sq)[NB], const float (&wq)[NB],
                                            const float (&c24)[NB]) {
    float s = 0.f;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const float cnt = signed_count(__popc(sk[b] ^ sq[b]), c24[b]);
        const float t = wk[b] * cnt;
        s = (b == 0) ? t * wq[0] : fmaf(t, wq[b], s);
    }
    return s;
}

// ------------------------------------------------------------------------------------
// K1-debug: dense predicted scores (parity aid).  Same staging and scoring code.
// ------------------------------------------------------------------------------------
template <int NB>
__global__ void __launch_bounds__(THREADS)
k_predict_scores(const PredParams p, int nkp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* s_ksign = reinterpret_cast<uint32_t*>(smem_raw);
    float* s_kw = reinterpret_cast<float*>(s_ksign + NB * nkp);
    const int head = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    stage_keys<NB>(p, head, nkp, s_ksign, s_kw);
    __syncthreads();
    float c24[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) c24[b] = block_width_const<NB>(b, p.hd);
    const int bb = head / p.H, hh = head % p.H;
    const float* qb = p.q.p + bb * p.q.sB + hh * p.q.sH;
    for (int i = blockIdx.y * WARPS + warp; i < p.Nq; i += WARPS * gridDim.y) {
        const int64_t row = (int64_t)head * p.Nq + i;
        uint32_t sq[NB];
        float wq[NB];
        quantize_query_row<NB>(p, qb + (int64_t)i * p.q.sN, sq, wq);
        for (int j = lane; j < p.Nk; j += 32) {
            uint32_t sk[NB];
            float wk[NB];
#pragma unroll
            for (int b = 0; b < NB; ++b) { sk[b] = s_ksign[b * nkp + j]; wk[b] = s_kw[b * nkp + j]; }
            p.scores[row * p.Nk + j] = pred_score<NB>(sk, wk, sq, wq, c24) + 0.0f;
        }
    }
}

// ------------------------------------------------------------------------------------
// K2 (Nk <= 256): exact MXINT8 attention over the kept keys of each row.
// One CTA per (head, row split).  Staged once per CTA in shared memory:
//   s_kt   [hd/4][NKP+1] u32   K codes, word c of key j (4 consecutive dims)
//   s_kwf  [NB][NKP]     f32   2^(ek-6)
//   s_v    [KPL][2][hd]  16 B  V codes quantised along TOKENS: window r, half, column d ->
//                              16 consecutive tokens of column d (dp4a runs along tokens)
//   s_vef  [KPL][hd]     f32   2^(eV-6) per (token window, column)
//   s_p    [WARPS][NKP]  u8    P codes of the row a warp is working on, dense key positions
// One warp per query row; lane l owns key positions l, l+32, ... = one P window per step.
// ------------------------------------------------------------------------------------
struct AttnCoreParams {          // CUDA-core (dp4a) attention path: consumes compact codes
    const int8_t *q_codes, *q_exps, *k_codes, *k_exps;
    View v;
    const uint32_t* mask;
    int B, H, Nq, Nk, hd;
    float scale;
    int bf16, flush;
    float* out;
    int64_t o_sB, o_sH, o_sN;
};

struct AttnSmem {
    int kt_stride;      // NKP + 1
    size_t off_kwf, off_vef, off_v, off_p, total;
};

__host__ __device__ inline AttnSmem attn_smem_layout(int nb, int kpl, int hd) {
    AttnSmem L;
    const int nkp = kpl * 32, hw = hd >> 2;
    L.kt_stride = nkp + 1;
    size_t o = (size_t)hw * L.kt_stride * 4;
    L.off_kwf = o; o += (size_t)nb * nkp * 4;
    L.off_vef = o; o += (size_t)kpl * hd * 4;
    o = (o + 15) & ~(size_t)15;
    L.off_v = o;   o += (size_t)kpl * 2 * hd * 16;
    L.off_p = o;   o += (size_t)WARPS * nkp;
    L.total = o;
    return L;
}

template <int NB, int KPL>
__global__ void __launch_bounds__(THREADS)
k_sparse_attention(const AttnCoreParams p) {
    constexpr int NKP = KPL * 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int hd = p.hd, HW = hd >> 2, Nk = p.Nk, Nq = p.Nq;
    const AttnSmem L = attn_smem_layout(NB, KPL, hd);
    uint32_t* s_kt = reinterpret_cast<uint32_t*>(smem_raw);
    float* s_kwf = reinterpret_cast<float*>(smem_raw + L.off_kwf);
    float* s_vef = reinterpret_cast<float*>(smem_raw + L.off_vef);
    uint4* s_v = reinterpret_cast<uint4*>(smem_raw + L.off_v);
    unsigned char* s_p = smem_raw + L.off_p;
    const int KS = L.kt_stride;

    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool bf16 = p.bf16, flush = p.flush;

    // ---- stage K codes (transposed to [word][key]) and 2^(ek-6)
    {
        const uint32_t* kc = reinterpret_cast<const uint32_t*>(p.k_codes + (int64_t)head * Nk * hd);
        for (int t = threadIdx.x; t < NKP * HW; t += THREADS) {
            const int j = t / HW, c = t - j * HW;
            s_kt[c * KS + j] = j < Nk ? __ldg(kc + t) : 0u;
        }
        const int8_t* ke = p.k_exps + (int64_t)head * Nk * NB;
        for (int t = threadIdx.x; t < NKP * NB; t += THREADS) {
            const int j = t / NB, b = t - j * NB;
            s_kwf[b * NKP + j] = j < Nk ? exp2i((int)ke[t] - 6) : 0.f;
        }
    }
    // ---- stage V: quantise along tokens, 32-token windows per column (matmul.py:76-83)
    {
        const float* vb = p.v.p + bb * p.v.sB + hh * p.v.sH;
        for (int r = warp; r < KPL; r += WARPS) {
            for (int dd = 0; dd < NB; ++dd) {
                const int d = dd * 32 + lane;
                uint32_t xb[32];
                uint32_t mx = 0u;
#pragma unroll
                for (int t = 0; t < 32; ++t) {
                    const int j = r * 32 + t;
                    const float x = (d < hd && j < Nk) ? __ldg(vb + (int64_t)j * p.v.sN + d) : 0.f;
                    uint32_t b = __float_as_uint(x);
                    if (bf16) b = bf16_half_away(b);
                    xb[t] = b;
                    mx = max(mx, b & 0x7fffffffu);
                }
                const int e = mx_shared_exp(mx);
                const bool dead = flush && e <= -127;
                uint32_t w[8];
#pragma unroll
                for (int qd = 0; qd < 8; ++qd) {
                    uint32_t word = 0u;
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        word |= ((uint32_t)mx_code(xb[qd * 4 + t], e, dead) & 0xffu) << (8 * t);
                    w[qd] = word;
                }
                if (d < hd) {
                    s_v[(r * 2 + 0) * hd + d] = make_uint4(w[0], w[1], w[2], w[3]);
                    s_v[(r * 2 + 1) * hd + d] = make_uint4(w[4], w[5], w[6], w[7]);
                    s_vef[r * hd + d] = exp2i(e - 6);
                }
            }
        }
    }
    __syncthreads();

    const int NW = (Nk + 31) >> 5;
    unsigned char* my_p = s_p + warp * NKP;
    for (int i = blockIdx.y * WARPS + warp; i < Nq; i += WARPS * gridDim.y) {
        const int64_t row = (int64_t)head * Nq + i;
        const uint32_t mymask = lane < NW ? __ldg(p.mask + row * NW + lane) : 0u;
        const uint32_t myq = lane < HW
            ? __ldg(reinterpret_cast<const uint32_t*>(p.q_codes + row * hd) + lane) : 0u;
        int qw[NB * 8];
#pragma unroll
        for (int c = 0; c < NB * 8; ++c) qw[c] = (int)__shfl_sync(FULL, myq, c);
        float wqf[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) wqf[b] = exp2i((int)__ldg(p.q_exps + row * NB + b) - 6);

        // ---- A7: true scores at the kept positions (block-exact int8 dots, fp32 combine)
        float val[KPL];
        float m = -INFINITY;
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            const int j = r * 32 + lane;
            float s = 0.f;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                int acc = 0;
#pragma unroll
                for (int c8 = 0; c8 < 8; ++c8) {
                    const int c = b * 8 + c8;
                    if (c < HW) acc = __dp4a(qw[c], (int)s_kt[c * KS + j], acc);
                }
                const float t = (float)acc * (wqf[b] * s_kwf[b * NKP + j]);
                s = (b == 0) ? t : s + t;
            }
            if (bf16) s = bf16_half_away(s);
            const float tv = s * p.scale;
            const bool kept = (__shfl_sync(FULL, mymask, r) >> lane) & 1u;
            val[r] = kept ? tv : -INFINITY;
            m = fmaxf(m, val[r]);
        }
        // ---- softmax over the kept keys (fp32)
        m = warp_max(m);
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            val[r] = expf(val[r] - m);      // expf(-inf) == 0 for pruned positions
            sum += val[r];
        }
        sum = warp_sum(sum);
        // ---- A8: P -> MXINT8 per 32-key window of original positions
        float pscale[KPL];
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            uint32_t pb = __float_as_uint(val[r] / sum);
            if (bf16) pb = bf16_half_away(pb);
            const uint32_t mx = __reduce_max_sync(FULL, pb);
            int c = 0;
            pscale[r] = 0.f;
            if (mx != 0u) {
                const int e = mx_shared_exp(mx);
                const bool dead = flush && e <= -127;
                c = mx_code(pb, e, dead);
                pscale[r] = exp2i(e - 6);
            }
            my_p[r * 32 + lane] = (unsigned char)c;
        }
        __syncwarp();
        // ---- P.V: int8 dot along the 32 tokens of each window, exponent rescale in fp32
        float o[NB];
#pragma unroll
        for (int dd = 0; dd < NB; ++dd) o[dd] = 0.f;
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            if (pscale[r] != 0.f) {
                const uint4 pa = *reinterpret_cast<const uint4*>(my_p + r * 32);
                const uint4 pc = *reinterpret_cast<const uint4*>(my_p + r * 32 + 16);
#pragma unroll
                for (int dd = 0; dd < NB; ++dd) {
                    const int d = dd * 32 + lane;
                    if (d < hd) {
                        const uint4 va = s_v[(r * 2 + 0) * hd + d];
                        const uint4 vc = s_v[(r * 2 + 1) * hd + d];
                        int acc = __dp4a((int)pa.x, (int)va.x, 0);
                        acc = __dp4a((int)pa.y, (int)va.y, acc);
                        acc = __dp4a((int)pa.z, (int)va.z, acc);
                        acc = __dp4a((int)pa.w, (int)va.w, acc);
                        acc = __dp4a((int)pc.x, (int)vc.x, acc);
                        acc = __dp4a((int)pc.y, (int)vc.y, acc);
                        acc = __dp4a((int)pc.z, (int)vc.z, acc);
                        acc = __dp4a((int)pc.w, (int)vc.w, acc);
                        o[dd] = fmaf((float)acc, pscale[r] * s_vef[r * hd + d], o[dd]);
                    }
                }
            }
        }
        __syncwarp();
        float* orow = p.out + bb * p.o_sB + hh * p.o_sH + (int64_t)i * p.o_sN;
#pragma unroll
        for (int dd = 0; dd < NB; ++dd) {
            const int d = dd * 32 + lane;
            if (d < hd) orow[d] = bf16 ? bf16_half_away(o[dd]) : o[dd];
        }
    }
}

// ------------------------------------------------------------------------------------
// dispatch helpers
// ------------------------------------------------------------------------------------
inline int pick_kpl(int Nk) {
    const int nw = (Nk + 31) / 32;
    if (nw <= 1) return 1;
    if (nw <= 2) return 2;
    if (nw <= 4) return 4;
    if (nw <= 7) return 7;
    return 8;
}

template <int NB, int DT = DT_F32, bool BIAS = false>
int launch_predict_topk_long(const PredParams& p, cudaStream_t st) {
    if (DT == DT_F32 && p.dt == DT_BF16) return launch_predict_topk_long<NB, DT_BF16, BIAS>(p, st);
    if (DT == DT_F32 && p.dt == DT_F16) return launch_predict_topk_long<NB, DT_F16, BIAS>(p, st);
    if (!BIAS && p.key_bias) return launch_predict_topk_long<NB, DT, true>(p, st);
    const K1LSmem L = k1l_smem_layout(NB, p.Nk, BIAS);
    // the staged bias (4 bytes per key) takes the layout past 200 KiB at 8192 keys and NB = 4; 227 KiB still hold it
    const size_t limit = BIAS ? SMEM_PER_SM : 200 * 1024;
    if (L.total > limit)
        return fail(MXP_E_UNSUPPORTED, "Nk=%d: key records need %zu bytes of shared memory (limit %zu bytes)", p.Nk,
                    L.total, limit);
    cudaError_t e = cudaFuncSetAttribute(k_predict_topk_long<NB, DT, BIAS>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
    if (e != cudaSuccess) return fail(MXP_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int heads = p.B * p.H;
    const int tiles = (p.Nq + K1T - 1) / K1T;
    int splits = (148 * 2 + heads - 1) / heads;
    if (splits > tiles) splits = tiles;
    if (splits < 1) splits = 1;
    dim3 grid((unsigned)heads, (unsigned)splits);
    k_predict_topk_long<NB, DT, BIAS><<<grid, K1T, L.total, st>>>(p);
    return check_launch("k_predict_topk_long");
}

template <int NB>
int launch_predict_topk_nb(const PredParams& p, cudaStream_t st) {
    if (p.Nk > K1_MAX_KEYS) return launch_predict_topk_long<NB>(p, st);
    if (p.dt != DT_F32)                     // only reached outside the tensor-core kernel's domain
        return fail(MXP_E_UNSUPPORTED, "16-bit q/k: Nk=%d hd=%d is outside the tensor-core predictor's domain", p.Nk, p.hd);
    const K1Smem L = k1_smem_layout(NB, p.Nk);
    cudaError_t e = cudaFuncSetAttribute(k_predict_topk_rows<NB>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
    if (e != cudaSuccess) return fail(MXP_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    const int heads = p.B * p.H;
    const int tiles = (p.Nq + K1T - 1) / K1T;
    int splits = (148 * 3 + heads - 1) / heads;         // 3 CTAs per SM resident
    if (splits > tiles) splits = tiles;
    if (splits < 1) splits = 1;
    dim3 grid((unsigned)heads, (unsigned)splits);
    k_predict_topk_rows<NB><<<grid, K1T, L.total, st>>>(p);
    return check_launch("k_predict_topk_rows");
}

template <int NB, int KPL>
int launch_attn_one(const AttnCoreParams& p, dim3 grid, cudaStream_t st) {
    const AttnSmem L = attn_smem_layout(NB, KPL, p.hd);
    cudaError_t e = cudaFuncSetAttribute(k_sparse_attention<NB, KPL>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total);
    if (e != cudaSuccess) return fail(MXP_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    k_sparse_attention<NB, KPL><<<grid, THREADS, L.total, st>>>(p);
    return check_launch("k_sparse_attention");
}

template <int NB>
int launch_attn_nb(const AttnCoreParams& p, dim3 grid, cudaStream_t st) {
    switch (pick_kpl(p.Nk)) {
        case 1: return launch_attn_one<NB, 1>(p, grid, st);
        case 2: return launch_attn_one<NB, 2>(p, grid, st);
        case 4: return launch_attn_one<NB, 4>(p, grid, st);
        case 7: return launch_attn_one<NB, 7>(p, grid, st);
        default: return launch_attn_one<NB, 8>(p, grid, st);
    }
}

thread_local cudaEvent_t g_ev[4] = {nullptr, nullptr, nullptr, nullptr};
thread_local bool g_profile = false;
inline void prof_mark(int i, cudaStream_t st) {
    if (!g_profile) return;
    if (!g_ev[i]) cudaEventCreate(&g_ev[i]);
    cudaEventRecord(g_ev[i], st);
}

// k_attend_pair with output element type OT (== p.out_dt); grid and dyn from launch_attend
template <int OT>
int launch_attend_pair_ot(const AttnParams& p, dim3 grid, size_t dyn, cudaStream_t st) {
    MXP_ENSURE_DYN_SMEM((k_attend_pair<true, false, OT>), 160 * 1024);
    MXP_ENSURE_DYN_SMEM((k_attend_pair<false, false, OT>), 160 * 1024);
    MXP_ENSURE_DYN_SMEM((k_attend_pair<true, true, OT>), 160 * 1024);
    MXP_ENSURE_DYN_SMEM((k_attend_pair<false, true, OT>), 160 * 1024);
    if (p.key_bias) {
        if (p.bf16) k_attend_pair<true, true, OT><<<grid, K2P_T, dyn, st>>>(p);
        else k_attend_pair<false, true, OT><<<grid, K2P_T, dyn, st>>>(p);
    } else {
        if (p.bf16) k_attend_pair<true, false, OT><<<grid, K2P_T, dyn, st>>>(p);
        else k_attend_pair<false, false, OT><<<grid, K2P_T, dyn, st>>>(p);
    }
    return check_launch("k_attend_pair");
}
// Exact attention over the MMA-ready operands: Nk > 256 streams key blocks of 128 (k_attend_long_pair,
// mxprune_attend_long.cuh), one key block runs k_attend_pair (two lanes per query row, 256 threads).
int launch_attend(const AttnParams& p, cudaStream_t st) {
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    if (!O.single) return launch_attend_long_pair(p, st);
    const K2Smem L = k2_smem_layout(O);
    if (L.total > 160 * 1024) return fail(MXP_E_UNSUPPORTED, "attention operands need %zu bytes of shared memory", L.total);
    const int heads = p.B * p.H;
    int splits = (148 * 2 + heads - 1) / heads;
    if (splits > O.q_tiles) splits = O.q_tiles;
    if (splits < 1) splits = 1;
    dim3 grid((unsigned)heads, (unsigned)splits);
    // Never let more CTAs become resident on an SM than its 512 TMEM columns can serve: a CTA
    // whose tcgen05.alloc cannot be satisfied would sit blocked inside the allocator.  Residency is
    // bounded through the dynamic shared-memory request (227 KiB per SM).
    const int max_ctas = 512 / k2p_tmem_cols(O);
    size_t dyn = L.total;
    const size_t floor_bytes = (size_t)232448 / (size_t)(max_ctas + 1) + 1024;
    if (dyn < floor_bytes) dyn = floor_bytes;
    if (p.out_dt == DT_BF16) return launch_attend_pair_ot<DT_BF16>(p, grid, dyn, st);
    if (p.out_dt == DT_F16) return launch_attend_pair_ot<DT_F16>(p, grid, dyn, st);
    return launch_attend_pair_ot<DT_F32>(p, grid, dyn, st);
}

// dt: element type of the V view (DT_*)
int launch_prep_v(const View& v, int B, int H, int Nq, int Nk, int hd, int bf16, int flush, unsigned char* v_op,
                  cudaStream_t st, int dt = DT_F32) {
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    VPrepParams vp{v, H, Nq, Nk, hd, bf16, flush, v_op};
    dim3 grid((unsigned)(B * H), (unsigned)((O.nblk * O.wpb + 3) / 4));
    if (dt == DT_BF16) k_prep_v<DT_BF16><<<grid, K2T, 0, st>>>(vp);
    else if (dt == DT_F16) k_prep_v<DT_F16><<<grid, K2T, 0, st>>>(vp);
    else k_prep_v<<<grid, K2T, 0, st>>>(vp);
    return check_launch("k_prep_v");
}

int launch_codes_to_ops(const int8_t* codes, const int8_t* exps, unsigned char* ops, int heads, int Nq, int Nk,
                        int hd, int which, cudaStream_t st) {
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const int64_t total = (int64_t)heads * (which == 0 ? O.q_tiles * K2T : O.nblk * O.kb_rows) * (O.hdp >> 3);
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_codes_to_ops<<<(unsigned)blocks, 256, 0, st>>>(codes, exps, ops, heads, Nq, Nk, hd, which);
    return check_launch("k_codes_to_ops");
}

struct OpsBytes { size_t q, k, v; };
inline OpsBytes ops_bytes(int B, int H, int Nq, int Nk, int hd) {
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const size_t bh = (size_t)B * H;
    return OpsBytes{bh * O.q_head_bytes, bh * O.k_head_bytes, bh * O.v_head_bytes};
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// returns 1 if the shape is outside the tensor-core kernel's domain (caller uses the CUDA-core kernel)
static int try_predict_topk_tc(const PredParams& p, cudaStream_t st, int* rc_out) {
    if (g_predict_path != 0 || p.Nk > 256 || p.hd < 32 || (p.hd & 7)) return 1;
    K1cMaps maps;
    if (!make_view_maps(p.q, p.B, p.H, p.Nq, p.hd, &maps.q_main, &maps.q_tail, p.dt) ||
        !make_view_maps(p.k, p.B, p.H, p.Nk, p.hd, &maps.k_main, &maps.k_tail, p.dt)) {
        if (p.dt == DT_F32) return 1;
        *rc_out = fail(MXP_E_UNSUPPORTED, "16-bit q/k: the views cannot be described by a TMA tensor map");
        return 0;
    }
    // step = 64 G rows (G = 2 when a 64-row box gives fewer than 256 block tasks); ring depth: as many
    // slots as fit with two CTAs per SM
    const size_t per_cta1 = K1C_PER_CTA1;
    const int nc = p.Nk <= 32 ? 1 : p.Nk <= 64 ? 2 : p.Nk <= 128 ? 4 : p.Nk <= 224 ? 7 : 8;
    const bool biased = p.key_bias != nullptr;
    const int G = k1c_G(p.hd, nc, biased), ring = k1c_ring(p.hd, nc, biased);
    K1cSmem L = k1c_smem_layout(p.hd, nc, ring, G, biased);
    if (L.total > per_cta1) return 1;
    const int heads = p.B * p.H;
    const int tiles = (p.Nq + K1C_TILE - 1) / K1C_TILE;
    int splits = (148 * 2 + heads - 1) / heads;
    if (splits > tiles) splits = tiles;
    if (splits < 1) splits = 1;
    dim3 grid((unsigned)heads, (unsigned)splits);
    // residency bounded by the 512 TMEM columns of an SM (see launch_attend)
    const int max_ctas = 512 / L.tmem_cols;
    size_t dyn = L.total;
    const size_t floor_bytes = (size_t)232448 / (size_t)(max_ctas + 1) + 1024;
    if (dyn < floor_bytes) dyn = floor_bytes;
    const bool codes = p.q_codes != nullptr || p.k_codes != nullptr;
    if (biased && codes) return 1;          // codes + bias: the CUDA-core kernel handles it
    // one instantiation policy for every element type (launch_predict_topk_tc_dt, mxprune_predict_tc.cuh); the 16-bit
    // instantiations are compiled in mxprune_predict16.cu
    *rc_out = p.dt == DT_F32 ? launch_predict_topk_tc_dt<DT_F32>(p, maps, L, dyn, grid, nc, st)
                             : launch_predict_topk_tc_16(p, maps, L, dyn, grid, nc, st);
    return 0;
}

// ---- K1-wide: partial_Q / partial_K / exact-score top-k (SURVEY 8 f3), Nk <= 256, tensor-core domain only
template <int NC, bool TWO, bool ELSA>
static int launch_predict_topk_wide_one(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn,
                                        dim3 grid, cudaStream_t st) {
    MXP_ENSURE_DYN_SMEM((k_predict_topk_wide<NC, TWO, ELSA>), 227 * 1024);
    k_predict_topk_wide<NC, TWO, ELSA><<<grid, K1C_T, dyn, st>>>(p, maps, L.ring, L.G);
    return check_launch("k_predict_topk_wide");
}

static int predict_topk_wide(const PredParams& p, cudaStream_t st) {
    if (p.Nk > 256 || p.hd < 32 || (p.hd & 7))
        return fail(MXP_E_UNSUPPORTED, "pred_mode %d needs Nk <= 256 and head_dim a multiple of 8, >= 32 (got Nk=%d hd=%d)",
                    p.pred_mode, p.Nk, p.hd);
    if (p.q_codes || p.k_codes)
        return fail(MXP_E_UNSUPPORTED, "pred_mode %d: code outputs are implemented for the exponent-sign predictor only",
                    p.pred_mode);
    K1cMaps maps;
    if (!make_view_maps(p.q, p.B, p.H, p.Nq, p.hd, &maps.q_main, &maps.q_tail) ||
        !make_view_maps(p.k, p.B, p.H, p.Nk, p.hd, &maps.k_main, &maps.k_tail))
        return fail(MXP_E_UNSUPPORTED, "pred_mode %d: the q/k views cannot be described by a TMA tensor map", p.pred_mode);
    // two_step_leading_ones carries two operand parts per side (twice the operand shared memory), ELSA keeps its
    // projection matrix in shared memory: one CTA per SM for both
    const bool two = p.pred_mode == PRED_TWO_STEP, elsa = p.pred_mode == PRED_ELSA;
    if (elsa) {
        if (!p.elsa_proj || ((uintptr_t)p.elsa_proj & 15))
            return fail(MXP_E_BADARG, "ELSA: the projection matrix must be a 16-byte aligned device pointer");
        if (p.Nq != p.Nk || p.hd > ELSA_MAX_HD)
            return fail(MXP_E_UNSUPPORTED, "ELSA needs Nq == Nk (the reference broadcasts the key norms over rows) and "
                        "head_dim <= %d (got Nq=%d Nk=%d hd=%d)", ELSA_MAX_HD, p.Nq, p.Nk, p.hd);
        if (p.key_bias) return fail(MXP_E_UNSUPPORTED, "ELSA takes no key bias (the reference's cross-attention has no ELSA branch)");
    }
    const int opw = two ? 2 : 1;
    const size_t extra = elsa ? 16 + (size_t)p.hd * p.hd * 4 : 0;
    const size_t per_cta1 = 232448 - 1024 - extra, per_cta2 = (two || elsa) ? per_cta1 : 232448 / 2 - 1024;
    const int nc = p.Nk <= 32 ? 1 : p.Nk <= 64 ? 2 : p.Nk <= 128 ? 4 : p.Nk <= 224 ? 7 : 8;
    const int nb = (p.hd + 31) / 32;
    int G = nb <= 2 ? 2 : 1;
    if (k1c_smem_layout(p.hd, nc, 2, G, false, opw).total > per_cta2) G = 1;
    int ring = K1C_MAXR;
    while (ring > (two ? 1 : 2) && k1c_smem_layout(p.hd, nc, ring, G, false, opw).total > per_cta2) --ring;
    K1cSmem L = k1c_smem_layout(p.hd, nc, ring, G, false, opw);
    if (L.total > per_cta1) return fail(MXP_E_UNSUPPORTED, "pred_mode %d: shape needs %zu bytes of shared memory", p.pred_mode, L.total);
    const int heads = p.B * p.H;
    const int tiles = (p.Nq + K1C_TILE - 1) / K1C_TILE;
    int splits = (148 * 2 + heads - 1) / heads;
    if (splits > tiles) splits = tiles;
    if (splits < 1) splits = 1;
    dim3 grid((unsigned)heads, (unsigned)splits);
    const int max_ctas = 512 / L.tmem_cols;
    size_t dyn = L.total + extra;
    const size_t floor_bytes = (size_t)232448 / (size_t)(max_ctas + 1) + 1024;
    if (dyn < floor_bytes) dyn = floor_bytes;
    if (elsa && dyn < 232448 / 2) dyn = 232448 / 2;                 // one CTA per SM (launch bounds assume it)
#define MXP_WIDE(NC_) (two ? launch_predict_topk_wide_one<NC_, true, false>(p, maps, L, dyn, grid, st)   \
                     : elsa ? launch_predict_topk_wide_one<NC_, false, true>(p, maps, L, dyn, grid, st) \
                            : launch_predict_topk_wide_one<NC_, false, false>(p, maps, L, dyn, grid, st))
    switch (nc) {
        case 1: return MXP_WIDE(1);
        case 2: return MXP_WIDE(2);
        case 4: return MXP_WIDE(4);
        case 7: return MXP_WIDE(7);
        default: return MXP_WIDE(8);
    }
#undef MXP_WIDE
}

// ---- K1-long-TC (Nk > 256): operand pre-pass + tensor-core radix select + CUDA-core clean-up ----
struct LongWsLayout { size_t q_pp, k_pp, q_ep, head_meta, flags, total; };
inline LongWsLayout long_ws_layout(int B, int H, int Nq, int Nk, int hd) {
    LongWsLayout W{};
    if (Nk <= K1_MAX_KEYS || hd < 32 || (hd & 7)) return W;
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const size_t bh = (size_t)B * H;
    size_t o = 0;
    W.q_pp = o;      o += align256(bh * O.q_head_bytes);
    W.k_pp = o;      o += align256(bh * O.k_head_bytes);
    W.q_ep = o;      o += align256(bh * (size_t)O.q_tiles * KL_TILE * 4);
    W.head_meta = o; o += align256(bh * 32);
    W.flags = o;     o += align256(bh * (size_t)Nq);
    W.total = o;
    return W;
}

// returns 1 if the shape is outside this path's domain or no workspace was supplied.  With an additive key bias the
// selection adds it to every score (k_select_long_tc<true>) and the flagged rows' kernel adds it to its fp32 keys
// (k_predict_topk_long<.., BIAS>)
static int try_predict_topk_long_tc(const PredParams& p, cudaStream_t st, int* rc_out) {
    if (g_predict_path != 0) return 1;
    const LongWsLayout W = long_ws_layout(p.B, p.H, p.Nq, p.Nk, p.hd);
    if (W.total == 0 || !p.long_ws || p.long_ws_bytes < W.total || ((uintptr_t)p.long_ws & 255)) return 1;
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    const bool biased = p.key_bias != nullptr;
    const KLSmem L = kl_smem_layout(O, biased);
    if (L.total > 227 * 1024) return 1;
    unsigned char* w = (unsigned char*)p.long_ws;
    const int heads = p.B * p.H, nb = (p.hd + 31) / 32;
    uint32_t* head_meta = (uint32_t*)(w + W.head_meta);
    uint8_t* flags = (uint8_t*)(w + W.flags);
    if (cudaMemsetAsync(head_meta, 0xFF, (size_t)heads * 32, st) != cudaSuccess) {
        *rc_out = fail(MXP_E_CUDA, "cudaMemsetAsync failed");
        return 0;
    }
    const bool codes = p.q_codes != nullptr || p.k_codes != nullptr;
    for (int which = 1; which >= 0; --which) {          // keys first (head_meta), then queries
        QuantOpsParams qp{};
        qp.x = which ? p.k : p.q;
        qp.H = p.H; qp.N = which ? p.Nk : p.Nq;
        qp.rows_pad = which ? O.nblk * O.kb_rows : O.q_tiles * KL_TILE;
        qp.hd = p.hd; qp.bf16 = p.bf16; qp.flush = p.flush; qp.which = which; qp.Nq = p.Nq; qp.Nk = p.Nk;
        qp.op = which ? p.k_op : p.q_op;
        qp.pp = w + (which ? W.k_pp : W.q_pp);
        qp.ep = which ? nullptr : (int8_t*)(w + W.q_ep);
        qp.head_meta = which ? head_meta : nullptr;
        qp.codes = which ? p.k_codes : p.q_codes;
        qp.exps = which ? p.k_exps : p.q_exps;
        const int ntask = qp.rows_pad * nb;
        int gy = (ntask + 255) / 256;
        const int want = (148 * 8 + heads - 1) / heads;
        if (gy > want) gy = want;
        dim3 grid((unsigned)heads, (unsigned)gy);
        if (p.dt == DT_BF16) {
            if (codes) k_quantize_ops<true, DT_BF16><<<grid, 256, 0, st>>>(qp);
            else k_quantize_ops<false, DT_BF16><<<grid, 256, 0, st>>>(qp);
        } else if (p.dt == DT_F16) {
            if (codes) k_quantize_ops<true, DT_F16><<<grid, 256, 0, st>>>(qp);
            else k_quantize_ops<false, DT_F16><<<grid, 256, 0, st>>>(qp);
        } else if (codes) {
            k_quantize_ops<true><<<grid, 256, 0, st>>>(qp);
        } else {
            k_quantize_ops<false><<<grid, 256, 0, st>>>(qp);
        }
        if ((*rc_out = check_launch("k_quantize_ops"))) return 0;
    }
    {
        {
            static std::atomic<uint64_t> done_{0}, done_b{0};
            if ((*rc_out = biased ? ensure_dyn_smem(k_select_long_tc<true>, 227 * 1024, done_b)
                                  : ensure_dyn_smem(k_select_long_tc<false>, 227 * 1024, done_))) return 0;
        }
        LongSelParams sp{};
        sp.q_pp = w + W.q_pp; sp.k_pp = w + W.k_pp; sp.q_ep = (const int8_t*)(w + W.q_ep);
        sp.head_meta = head_meta; sp.flags = flags; sp.mask = p.mask; sp.idx = p.idx;
        sp.H = p.H; sp.Nq = p.Nq; sp.Nk = p.Nk; sp.hd = p.hd; sp.top_k = p.top_k;
        sp.adaptive = g_fused_path.load() != 0;                     // mxp_set_fused_path(0): radix levels only (A/B)
        // one CTA (a pair of query tiles) per SM - its shared memory and 512 TMEM columns fill it; a pair is
        // ~Nk/128 times the work of a short-kernel tile: spread the pairs over enough CTAs for >= 8 waves
        const int n_pairs = (O.q_tiles + 1) / 2;
        int splits = (148 * 8 + heads - 1) / heads;
        if (splits > n_pairs) splits = n_pairs;
        if (splits < 1) splits = 1;
        // equal shares where the pair count allows: the next divisor of n_pairs (N = 4096: 16 pairs over 8 CTAs, not 4 + 3 + 3 + 3 + 3)
        for (int d = splits; d <= n_pairs && d <= 2 * splits; ++d)
            if (n_pairs % d == 0) { splits = d; break; }
        const size_t dyn = L.total;
        sp.splits = splits;
        sp.key_bias = p.key_bias; sp.kb_sB = p.kb_sB;
        if (biased) k_select_long_tc<true><<<dim3((unsigned)((size_t)heads * splits)), KL_T, dyn, st>>>(sp);
        else k_select_long_tc<false><<<dim3((unsigned)((size_t)heads * splits)), KL_T, dyn, st>>>(sp);
        if ((*rc_out = check_launch("k_select_long_tc"))) return 0;
    }
    // rows outside the integer-key window: the CUDA-core kernel, restricted to the flagged rows
    PredParams pf = p;
    pf.q_op = nullptr; pf.k_op = nullptr;
    pf.q_codes = nullptr; pf.q_exps = nullptr; pf.k_codes = nullptr; pf.k_exps = nullptr;
    pf.row_filter = flags;
    switch (nb) {
        case 1: *rc_out = launch_predict_topk_long<1>(pf, st); break;
        case 2: *rc_out = launch_predict_topk_long<2>(pf, st); break;
        case 3: *rc_out = launch_predict_topk_long<3>(pf, st); break;
        default: *rc_out = launch_predict_topk_long<4>(pf, st); break;
    }
    return 0;
}

}  // namespace

// ======================================================================================
// C ABI
// ======================================================================================
extern "C" {

int mxp_abi_version(void) { return MXP_ABI_VERSION; }
int mxp_set_attention_path(int path) {
    if (path != 0 && path != 1) return fail(MXP_E_BADARG, "attention path %d: 0 = tcgen05, 1 = CUDA-core dp4a", path);
    g_attn_path = path;
    return MXP_OK;
}
int mxp_set_predict_path(int path) {
    if (path != 0 && path != 1) return fail(MXP_E_BADARG, "predict path %d: 0 = tensor-core scoring, 1 = CUDA-core XOR/POPC", path);
    g_predict_path = path;
    return MXP_OK;
}
int mxp_set_fused_path(int path) {
    if (path < 0 || path > 2)
        return fail(MXP_E_BADARG, "fused path %d: 0 = off, 1 = where measured faster (default), 2 = wherever in domain", path);
    g_fused_path = path;
    return MXP_OK;
}
int mxp_debug_fused_pingpong(int on) {
    fused_set_pingpong(on != 0);
    return MXP_OK;
}
int mxp_debug_fused_timing(void* device_buffer) {
    fused_set_timing_buffer((unsigned long long*)device_buffer);
    return MXP_OK;
}
const char* mxp_last_error(void) { return g_err; }
int mxp_last_launch_count(void) { return g_launches; }
void mxp_limits(int* max_keys, int* max_head_dim) {
    if (max_keys) *max_keys = MAX_KEYS;
    if (max_head_dim) *max_head_dim = MAX_HD;
}

static int quantize_common(const void* xp, int dt, int64_t sB, int64_t sH, int64_t sN, int B, int H, int N,
                           int hd, int bfloat_bits, int flush, int8_t* codes, int8_t* exps,
                           uint32_t* signs, float* approx, void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, N, N, hd, bfloat_bits);
    if (rc) return rc;
    if ((rc = check_dtype("x", dt))) return rc;
    if (dt != DT_F32 && (hd & 7))          // 16-byte loads of 8 elements: a row holds whole chunks
        return fail(MXP_E_UNSUPPORTED, "head_dim %d: 16-bit x needs a multiple of 8", hd);
    rc = check_view("x", xp, sB, sH, sN, hd, dt);
    if (rc) return rc;
    const float* x = (const float*)xp;
    const int64_t rows = (int64_t)B * H * N;
    int64_t blocks = (rows + WARPS - 1) / WARPS;
    if (blocks > 148 * 16) blocks = 148 * 16;
    View v{x, sB, sH, sN};
    cudaStream_t st = (cudaStream_t)stream;
    if (approx) {
        k_quantize<<<(unsigned)blocks, THREADS, 0, st>>>(v, N, H, rows, hd, bfloat_bits == 16, flush != 0, approx);
        return check_launch("k_quantize");
    }
    const int nb = (hd + 31) / 32;
    int64_t qblocks = (rows * nb + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 32;
    if (qblocks > cap) qblocks = cap;
#define MXP_QB(S_, DT_) k_quantize_blocks<S_, DT_><<<(unsigned)qblocks, 256, 0, st>>>(v, N, H, rows, hd, nb, bfloat_bits == 16, \
                                                                               flush != 0, codes, exps, signs)
    if (dt == DT_BF16) { if (signs) MXP_QB(true, DT_BF16); else MXP_QB(false, DT_BF16); }
    else if (dt == DT_F16) { if (signs) MXP_QB(true, DT_F16); else MXP_QB(false, DT_F16); }
    else if (signs) MXP_QB(true, DT_F32);
    else MXP_QB(false, DT_F32);
#undef MXP_QB
    return check_launch("k_quantize_blocks");
}

int mxp_quantize_mxint8_dt(const void* x, int x_dtype, int64_t sB, int64_t sH, int64_t sN, int B, int H, int N,
                           int hd, int bfloat_bits, int flush, int8_t* codes, int8_t* exps,
                           uint32_t* signs, void* stream) {
    if (!codes || !exps) return fail(MXP_E_BADARG, "codes/exps: null pointer");
    return quantize_common(x, x_dtype, sB, sH, sN, B, H, N, hd, bfloat_bits, flush, codes, exps, signs, nullptr, stream);
}

int mxp_quantize_mxint8(const float* x, int64_t sB, int64_t sH, int64_t sN, int B, int H, int N,
                        int hd, int bfloat_bits, int flush, int8_t* codes, int8_t* exps,
                        uint32_t* signs, void* stream) {
    return mxp_quantize_mxint8_dt(x, MXP_DT_F32, sB, sH, sN, B, H, N, hd, bfloat_bits, flush, codes, exps, signs, stream);
}

int mxp_exp_sign_approx(const float* x, int64_t sB, int64_t sH, int64_t sN, int B, int H, int N,
                        int hd, int bfloat_bits, int flush, float* approx, void* stream) {
    if (!approx) return fail(MXP_E_BADARG, "approx: null pointer");
    return quantize_common(x, DT_F32, sB, sH, sN, B, H, N, hd, bfloat_bits, flush, nullptr, nullptr, nullptr, approx, stream);
}

int mxp_predict_scores(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                       const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                       int B, int H, int Nq, int Nk, int hd, int bfloat_bits, int flush,
                       float* scores, void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, Nq, Nk, hd, bfloat_bits);
    if (rc || (rc = check_keys(Nk))) return rc;
    if ((rc = check_view("q", q, q_sB, q_sH, q_sN, hd))) return rc;
    if ((rc = check_view("k", k, k_sB, k_sH, k_sN, hd))) return rc;
    if (!scores) return fail(MXP_E_BADARG, "scores: null pointer");
    const int nb = (hd + 31) / 32;
    const int nkp = ((Nk + 31) / 32) * 32;
    const size_t smem = (size_t)nb * nkp * 8;
    if (smem > 200 * 1024) return fail(MXP_E_UNSUPPORTED, "Nk=%d too large for the dense score aid", Nk);
    PredParams p{};
    p.q = View{q, q_sB, q_sH, q_sN};
    p.k = View{k, k_sB, k_sH, k_sN};
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.hd = hd; p.top_k = 0;
    p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
    p.scores = scores;
    dim3 grid((unsigned)(B * H), (unsigned)row_splits(B * H, Nq));
    cudaStream_t st = (cudaStream_t)stream;
#define MXP_SCORES(NB_)                                                                        \
    do {                                                                                       \
        cudaError_t e_ = cudaFuncSetAttribute(k_predict_scores<NB_>,                           \
                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
        if (e_ != cudaSuccess) return fail(MXP_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e_)); \
        k_predict_scores<NB_><<<grid, THREADS, smem, st>>>(p, nkp);                            \
    } while (0)
    switch (nb) {
        case 1: MXP_SCORES(1); break;
        case 2: MXP_SCORES(2); break;
        case 3: MXP_SCORES(3); break;
        default: MXP_SCORES(4); break;
    }
#undef MXP_SCORES
    return check_launch("k_predict_scores");
}

size_t mxp_predict_topk_workspace_bytes(int B, int H, int Nq, int Nk, int hd) {
    return long_ws_layout(B, H, Nq, Nk, hd).total;
}

static int predict_topk_impl(const PredParams& p, cudaStream_t st) {
    int rc = MXP_OK;
    if (p.pred_mode < 0 || p.pred_mode > 7) return fail(MXP_E_BADARG, "pred_mode=%d outside [0, 7]", p.pred_mode);
    if (p.pred_mode != 0) return predict_topk_wide(p, st);
    if (try_predict_topk_tc(p, st, &rc) == 0) return rc;
    if (try_predict_topk_long_tc(p, st, &rc) == 0) return rc;
    switch ((p.hd + 31) / 32) {
        case 1: return launch_predict_topk_nb<1>(p, st);
        case 2: return launch_predict_topk_nb<2>(p, st);
        case 3: return launch_predict_topk_nb<3>(p, st);
        default: return launch_predict_topk_nb<4>(p, st);
    }
}

int mxp_predict_topk_dt(const void* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                        const void* k, int64_t k_sB, int64_t k_sH, int64_t k_sN, int in_dtype,
                        int B, int H, int Nq, int Nk, int hd, int top_k, int bfloat_bits, int flush,
                        uint32_t* mask, int32_t* idx, int8_t* q_codes, int8_t* q_exps,
                        int8_t* k_codes, int8_t* k_exps, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, Nq, Nk, hd, bfloat_bits);
    if (rc || (rc = check_keys(Nk))) return rc;
    if ((rc = check_dtype("q/k", in_dtype)) || (rc = check_half_scope(in_dtype, hd))) return rc;
    if ((rc = check_view("q", q, q_sB, q_sH, q_sN, hd, in_dtype))) return rc;
    if ((rc = check_view("k", k, k_sB, k_sH, k_sN, hd, in_dtype))) return rc;
    if (!mask) return fail(MXP_E_BADARG, "mask: null pointer");
    if (top_k < 1 || top_k > Nk) return fail(MXP_E_BADARG, "top_k=%d outside [1, Nk=%d]", top_k, Nk);
    if ((q_codes == nullptr) != (q_exps == nullptr) || (k_codes == nullptr) != (k_exps == nullptr))
        return fail(MXP_E_BADARG, "codes and exps outputs must be given together");
    PredParams p{};
    p.q = View{(const float*)q, q_sB, q_sH, q_sN};
    p.k = View{(const float*)k, k_sB, k_sH, k_sN};
    p.dt = in_dtype;
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.hd = hd; p.top_k = top_k;
    p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
    p.mask = mask; p.idx = idx;
    p.q_codes = q_codes; p.q_exps = q_exps; p.k_codes = k_codes; p.k_exps = k_exps;
    p.long_ws = workspace; p.long_ws_bytes = workspace_bytes;
    return predict_topk_impl(p, (cudaStream_t)stream);
}

int mxp_predict_topk(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                     const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                     int B, int H, int Nq, int Nk, int hd, int top_k, int bfloat_bits, int flush,
                     uint32_t* mask, int32_t* idx, int8_t* q_codes, int8_t* q_exps,
                     int8_t* k_codes, int8_t* k_exps, void* workspace, size_t workspace_bytes, void* stream) {
    return mxp_predict_topk_dt(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, MXP_DT_F32, B, H, Nq, Nk, hd, top_k, bfloat_bits,
                               flush, mask, idx, q_codes, q_exps, k_codes, k_exps, workspace, workspace_bytes, stream);
}

size_t mxp_sparse_attention_workspace_bytes(int B, int H, int Nq, int Nk, int hd) {
    const OpsBytes ob = ops_bytes(B, H, Nq, Nk, hd);
    return align256(ob.q) + align256(ob.k) + align256(ob.v);
}

static int attend_core_impl(const AttnCoreParams& p, cudaStream_t st) {
    if (p.Nk > MAX_KEYS_FUSED)
        return fail(MXP_E_UNSUPPORTED, "Nk=%d: the CUDA-core attention path covers Nk <= %d", p.Nk, MAX_KEYS_FUSED);
    dim3 grid((unsigned)(p.B * p.H), (unsigned)row_splits(p.B * p.H, p.Nq));
    switch ((p.hd + 31) / 32) {
        case 1: return launch_attn_nb<1>(p, grid, st);
        case 2: return launch_attn_nb<2>(p, grid, st);
        case 3: return launch_attn_nb<3>(p, grid, st);
        default: return launch_attn_nb<4>(p, grid, st);
    }
}

int mxp_sparse_attention_dt(const int8_t* q_codes, const int8_t* q_exps, const int8_t* k_codes,
                            const int8_t* k_exps, const void* vp, int64_t v_sB, int64_t v_sH,
                            int64_t v_sN, int v_dtype, const uint32_t* mask, int B, int H, int Nq, int Nk, int hd,
                            float scale, int bfloat_bits, int flush, void* outp, int64_t o_sB,
                            int64_t o_sH, int64_t o_sN, int out_dtype, void* workspace, size_t workspace_bytes,
                            void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, Nq, Nk, hd, bfloat_bits);
    if (rc || (rc = check_keys(Nk))) return rc;
    if ((rc = check_dtype("v", v_dtype)) || (rc = check_dtype("out", out_dtype))) return rc;
    if (out_dtype != DT_F32 && out_dtype != v_dtype)
        return fail(MXP_E_BADARG, "out: element type %d must be fp32 or v's (%d)", out_dtype, v_dtype);
    if ((rc = check_half_scope(v_dtype, hd))) return rc;
    if ((rc = check_view("v", vp, v_sB, v_sH, v_sN, hd, v_dtype))) return rc;
    if ((rc = check_view("out", outp, o_sB, o_sH, o_sN, hd, out_dtype))) return rc;
    const float* v = (const float*)vp;
    float* out = (float*)outp;
    if (!q_codes || !q_exps || !k_codes || !k_exps || !mask)
        return fail(MXP_E_BADARG, "codes/exps/mask: null pointer");
    if (((uintptr_t)q_codes & 7) || ((uintptr_t)k_codes & 7) || ((uintptr_t)mask & 3))
        return fail(MXP_E_BADARG, "codes must be 8-byte aligned, mask 4-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (g_attn_path == 1) {
        AttnCoreParams p{};
        p.q_codes = q_codes; p.q_exps = q_exps; p.k_codes = k_codes; p.k_exps = k_exps;
        p.v = View{v, v_sB, v_sH, v_sN};
        p.mask = mask;
        p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.hd = hd;
        p.scale = scale; p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
        p.out = out; p.o_sB = o_sB; p.o_sH = o_sH; p.o_sN = o_sN;
        return attend_core_impl(p, st);
    }
    if (hd & 7) return fail(MXP_E_UNSUPPORTED, "head_dim %d: the tensor-core attention path needs a multiple of 8", hd);
    const size_t need = mxp_sparse_attention_workspace_bytes(B, H, Nq, Nk, hd);
    if (!workspace || workspace_bytes < need || ((uintptr_t)workspace & 255))
        return fail(MXP_E_BADARG, "workspace: need %zu bytes, 256-byte aligned", need);
    const OpsBytes ob = ops_bytes(B, H, Nq, Nk, hd);
    unsigned char* w = (unsigned char*)workspace;
    unsigned char* q_op = w; w += align256(ob.q);
    unsigned char* k_op = w; w += align256(ob.k);
    unsigned char* v_op = w;
    if ((rc = launch_codes_to_ops(q_codes, q_exps, q_op, B * H, Nq, Nk, hd, 0, st))) return rc;
    if ((rc = launch_codes_to_ops(k_codes, k_exps, k_op, B * H, Nq, Nk, hd, 1, st))) return rc;
    if ((rc = launch_prep_v(View{v, v_sB, v_sH, v_sN}, B, H, Nq, Nk, hd, bfloat_bits == 16, flush != 0, v_op, st,
                            v_dtype))) return rc;
    AttnParams p{};
    p.q_op = q_op; p.k_op = k_op; p.v_op = v_op; p.mask = mask;
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.hd = hd;
    p.scale = scale; p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
    p.out = out; p.o_sB = o_sB; p.o_sH = o_sH; p.o_sN = o_sN; p.out_dt = out_dtype;
    return launch_attend(p, st);
}

int mxp_sparse_attention(const int8_t* q_codes, const int8_t* q_exps, const int8_t* k_codes,
                         const int8_t* k_exps, const float* v, int64_t v_sB, int64_t v_sH,
                         int64_t v_sN, const uint32_t* mask, int B, int H, int Nq, int Nk, int hd,
                         float scale, int bfloat_bits, int flush, float* out, int64_t o_sB,
                         int64_t o_sH, int64_t o_sN, void* workspace, size_t workspace_bytes, void* stream) {
    return mxp_sparse_attention_dt(q_codes, q_exps, k_codes, k_exps, v, v_sB, v_sH, v_sN, MXP_DT_F32, mask, B, H, Nq, Nk,
                                   hd, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, MXP_DT_F32, workspace,
                                   workspace_bytes, stream);
}

size_t mxp_pruned_attention_workspace_bytes(int B, int H, int Nq, int Nk, int hd) {
    const size_t bh = (size_t)B * H, nb = (size_t)(hd + 31) / 32, nw = (size_t)(Nk + 31) / 32;
    const OpsBytes ob = ops_bytes(B, H, Nq, Nk, hd);
    const size_t ops = align256(ob.q) + align256(ob.k) + align256(ob.v);
    const size_t codes = align256(bh * Nq * hd) + align256(bh * Nq * nb) + align256(bh * Nk * hd) + align256(bh * Nk * nb);
    size_t base = (ops > codes ? ops : codes) + align256(bh * Nq * nw * 4);
    const size_t fused = align256(fused_workspace_bytes(Nq, Nk, hd));      // operand slots of the fused kernel
    if (base < fused) base = fused;
    return base + long_ws_layout(B, H, Nq, Nk, hd).total;
}

static int pruned_attention_impl(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                                 const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                                 const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                                 int B, int H, int Nq, int Nk, int hd, int top_k, float scale,
                                 int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                                 int64_t o_sN, const float* key_bias, int64_t kb_sB, uint32_t* mask_out,
                                 void* workspace, size_t workspace_bytes, void* stream, int pred_mode = 0,
                                 const float* elsa_proj = nullptr, float elsa_cap = 0.f, int dt = DT_F32,
                                 int out_dt = DT_F32) {
    g_launches = 0;
    if (check_dtype("q/k/v", dt) || check_dtype("out", out_dt)) return MXP_E_BADARG;
    if (out_dt != DT_F32 && out_dt != dt)
        return fail(MXP_E_BADARG, "out: element type %d must be fp32 or the inputs' (%d)", out_dt, dt);
    if (dt != DT_F32 && pred_mode != 0)
        return fail(MXP_E_UNSUPPORTED, "pred_mode %d: 16-bit inputs are implemented for the exponent-sign predictor only",
                    pred_mode);
    if (pred_mode != 0 && g_attn_path != 0)
        return fail(MXP_E_UNSUPPORTED, "pred_mode %d needs the tcgen05 attention path", pred_mode);
    if (key_bias && (g_attn_path != 0 || ((uintptr_t)key_bias & 3)))
        return fail(MXP_E_UNSUPPORTED, "key_bias needs the tcgen05 attention path and a 4-byte aligned pointer");
    int rc = check_shape(B, H, Nq, Nk, hd, bfloat_bits);
    if (rc || (rc = check_keys(Nk))) return rc;
    if ((rc = check_half_scope(dt, hd))) return rc;
    if ((rc = check_view("q", q, q_sB, q_sH, q_sN, hd, dt))) return rc;
    if ((rc = check_view("k", k, k_sB, k_sH, k_sN, hd, dt))) return rc;
    if ((rc = check_view("v", v, v_sB, v_sH, v_sN, hd, dt))) return rc;
    if ((rc = check_view("out", out, o_sB, o_sH, o_sN, hd, out_dt))) return rc;
    if (top_k < 1 || top_k > Nk) return fail(MXP_E_BADARG, "top_k=%d outside [1, Nk=%d]", top_k, Nk);
    const size_t need = mxp_pruned_attention_workspace_bytes(B, H, Nq, Nk, hd);
    if (!workspace || workspace_bytes < need || ((uintptr_t)workspace & 255))
        return fail(MXP_E_BADARG, "workspace: need %zu bytes, 256-byte aligned", need);
    const bool tc = g_attn_path == 0;
    if (tc && (hd & 7)) return fail(MXP_E_UNSUPPORTED, "head_dim %d: the tensor-core attention path needs a multiple of 8", hd);
    const size_t bh = (size_t)B * H, nb = (size_t)(hd + 31) / 32, nw = (size_t)(Nk + 31) / 32;
    const OpsBytes ob = ops_bytes(B, H, Nq, Nk, hd);
    unsigned char* w = (unsigned char*)workspace;
    const size_t long_bytes = long_ws_layout(B, H, Nq, Nk, hd).total;
    uint32_t* mask = mask_out ? mask_out : (uint32_t*)(w + need - long_bytes - align256(bh * Nq * nw * 4));
    cudaStream_t st = (cudaStream_t)stream;

    PredParams pp{};
    pp.q = View{q, q_sB, q_sH, q_sN};
    pp.k = View{k, k_sB, k_sH, k_sN};
    pp.dt = dt;
    pp.B = B; pp.H = H; pp.Nq = Nq; pp.Nk = Nk; pp.hd = hd; pp.top_k = top_k;
    pp.bf16 = bfloat_bits == 16; pp.flush = flush != 0;
    pp.mask = mask; pp.idx = nullptr;
    pp.key_bias = key_bias; pp.kb_sB = kb_sB;
    pp.pred_mode = pred_mode; pp.score_scale = scale;
    pp.elsa_proj = elsa_proj; pp.elsa_cap = elsa_cap;
    pp.long_ws = long_bytes ? w + need - long_bytes : nullptr;
    pp.long_ws_bytes = long_bytes;
    if (tc && pred_mode == 0 && !key_bias) {
        // one persistent launch for the whole path (mxprune_fused.cuh) where it applies
        FusedArgs fa{};
        fa.q = pp.q; fa.k = pp.k; fa.v = View{v, v_sB, v_sH, v_sN};
        fa.dt = dt; fa.out_dt = out_dt;
        fa.B = B; fa.H = H; fa.Nq = Nq; fa.Nk = Nk; fa.hd = hd; fa.top_k = top_k;
        fa.bf16 = bfloat_bits == 16; fa.flush = flush != 0; fa.scale = scale;
        fa.out = out; fa.o_sB = o_sB; fa.o_sH = o_sH; fa.o_sN = o_sN;
        fa.mask_out = mask_out;
        fa.slots = w; fa.slots_bytes = need - long_bytes;
        prof_mark(0, st);
        if (fused_try(fa, st, &rc) == 0) {
            prof_mark(1, st); prof_mark(2, st); prof_mark(3, st);
            return rc;
        }
        rc = MXP_OK;
    }
    if (tc) {
        unsigned char* q_op = w; w += align256(ob.q);
        unsigned char* k_op = w; w += align256(ob.k);
        unsigned char* v_op = w;
        pp.q_op = q_op; pp.k_op = k_op;
        prof_mark(0, st);
        if ((rc = predict_topk_impl(pp, st))) return rc;
        prof_mark(1, st);
        if ((rc = launch_prep_v(View{v, v_sB, v_sH, v_sN}, B, H, Nq, Nk, hd, bfloat_bits == 16, flush != 0, v_op, st, dt)))
            return rc;
        prof_mark(2, st);
        AttnParams ap{};
        ap.q_op = q_op; ap.k_op = k_op; ap.v_op = v_op; ap.mask = mask;
        ap.B = B; ap.H = H; ap.Nq = Nq; ap.Nk = Nk; ap.hd = hd;
        ap.scale = scale; ap.bf16 = bfloat_bits == 16; ap.flush = flush != 0;
        ap.out = out; ap.o_sB = o_sB; ap.o_sH = o_sH; ap.o_sN = o_sN; ap.out_dt = out_dt;
        ap.key_bias = key_bias; ap.kb_sB = kb_sB;
        int rc2 = MXP_OK;
        if (attend_sparse_try(ap, top_k, st, &rc2) == 0) rc = rc2;      // cost follows top_k (small top_k / Nk)
        else rc = launch_attend(ap, st);
        prof_mark(3, st);
        return rc;
    }
    int8_t* qc = (int8_t*)w; w += align256(bh * Nq * hd);
    int8_t* qe = (int8_t*)w; w += align256(bh * Nq * nb);
    int8_t* kc = (int8_t*)w; w += align256(bh * Nk * hd);
    int8_t* ke = (int8_t*)w;
    pp.q_codes = qc; pp.q_exps = qe; pp.k_codes = kc; pp.k_exps = ke;
    if ((rc = predict_topk_impl(pp, st))) return rc;
    AttnCoreParams ap{};
    ap.q_codes = qc; ap.q_exps = qe; ap.k_codes = kc; ap.k_exps = ke;
    ap.v = View{v, v_sB, v_sH, v_sN};
    ap.mask = mask;
    ap.B = B; ap.H = H; ap.Nq = Nq; ap.Nk = Nk; ap.hd = hd;
    ap.scale = scale; ap.bf16 = bfloat_bits == 16; ap.flush = flush != 0;
    ap.out = out; ap.o_sB = o_sB; ap.o_sH = o_sH; ap.o_sN = o_sN;
    return attend_core_impl(ap, st);
}

int mxp_pruned_attention_dt(const void* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                            const void* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                            const void* v, int64_t v_sB, int64_t v_sH, int64_t v_sN, int in_dtype,
                            int B, int H, int Nq, int Nk, int hd, int top_k, float scale,
                            int bfloat_bits, int flush, void* out, int64_t o_sB, int64_t o_sH,
                            int64_t o_sN, int out_dtype, const float* key_bias, int64_t kb_sB, uint32_t* mask_out,
                            void* workspace, size_t workspace_bytes, void* stream) {
    return pruned_attention_impl((const float*)q, q_sB, q_sH, q_sN, (const float*)k, k_sB, k_sH, k_sN,
                                 (const float*)v, v_sB, v_sH, v_sN, B, H, Nq, Nk, hd, top_k, scale, bfloat_bits, flush,
                                 (float*)out, o_sB, o_sH, o_sN, key_bias, kb_sB, mask_out, workspace, workspace_bytes,
                                 stream, 0, nullptr, 0.f, in_dtype, out_dtype);
}

int mxp_pruned_attention(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                         const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                         const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                         int B, int H, int Nq, int Nk, int hd, int top_k, float scale,
                         int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                         int64_t o_sN, uint32_t* mask_out, void* workspace, size_t workspace_bytes,
                         void* stream) {
    return mxp_pruned_attention_dt(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, v, v_sB, v_sH, v_sN, MXP_DT_F32, B, H, Nq,
                                   Nk, hd, top_k, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, MXP_DT_F32, nullptr, 0,
                                   mask_out, workspace, workspace_bytes, stream);
}

int mxp_pruned_attention_biased(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                                const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                                const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                                int B, int H, int Nq, int Nk, int hd, int top_k, float scale,
                                int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                                int64_t o_sN, const float* key_bias, int64_t kb_sB, uint32_t* mask_out,
                                void* workspace, size_t workspace_bytes, void* stream) {
    if (!key_bias) return fail(MXP_E_BADARG, "key_bias: null pointer (use mxp_pruned_attention)");
    return mxp_pruned_attention_dt(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, v, v_sB, v_sH, v_sN, MXP_DT_F32, B, H, Nq,
                                   Nk, hd, top_k, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, MXP_DT_F32, key_bias,
                                   kb_sB, mask_out, workspace, workspace_bytes, stream);
}

int mxp_pruned_attention_mode(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                              const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                              const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                              int B, int H, int Nq, int Nk, int hd, int top_k, int pred_mode, float scale,
                              int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                              int64_t o_sN, const float* key_bias, int64_t kb_sB, uint32_t* mask_out,
                              void* workspace, size_t workspace_bytes, void* stream) {
    if (pred_mode < MXP_PRED_EXP_SIGN || pred_mode > MXP_PRED_TRUE_EX)
        return fail(MXP_E_BADARG, "pred_mode=%d outside [0, 6]", pred_mode);
    return pruned_attention_impl(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, v, v_sB, v_sH, v_sN, B, H, Nq, Nk, hd,
                                 top_k, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, key_bias, kb_sB, mask_out,
                                 workspace, workspace_bytes, stream, pred_mode);
}

int mxp_predict_topk_mode(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                          const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                          int B, int H, int Nq, int Nk, int hd, int top_k, int pred_mode, float scale,
                          int bfloat_bits, int flush, const float* key_bias, int64_t kb_sB,
                          uint32_t* mask, int32_t* idx, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, Nq, Nk, hd, bfloat_bits);
    if (rc || (rc = check_keys(Nk))) return rc;
    if ((rc = check_view("q", q, q_sB, q_sH, q_sN, hd))) return rc;
    if ((rc = check_view("k", k, k_sB, k_sH, k_sN, hd))) return rc;
    if (!mask) return fail(MXP_E_BADARG, "mask: null pointer");
    if (top_k < 1 || top_k > Nk) return fail(MXP_E_BADARG, "top_k=%d outside [1, Nk=%d]", top_k, Nk);
    if (pred_mode < MXP_PRED_EXP_SIGN || pred_mode > MXP_PRED_TRUE_EX)
        return fail(MXP_E_BADARG, "pred_mode=%d outside [0, 6]", pred_mode);
    PredParams p{};
    p.q = View{q, q_sB, q_sH, q_sN};
    p.k = View{k, k_sB, k_sH, k_sN};
    p.B = B; p.H = H; p.Nq = Nq; p.Nk = Nk; p.hd = hd; p.top_k = top_k;
    p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
    p.mask = mask; p.idx = idx;
    p.pred_mode = pred_mode; p.score_scale = scale;
    p.key_bias = key_bias; p.kb_sB = kb_sB;
    p.long_ws = workspace; p.long_ws_bytes = workspace_bytes;
    return predict_topk_impl(p, (cudaStream_t)stream);
}

int mxp_pruned_attention_elsa(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                              const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                              const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                              int B, int H, int N, int hd, int top_k, const float* proj, float rank_cap,
                              float scale, int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                              int64_t o_sN, uint32_t* mask_out, void* workspace, size_t workspace_bytes,
                              void* stream) {
    return pruned_attention_impl(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, v, v_sB, v_sH, v_sN, B, H, N, N, hd,
                                 top_k, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, nullptr, 0, mask_out,
                                 workspace, workspace_bytes, stream, PRED_ELSA, proj, rank_cap);
}

int mxp_predict_topk_elsa(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                          const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                          int B, int H, int N, int hd, int top_k, const float* proj, float rank_cap,
                          int bfloat_bits, int flush, uint32_t* mask, int32_t* idx, void* stream) {
    g_launches = 0;
    int rc = check_shape(B, H, N, N, hd, bfloat_bits);
    if (rc || (rc = check_keys(N))) return rc;
    if ((rc = check_view("q", q, q_sB, q_sH, q_sN, hd))) return rc;
    if ((rc = check_view("k", k, k_sB, k_sH, k_sN, hd))) return rc;
    if (!mask) return fail(MXP_E_BADARG, "mask: null pointer");
    if (top_k < 1 || top_k > N) return fail(MXP_E_BADARG, "top_k=%d outside [1, N=%d]", top_k, N);
    PredParams p{};
    p.q = View{q, q_sB, q_sH, q_sN};
    p.k = View{k, k_sB, k_sH, k_sN};
    p.B = B; p.H = H; p.Nq = N; p.Nk = N; p.hd = hd; p.top_k = top_k;
    p.bf16 = bfloat_bits == 16; p.flush = flush != 0;
    p.mask = mask; p.idx = idx;
    p.pred_mode = PRED_ELSA; p.elsa_proj = proj; p.elsa_cap = rank_cap;
    return predict_topk_impl(p, (cudaStream_t)stream);
}

// ---- MX Linear (SURVEY 8 f2) ---------------------------------------------------------------------
static int check_linear(int M, int N, int K, int bfloat_bits) {
    if (M <= 0 || N <= 0 || K <= 0) return fail(MXP_E_BADARG, "empty shape M=%d N=%d K=%d", M, N, K);
    if (K % GL_BK) return fail(MXP_E_UNSUPPORTED, "in_features %d: need a multiple of %d", K, GL_BK);
    if (N & 3) return fail(MXP_E_UNSUPPORTED, "out_features %d: need a multiple of 4", N);
    if (bfloat_bits != 16 && bfloat_bits != 32) return fail(MXP_E_UNSUPPORTED, "bfloat=%d: only 16 or 32 are on the path", bfloat_bits);
    return MXP_OK;
}
// mod: the adaLN modulation of x (ModParams), or null; norm_kind / norm: the LayerNorm of x (LN_PLAIN / LN_AFFINE,
// with the row statistics k_layer_norm wrote to norm->mean / rstd), or LN_NONE
static int launch_quantize_gemm_operand(const void* x, int dt, int64_t ld, int rows, int K, int rows_tile, int bf16,
                                        int flush, void* op, cudaStream_t st, const ModParams* mod = nullptr,
                                        int norm_kind = LN_NONE, const NormParams* norm = nullptr) {
    const int rows_pad = (rows + rows_tile - 1) / rows_tile * rows_tile;
    const int64_t ntask = (int64_t)rows_pad * (K / 32);
    int64_t blocks = (ntask + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    const NormParams np = norm ? *norm : NormParams{};
#define MXP_QG2(DT_, MOD_, NORM_) k_quantize_gemm_operand<DT_, MOD_, NORM_><<<(unsigned)blocks, 256, 0, st>>>( \
        (const float*)x, ld, rows, rows_pad, K, rows_tile, bf16, flush, (unsigned char*)op, mod ? *mod : ModParams{}, np)
#define MXP_QG1(DT_, NORM_) (mod ? MXP_QG2(DT_, true, NORM_) : MXP_QG2(DT_, false, NORM_))
#define MXP_QG(DT_) (norm_kind == LN_AFFINE ? MXP_QG1(DT_, LN_AFFINE) \
                     : norm_kind == LN_PLAIN ? MXP_QG1(DT_, LN_PLAIN) : MXP_QG1(DT_, LN_NONE))
    if (dt == DT_BF16) MXP_QG(DT_BF16);
    else if (dt == DT_F16) MXP_QG(DT_F16);
    else MXP_QG(DT_F32);
#undef MXP_QG
#undef MXP_QG1
#undef MXP_QG2
    return check_launch("k_quantize_gemm_operand");
}

// k_layer_norm<dt, norm_kind>: one warp per row; y (the normalized rows) may be null (statistics only)
static int launch_layer_norm(const void* x, int dt, int64_t ld, int rows, int K, float eps, int norm_kind,
                             const void* w, const void* b, float* mean, float* rstd, void* y, cudaStream_t st) {
    const unsigned grid = (unsigned)((rows + LN_ROWS - 1) / LN_ROWS);
    const float *xp = (const float*)x, *wp = (const float*)w, *bp = (const float*)b;
#define MXP_LN(DT_) (norm_kind == LN_AFFINE ? k_layer_norm<DT_, LN_AFFINE><<<grid, LN_ROWS * 32, 0, st>>>( \
                         xp, ld, rows, K, eps, wp, bp, mean, rstd, (float*)y) \
                     : k_layer_norm<DT_, LN_PLAIN><<<grid, LN_ROWS * 32, 0, st>>>(xp, ld, rows, K, eps, wp, bp, mean, \
                                                                                  rstd, (float*)y))
    if (dt == DT_BF16) MXP_LN(DT_BF16);
    else if (dt == DT_F16) MXP_LN(DT_F16);
    else MXP_LN(DT_F32);
#undef MXP_LN
    return check_launch("k_layer_norm");
}

// rows of a GEMM input (x or W): a 16-byte aligned base, a row stride >= K whose rows stay 16-byte aligned
// (a multiple of 4 fp32 or 8 16-bit elements)
static int check_linear_rows(const char* name, const void* p, int dt, int64_t ld, int K) {
    const int64_t m = dt == DT_F32 ? 3 : 7;
    if (!p || ((uintptr_t)p & 15) || (ld & m) || ld < K)
        return fail(MXP_E_BADARG, "%s: null or misaligned pointer, or row stride %lld not >= %d and a multiple of %d elements",
                    name, (long long)ld, K, (int)m + 1);
    return MXP_OK;
}

// bias of element type dt -> A1(bias), N floats
static int launch_round_bias(const void* bias, int dt, float* rbias, int N, int bf16, cudaStream_t st) {
    const float* b = (const float*)bias;
    const unsigned nblk = (unsigned)((N + 255) / 256);
    if (dt == DT_BF16) k_round_bias<DT_BF16><<<nblk, 256, 0, st>>>(b, rbias, N, bf16);
    else if (dt == DT_F16) k_round_bias<DT_F16><<<nblk, 256, 0, st>>>(b, rbias, N, bf16);
    else k_round_bias<DT_F32><<<nblk, 256, 0, st>>>(b, rbias, N, bf16);
    return check_launch("k_round_bias");
}

// k_mx_linear_umma<out_dt, EPI>: persistent, one CTA per SM (4 stages of 48 KiB, 512 TMEM columns for the
// double-buffered accumulator); the same grid and shared memory for every output type and epilogue
extern "C++" {
template <int EPI>
static int launch_linear_gemm(const LinearParams& lp, int out_dt, cudaStream_t st) {
    const GemmOpLayout L = gemm_op_layout(lp.K);
    const size_t dyn = lp.stages * (L.a_stage + L.b_stage) + 2048 + 4 * 32 * 36 * 4 + 1024;
    const int ntiles = ((lp.M + GL_BM - 1) / GL_BM) * ((lp.N + GL_BN - 1) / GL_BN);
    const int sms = sm_count();
    const unsigned grid = (unsigned)(ntiles < sms ? ntiles : sms);
    if (out_dt == DT_BF16) {
        MXP_ENSURE_DYN_SMEM((k_mx_linear_umma<DT_BF16, EPI>), 227 * 1024);
        k_mx_linear_umma<DT_BF16, EPI><<<grid, GL_T, dyn, st>>>(lp);
    } else if (out_dt == DT_F16) {
        MXP_ENSURE_DYN_SMEM((k_mx_linear_umma<DT_F16, EPI>), 227 * 1024);
        k_mx_linear_umma<DT_F16, EPI><<<grid, GL_T, dyn, st>>>(lp);
    } else {
        MXP_ENSURE_DYN_SMEM((k_mx_linear_umma<DT_F32, EPI>), 227 * 1024);
        k_mx_linear_umma<DT_F32, EPI><<<grid, GL_T, dyn, st>>>(lp);
    }
    return check_launch("k_mx_linear_umma");
}
}  // extern "C++"

size_t mxp_mx_linear_weight_bytes(int N, int K) {
    return (size_t)((N + GL_BN - 1) / GL_BN) * GL_BN * (size_t)K * 2;
}
size_t mxp_mx_linear_workspace_bytes(int M, int N, int K) {
    return align256((size_t)((M + GL_BM - 1) / GL_BM) * GL_BM * (size_t)K * 2) + align256((size_t)N * 4);
}

int mxp_mx_linear_prepare_weight_dt(const void* w, int w_dtype, int64_t ldw, int N, int K, int bfloat_bits, int flush,
                                    void* w_op, void* stream) {
    g_launches = 0;
    int rc = check_linear(1, N, K, bfloat_bits);
    if (rc) return rc;
    if ((rc = check_dtype("weight", w_dtype))) return rc;
    if ((rc = check_linear_rows("weight", w, w_dtype, ldw, K))) return rc;
    if (!w_op || ((uintptr_t)w_op & 15)) return fail(MXP_E_BADARG, "w_op: null or misaligned pointer");
    return launch_quantize_gemm_operand(w, w_dtype, ldw, N, K, GL_BN, bfloat_bits == 16, flush != 0, w_op,
                                        (cudaStream_t)stream);
}

int mxp_mx_linear_prepare_weight(const float* w, int64_t ldw, int N, int K, int bfloat_bits, int flush, void* w_op,
                                 void* stream) {
    return mxp_mx_linear_prepare_weight_dt(w, MXP_DT_F32, ldw, N, K, bfloat_bits, flush, w_op, stream);
}

// ---- additions of the adaLN and the _ex entry points: the LayerNorm of x (K wide), the modulation of x (mod, K wide)
// and the residual (gated, or with plain_add a plain add) of the output (N wide), each optional
struct Adaln {
    int tokens;
    const void *shift, *scale, *residual, *gate;
    int64_t ld_shift, ld_scale, ld_residual, ld_gate;
    bool plain_add;                   // a residual without a gate is a plain add (the _ex entry points)
    int layer_norm;                   // 0 or 1
    const void *ln_weight, *ln_bias;
    float ln_eps;
    int norm_kind() const { return !layer_norm ? LN_NONE : ln_weight ? LN_AFFINE : LN_PLAIN; }
};

// an (M / tokens, N) gate or (M, N) residual of x's type: the alignment and row-stride rules of out
static int check_out_like(const char* name, const void* p, int dt, int64_t ld, int N) {
    const uintptr_t align = dt == DT_F32 ? 15 : 7;
    if (!p || ((uintptr_t)p & align) || (ld & 3) || ld < N)
        return fail(MXP_E_BADARG, "%s: null or misaligned pointer, or row stride %lld not >= %d and a multiple of 4",
                    name, (long long)ld, N);
    return MXP_OK;
}

static int check_adaln(const Adaln& a, int dt, int M, int K, int N) {
    if (a.tokens <= 0 || M % a.tokens)
        return fail(MXP_E_BADARG, "tokens %d: need a positive divisor of the row count M=%d", a.tokens, M);
    if (!a.shift != !a.scale) return fail(MXP_E_BADARG, "shift and scale: give both or neither");
    if (a.gate && !a.residual) return fail(MXP_E_BADARG, "gate without residual");
    if (a.residual && !a.gate && !a.plain_add) return fail(MXP_E_BADARG, "residual and gate: give both or neither");
    if (a.layer_norm != 0 && a.layer_norm != 1) return fail(MXP_E_BADARG, "layer_norm %d: 0 or 1", a.layer_norm);
    if (!a.ln_weight != !a.ln_bias) return fail(MXP_E_BADARG, "ln_weight and ln_bias: give both or neither");
    if (a.ln_weight && !a.layer_norm) return fail(MXP_E_BADARG, "ln_weight / ln_bias without layer_norm");
    // the norm's weight and bias are read 4 elements (16 or 8 bytes) at a time
    const uintptr_t ln_align = dt == DT_F32 ? 15 : 7;
    if (a.ln_weight && (((uintptr_t)a.ln_weight & ln_align) || ((uintptr_t)a.ln_bias & ln_align)))
        return fail(MXP_E_BADARG, "ln_weight / ln_bias: misaligned pointer");
    if (a.layer_norm && !(a.ln_eps >= 0.f)) return fail(MXP_E_BADARG, "ln_eps: need a number >= 0");
    int rc = MXP_OK;
    // shift / scale are read in 32-element blocks, 16 bytes at a time: the rules of x
    if (a.shift && ((rc = check_linear_rows("shift", a.shift, dt, a.ld_shift, K)) ||
                    (rc = check_linear_rows("scale", a.scale, dt, a.ld_scale, K))))
        return rc;
    if (a.residual && (rc = check_out_like("residual", a.residual, dt, a.ld_residual, N))) return rc;
    if (a.gate && (rc = check_out_like("gate", a.gate, dt, a.ld_gate, N))) return rc;
    return MXP_OK;
}

static ModParams make_mod(const Adaln& a) {
    return ModParams{(const float*)a.shift, (const float*)a.scale, a.ld_shift, a.ld_scale, a.tokens};
}
// the store of the GEMM's output: plain, or with the residual (gated or plain add)
static int launch_output_gemm(LinearParams& lp, const Adaln* a, int out_dt, cudaStream_t st) {
    if (!a || !a->residual) return launch_linear_gemm<EPI_STORE>(lp, out_dt, st);
    lp.residual = (const float*)a->residual; lp.ldr = a->ld_residual;
    if (!a->gate) return launch_linear_gemm<EPI_RESIDUAL>(lp, out_dt, st);
    lp.gate = (const float*)a->gate; lp.ldg = a->ld_gate; lp.tokens = a->tokens;
    return launch_linear_gemm<EPI_GATED_RESIDUAL>(lp, out_dt, st);
}

// x's operand: the per-row LayerNorm statistics into `stats` (when the norm is on), then the quantizer
static int launch_activation_operand(const void* x, int dt, int64_t ldx, int M, int K, int bf16, int flush,
                                     unsigned char* a_op, float* stats, const Adaln* ad, cudaStream_t st) {
    ModParams mod{};
    if (ad && ad->shift) mod = make_mod(*ad);
    const int nk = ad ? ad->norm_kind() : LN_NONE;
    float *mean = stats, *rstd = stats + align256((size_t)M * 4) / 4;
    const NormParams np{mean, rstd, (const float*)(ad ? ad->ln_weight : nullptr), (const float*)(ad ? ad->ln_bias : nullptr)};
    int rc;
    if (nk != LN_NONE && (rc = launch_layer_norm(x, dt, ldx, M, K, ad->ln_eps, nk, np.w, np.b, mean, rstd, nullptr, st)))
        return rc;
    return launch_quantize_gemm_operand(x, dt, ldx, M, K, GL_BM, bf16, flush, a_op, st, ad && ad->shift ? &mod : nullptr,
                                        nk, &np);
}

// the per-row mean and rstd (fp32 each) of the _ex entry points: after the plain call's workspace
static size_t ln_stats_bytes(int M) { return 2 * align256((size_t)M * 4); }

static int mx_linear_impl(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                          const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                          const Adaln* ad, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    int rc = check_linear(M, N, K, bfloat_bits);
    if (rc) return rc;
    if ((rc = check_dtype("x", x_dtype)) || (rc = check_dtype("bias", bias_dtype))) return rc;
    if ((rc = check_linear_rows("x", x, x_dtype, ldx, K))) return rc;
    // out has x's element type; its rows take 16-byte (fp32) or 8-byte (16-bit) stores of four elements
    const uintptr_t out_align = x_dtype == DT_F32 ? 15 : 7;
    if (!w_op || !out || ((uintptr_t)w_op & 15) || ((uintptr_t)out & out_align) || (ldo & 3) || ldo < N)
        return fail(MXP_E_BADARG, "w_op / out: null or misaligned pointer, or out row stride %lld not >= %d and a multiple "
                    "of 4", (long long)ldo, N);
    if (ad && (rc = check_adaln(*ad, x_dtype, M, K, N))) return rc;
    const size_t plain = mxp_mx_linear_workspace_bytes(M, N, K);
    const size_t need = plain + (ad && ad->layer_norm ? ln_stats_bytes(M) : 0);
    if (!workspace || workspace_bytes < need || ((uintptr_t)workspace & 255))
        return fail(MXP_E_BADARG, "workspace: need %zu bytes, 256-byte aligned", need);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* a_op = (unsigned char*)workspace;
    float* rbias = (float*)(a_op + align256((size_t)((M + GL_BM - 1) / GL_BM) * GL_BM * (size_t)K * 2));
    float* stats = (float*)((unsigned char*)workspace + plain);
    if ((rc = launch_activation_operand(x, x_dtype, ldx, M, K, bfloat_bits == 16, flush != 0, a_op, stats, ad, st)))
        return rc;
    if (bias && (rc = launch_round_bias(bias, bias_dtype, rbias, N, bfloat_bits == 16, st))) return rc;
    LinearParams lp{};
    lp.a_op = a_op; lp.w_op = (const unsigned char*)w_op; lp.bias = bias ? rbias : nullptr;
    lp.out = (float*)out; lp.ldo = ldo; lp.M = M; lp.N = N; lp.K = K; lp.bf16 = bfloat_bits == 16; lp.stages = 4;
    return launch_output_gemm(lp, ad, x_dtype, st);
}

int mxp_mx_linear_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N, const void* bias,
                     int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo, void* workspace,
                     size_t workspace_bytes, void* stream) {
    return mx_linear_impl(x, x_dtype, ldx, M, K, w_op, N, bias, bias_dtype, bfloat_bits, flush, out, ldo, nullptr,
                          workspace, workspace_bytes, stream);
}

int mxp_mx_linear_adaln_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                           const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                           int tokens, const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale,
                           const void* residual, int64_t ld_residual, const void* gate, int64_t ld_gate,
                           void* workspace, size_t workspace_bytes, void* stream) {
    const Adaln ad{tokens, shift, scale, residual, gate, ld_shift, ld_scale, ld_residual, ld_gate, false, 0, nullptr,
                   nullptr, 0.f};
    return mx_linear_impl(x, x_dtype, ldx, M, K, w_op, N, bias, bias_dtype, bfloat_bits, flush, out, ldo, &ad,
                          workspace, workspace_bytes, stream);
}

// ---- fused MX MLP: mx_linear(act(mx_linear(x, W1, b1)), W2, b2) with fc1's epilogue writing fc2's operand --------
// workspace: x's operand | the hidden operand (fc2's A, K = N1) | A1(b1) | A1(b2)
size_t mxp_mx_mlp_workspace_bytes(int M, int K, int N1, int N2) {
    const size_t rows = (size_t)((M + GL_BM - 1) / GL_BM) * GL_BM;
    return align256(rows * (size_t)K * 2) + align256(rows * (size_t)N1 * 2) + align256((size_t)N1 * 4) +
           align256((size_t)N2 * 4);
}

static int mx_mlp_impl(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1, const void* b1,
                       int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype, int bfloat_bits,
                       int flush, void* out, int64_t ldo, const Adaln* ad, void* workspace, size_t workspace_bytes,
                       void* stream) {
    g_launches = 0;
    int rc = check_linear(M, N1, K, bfloat_bits);
    if (rc || (rc = check_linear(M, N2, N1, bfloat_bits))) return rc;         // fc2: K = N1, a multiple of 64
    if (act != MXP_ACT_GELU && act != MXP_ACT_GELU_TANH)
        return fail(MXP_E_BADARG, "act %d: MXP_ACT_GELU (0) or MXP_ACT_GELU_TANH (1)", act);
    if ((rc = check_dtype("x", x_dtype)) || (rc = check_dtype("b1", b1_dtype)) || (rc = check_dtype("b2", b2_dtype)))
        return rc;
    if ((rc = check_linear_rows("x", x, x_dtype, ldx, K))) return rc;
    const uintptr_t out_align = x_dtype == DT_F32 ? 15 : 7;
    if (!w1_op || !w2_op || !out || ((uintptr_t)w1_op & 15) || ((uintptr_t)w2_op & 15) || ((uintptr_t)out & out_align) ||
        (ldo & 3) || ldo < N2)
        return fail(MXP_E_BADARG, "w1_op / w2_op / out: null or misaligned pointer, or out row stride %lld not >= %d and "
                    "a multiple of 4", (long long)ldo, N2);
    if (ad && (rc = check_adaln(*ad, x_dtype, M, K, N2))) return rc;
    const size_t plain = mxp_mx_mlp_workspace_bytes(M, K, N1, N2);
    const size_t need = plain + (ad && ad->layer_norm ? ln_stats_bytes(M) : 0);
    if (!workspace || workspace_bytes < need || ((uintptr_t)workspace & 255))
        return fail(MXP_E_BADARG, "workspace: need %zu bytes, 256-byte aligned", need);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t rows = (size_t)((M + GL_BM - 1) / GL_BM) * GL_BM;
    unsigned char* a_op = (unsigned char*)workspace;
    unsigned char* h_op = a_op + align256(rows * (size_t)K * 2);
    float* rb1 = (float*)(h_op + align256(rows * (size_t)N1 * 2));
    float* rb2 = (float*)((unsigned char*)rb1 + align256((size_t)N1 * 4));
    const int bf16 = bfloat_bits == 16;
    float* stats = (float*)((unsigned char*)workspace + plain);
    if ((rc = launch_activation_operand(x, x_dtype, ldx, M, K, bf16, flush != 0, a_op, stats, ad, st))) return rc;
    if (b1 && (rc = launch_round_bias(b1, b1_dtype, rb1, N1, bf16, st))) return rc;
    if (b2 && (rc = launch_round_bias(b2, b2_dtype, rb2, N2, bf16, st))) return rc;
    LinearParams l1{};
    l1.a_op = a_op; l1.w_op = (const unsigned char*)w1_op; l1.bias = b1 ? rb1 : nullptr;
    l1.M = M; l1.N = N1; l1.K = K; l1.bf16 = bf16; l1.stages = 4; l1.flush = flush != 0; l1.h_op = h_op;
    rc = act == MXP_ACT_GELU_TANH ? launch_linear_gemm<EPI_GELU_TANH>(l1, x_dtype, st)
                                  : launch_linear_gemm<EPI_GELU>(l1, x_dtype, st);
    if (rc) return rc;
    LinearParams l2{};
    l2.a_op = h_op; l2.w_op = (const unsigned char*)w2_op; l2.bias = b2 ? rb2 : nullptr;
    l2.out = (float*)out; l2.ldo = ldo; l2.M = M; l2.N = N2; l2.K = N1; l2.bf16 = bf16; l2.stages = 4;
    return launch_output_gemm(l2, ad, x_dtype, st);
}

int mxp_mx_mlp_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1, const void* b1,
                  int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype, int bfloat_bits,
                  int flush, void* out, int64_t ldo, void* workspace, size_t workspace_bytes, void* stream) {
    return mx_mlp_impl(x, x_dtype, ldx, M, K, w1_op, N1, b1, b1_dtype, act, w2_op, N2, b2, b2_dtype, bfloat_bits, flush,
                       out, ldo, nullptr, workspace, workspace_bytes, stream);
}

int mxp_mx_mlp_adaln_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1,
                        const void* b1, int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype,
                        int bfloat_bits, int flush, void* out, int64_t ldo, int tokens, const void* shift,
                        int64_t ld_shift, const void* scale, int64_t ld_scale, const void* residual,
                        int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                        size_t workspace_bytes, void* stream) {
    const Adaln ad{tokens, shift, scale, residual, gate, ld_shift, ld_scale, ld_residual, ld_gate, false, 0, nullptr,
                   nullptr, 0.f};
    return mx_mlp_impl(x, x_dtype, ldx, M, K, w1_op, N1, b1, b1_dtype, act, w2_op, N2, b2, b2_dtype, bfloat_bits, flush,
                       out, ldo, &ad, workspace, workspace_bytes, stream);
}

size_t mxp_mx_linear_ex_workspace_bytes(int M, int N, int K) {
    return mxp_mx_linear_workspace_bytes(M, N, K) + ln_stats_bytes(M);
}
size_t mxp_mx_mlp_ex_workspace_bytes(int M, int K, int N1, int N2) {
    return mxp_mx_mlp_workspace_bytes(M, K, N1, N2) + ln_stats_bytes(M);
}

int mxp_mx_linear_ex_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                        const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                        int layer_norm, const void* ln_weight, const void* ln_bias, float ln_eps, int tokens,
                        const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale, const void* residual,
                        int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                        size_t workspace_bytes, void* stream) {
    const Adaln ad{tokens, shift, scale, residual, gate, ld_shift, ld_scale, ld_residual, ld_gate, true, layer_norm,
                   ln_weight, ln_bias, ln_eps};
    return mx_linear_impl(x, x_dtype, ldx, M, K, w_op, N, bias, bias_dtype, bfloat_bits, flush, out, ldo, &ad,
                          workspace, workspace_bytes, stream);
}

int mxp_mx_mlp_ex_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1, const void* b1,
                     int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype, int bfloat_bits,
                     int flush, void* out, int64_t ldo, int layer_norm, const void* ln_weight, const void* ln_bias,
                     float ln_eps, int tokens, const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale,
                     const void* residual, int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                     size_t workspace_bytes, void* stream) {
    const Adaln ad{tokens, shift, scale, residual, gate, ld_shift, ld_scale, ld_residual, ld_gate, true, layer_norm,
                   ln_weight, ln_bias, ln_eps};
    return mx_mlp_impl(x, x_dtype, ldx, M, K, w1_op, N1, b1, b1_dtype, act, w2_op, N2, b2, b2_dtype, bfloat_bits, flush,
                       out, ldo, &ad, workspace, workspace_bytes, stream);
}

int mxp_layer_norm_dt(const void* x, int dtype, int64_t ldx, int M, int K, const void* weight, const void* bias,
                      float eps, void* y, float* mean, float* rstd, void* stream) {
    g_launches = 0;
    int rc = check_dtype("x", dtype);
    if (rc) return rc;
    if (M <= 0 || K <= 0 || (K & 3) || K > (1 << 24))
        return fail(MXP_E_UNSUPPORTED, "shape M=%d K=%d: need M > 0 and K a positive multiple of 4 up to 2^24", M, K);
    const uintptr_t al = dtype == DT_F32 ? 15 : 7;
    if (!x || ((uintptr_t)x & al) || (ldx & 3) || ldx < K || !y || ((uintptr_t)y & al))
        return fail(MXP_E_BADARG, "x / y: null or misaligned pointer, or x row stride %lld not >= %d and a multiple of 4",
                    (long long)ldx, K);
    if (!weight != !bias) return fail(MXP_E_BADARG, "weight and bias: give both or neither");
    if (weight && (((uintptr_t)weight & al) || ((uintptr_t)bias & al)))
        return fail(MXP_E_BADARG, "weight / bias: misaligned pointer");
    if (!(eps >= 0.f)) return fail(MXP_E_BADARG, "eps: need a number >= 0");
    if (!mean || !rstd) return fail(MXP_E_BADARG, "mean / rstd: null pointer");
    return launch_layer_norm(x, dtype, ldx, M, K, eps, weight ? LN_AFFINE : LN_PLAIN, weight, bias, mean, rstd, y,
                             (cudaStream_t)stream);
}

int mxp_activation_dt(const void* x, int dtype, int64_t n, int act, void* out, void* stream) {
    g_launches = 0;
    int rc = check_dtype("x", dtype);
    if (rc) return rc;
    if (act != MXP_ACT_GELU && act != MXP_ACT_GELU_TANH)
        return fail(MXP_E_BADARG, "act %d: MXP_ACT_GELU (0) or MXP_ACT_GELU_TANH (1)", act);
    if (n < 0 || (n > 0 && (!x || !out))) return fail(MXP_E_BADARG, "x / out: null pointer, or n = %lld < 0", (long long)n);
    if (n == 0) return MXP_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > (int64_t)sm_count() * 32) blocks = (int64_t)sm_count() * 32;
    cudaStream_t st = (cudaStream_t)stream;
    const float* xp = (const float*)x;
    float* o = (float*)out;
#define MXP_ACT(DT_) (act == MXP_ACT_GELU_TANH ? k_activation<DT_, EPI_GELU_TANH><<<(unsigned)blocks, 256, 0, st>>>(xp, n, o) \
                                               : k_activation<DT_, EPI_GELU><<<(unsigned)blocks, 256, 0, st>>>(xp, n, o))
    if (dtype == DT_BF16) MXP_ACT(DT_BF16);
    else if (dtype == DT_F16) MXP_ACT(DT_F16);
    else MXP_ACT(DT_F32);
#undef MXP_ACT
    return check_launch("k_activation");
}

int mxp_mx_linear(const float* x, int64_t ldx, int M, int K, const void* w_op, int N, const float* bias,
                  int bfloat_bits, int flush, float* out, int64_t ldo, void* workspace, size_t workspace_bytes,
                  void* stream) {
    return mxp_mx_linear_dt(x, MXP_DT_F32, ldx, M, K, w_op, N, bias, MXP_DT_F32, bfloat_bits, flush, out, ldo, workspace,
                            workspace_bytes, stream);
}

int mxp_pruned_attention_profile(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                                 const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                                 const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                                 int B, int H, int Nq, int Nk, int hd, int top_k, float scale,
                                 int bfloat_bits, int flush, float* out, int64_t o_sB, int64_t o_sH,
                                 int64_t o_sN, uint32_t* mask_out, void* workspace, size_t workspace_bytes,
                                 void* stream, float* kernel_ms) {
    if (!kernel_ms) return fail(MXP_E_BADARG, "kernel_ms: null pointer");
    if (g_attn_path != 0) return fail(MXP_E_UNSUPPORTED, "per-kernel profile is implemented for the tcgen05 path");
    g_profile = true;
    int rc = mxp_pruned_attention(q, q_sB, q_sH, q_sN, k, k_sB, k_sH, k_sN, v, v_sB, v_sH, v_sN, B, H, Nq, Nk, hd,
                                  top_k, scale, bfloat_bits, flush, out, o_sB, o_sH, o_sN, mask_out, workspace,
                                  workspace_bytes, stream);
    g_profile = false;
    if (rc) return rc;
    if (cudaEventSynchronize(g_ev[3]) != cudaSuccess) return fail(MXP_E_CUDA, "cudaEventSynchronize failed");
    for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&kernel_ms[i], g_ev[i], g_ev[i + 1]);
    return MXP_OK;
}

}  // extern "C"
