// K1: fused MX quantizer + exponent-sign predictor + exact per-row top-k (Nk <= 256).
//
// Mapping: one CTA per (head, row split); ONE THREAD PER QUERY ROW (128 rows per tile); the keys
// of the head are staged once per CTA in shared memory and broadcast to every row.
//
//   stage   each thread quantizes whole key rows (A1+A2): sign words, block exponents, int8 codes
//           (codes/exps go to HBM for the exact-attention kernel);  per block b the CTA reduces
//           kmin_b = min_j ek_b(j) and stores per key the integer multiplier 2^(ek_b(j)-kmin_b).
//   score   score(i,j) = sum_b 2^(eq_b+ek_b) * (n_b - 2 popc(sq_b ^ sk_b))            (A5)
//           = 2^g * S  with  S = sum_b 2^(eq_b+kmin_b-g) * 2^(ek_b-kmin_b) * (n_b - 2 popc),
//           g = min_b(eq_b+kmin_b).  S is a small even integer, so the row is ranked on the
//           15-bit key u = (S + M)/2 + 1 - no floating point, no rounding, same order and same
//           ties as the fp32 scores (which are exact whenever S fits 24 bits).
//   select  the thread's keys live in shared memory, two per 32-bit word; the top_k-th largest
//           key is found by bit-wise bisection, each step counting (key >= candidate) with one
//           subtraction per two keys (SWAR) and one POPC per eight keys.                  (A6)
//   emit    keys > T are kept, keys == T are kept in ascending key index until top_k is reached
//           (= first top_k of a stable descending sort); the row bitmask is written.
//
// Rows whose exponent spread does not fit the 15-bit key (M > 32766: an all-zero block, or
// > 2^14 dynamic range between tokens) take the generic path: the warp recomputes that row's
// fp32 scores cooperatively and radix-selects on order-preserving float keys.  Both paths return
// identical sets wherever both apply.
#pragma once
#include <cuda_fp16.h>

#include "mxprune_device.cuh"
#include "mxprune_attend.cuh"

namespace mxp {

constexpr int K1T = 128;          // threads per CTA == query rows per tile
constexpr int K1_MAX_SPREAD = 14;
constexpr int K1_MAX_KEYS = 256;
constexpr uint32_t SW_H = 0x80008000u;

struct K1Smem {
    int nkp;        // keys padded to a multiple of 8
    int sstr;       // 32-bit words per thread in the key array, == 4 (mod 32): conflict-free 128-bit access
    size_t off_kexp, off_sc, off_misc, total;
};

__host__ __device__ inline K1Smem k1_smem_layout(int nb, int Nk) {
    K1Smem L;
    L.nkp = (Nk + 7) & ~7;
    L.sstr = L.nkp / 2;
    while ((L.sstr & 31) != 4) L.sstr += 4;
    size_t o = (size_t)L.nkp * 2 * nb * 4;              // records: {sign word, multiplier} per block
    L.off_kexp = o; o += (size_t)nb * L.nkp;            // predictor exponents, int8 [nb][nkp]
    o = (o + 15) & ~(size_t)15;
    L.off_sc = o;   o += (size_t)K1T * L.sstr * 4;      // packed 15-bit keys, [thread][sstr]
    L.off_misc = o; o += 64;                            // kmin[4], kmax[4]
    L.total = o;
    return L;
}

template <int NB>
struct RowQ {
    uint32_t sign[NB];
    int e[NB];      // A2 block exponent
    int ep[NB];     // predictor exponent (A3)
};

// One thread quantizes one row of hd fp32 values (16-byte aligned).  Optionally writes the int8
// codes (4-byte aligned destination).
// op_row (optional): address of this row's first 16-byte bf16 operand chunk, chunks op_stride apart.
// DT: element type of the row (DT_*; 16-bit rows are widened to their exact fp32 bit patterns as they are loaded).
template <int NB, int DT = DT_F32>
__device__ __forceinline__ void quantize_row_thread(const float* __restrict__ row, int hd, bool bf16,
                                                    bool flush, RowQ<NB>& rq, int8_t* codes_out,
                                                    unsigned char* op_row = nullptr, int op_stride = 0) {
    // all loads of the row are issued before the first use: one exposed memory latency per row
    uint32_t xall[NB][32];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int nd = min(32, hd - 32 * b);
        if constexpr (DT == DT_F32) {
#pragma unroll
            for (int v = 0; v < 8; ++v) {
                float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
                if (4 * v < nd) f = __ldg(reinterpret_cast<const float4*>(row + 32 * b) + v);
                xall[b][4 * v + 0] = __float_as_uint(f.x);
                xall[b][4 * v + 1] = __float_as_uint(f.y);
                xall[b][4 * v + 2] = __float_as_uint(f.z);
                xall[b][4 * v + 3] = __float_as_uint(f.w);
            }
        } else {
            load_block_bits<DT>(view_elem<DT>(row, 32 * b), nd, true, xall[b]);
        }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int nd = min(32, hd - 32 * b);
        uint32_t (&xb)[32] = xall[b];
        uint32_t mx4[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int t = 0; t < 32; ++t) {
            if (bf16) xb[t] = bf16_half_away(xb[t]);
            mx4[t & 3] = max(mx4[t & 3], xb[t] & 0x7fffffffu);
        }
        const uint32_t mx = max(max(mx4[0], mx4[1]), max(mx4[2], mx4[3]));
        const int e = mx_shared_exp(mx);
        const bool dead = flush && e <= -127;
        const float s1 = exp2i(-e);
        const float wgt = exp2i(e - 6);
        uint32_t sw = 0u;
        uint32_t cw[8];
        uint32_t ow[16];                                    // dequantised values as bf16 pairs
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            uint32_t word = 0u;
            float fq[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const uint32_t xv = xb[4 * v + t];
                const float r = __uint_as_float(xv & 0x7fffffffu) * s1 * 64.0f + 0.5f;
                int c = min(__float2int_rz(r), 127);       // r >= 0.5: truncation == floor
                if (dead) c = 0;
                const bool neg = (xv >> 31) && c != 0;
                sw |= (neg ? 1u : 0u) << (4 * v + t);
                const int sc = neg ? -c : c;
                word |= ((uint32_t)sc & 0xffu) << (8 * t);
                fq[t] = (float)sc * wgt;                    // c * 2^(e-6): exact in bf16
            }
            cw[v] = word;
            ow[2 * v] = pack_bf16_trunc(fq[0], fq[1]);
            ow[2 * v + 1] = pack_bf16_trunc(fq[2], fq[3]);
        }
        if (op_row) {
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
                if (8 * ch < nd)
                    *reinterpret_cast<uint4*>(op_row + (size_t)(b * 4 + ch) * op_stride) =
                        make_uint4(ow[4 * ch], ow[4 * ch + 1], ow[4 * ch + 2], ow[4 * ch + 3]);
        }
        rq.sign[b] = sw;
        rq.e[b] = e;
        rq.ep[b] = dead ? ZERO_BLOCK_EXP : e;
        if (codes_out) {
            uint32_t* dst = reinterpret_cast<uint32_t*>(codes_out + 32 * b);
#pragma unroll
            for (int v = 0; v < 8; ++v)
                if (4 * v < nd) dst[v] = cw[v];
        }
    }
}

// ask L2 for the hd fp32 values of a row this thread will quantize later
__device__ __forceinline__ void prefetch_row_l2(const float* row, int hd) {
    for (int o = 0; o < hd; o += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + o));
}

// Keys are stored two per 32-bit word as u + K1_KEY_BIAS (<= 0x7BFF): as fp16 BIT PATTERNS they
// are finite, normal, positive numbers whose float order equals their integer order, so one
// HSET2.GE compares two keys and one HADD2 accumulates both counts - on the half/FMA pipe, which
// the rest of this ALU-bound kernel leaves idle.  Padding keys are stored as 0 (below any
// candidate).  Counts stay exact: at most 128 per half lane, far below fp16's 2048.
constexpr uint32_t K1_KEY_BIAS = 0x0400u;        // first normal fp16 bit pattern
constexpr int K1_MAX_M = 0x7BFF - 0x0400 - 2;    // largest |S| bound that keeps biased keys finite fp16

__device__ __forceinline__ uint32_t h2_as_u32(__half2 x) {
    return *reinterpret_cast<const uint32_t*>(&x);
}
__device__ __forceinline__ __half2 u32_as_h2(uint32_t x) {
    return *reinterpret_cast<const __half2*>(&x);
}
// number of this thread's keys >= cand (cand given WITH bias)
__device__ __forceinline__ int h2_count_ge(const uint32_t* sc, int ng, uint32_t cand) {
    const __half2 c2 = u32_as_h2(cand * 0x00010001u);
    __half2 a0 = u32_as_h2(0u), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll 4
    for (int jg = 0; jg < ng; ++jg) {
        const uint4 w = *reinterpret_cast<const uint4*>(sc + jg * 4);
        a0 = __hadd2(a0, __hge2(u32_as_h2(w.x), c2));
        a1 = __hadd2(a1, __hge2(u32_as_h2(w.y), c2));
        a2 = __hadd2(a2, __hge2(u32_as_h2(w.z), c2));
        a3 = __hadd2(a3, __hge2(u32_as_h2(w.w), c2));
    }
    const __half2 t = __hadd2(__hadd2(a0, a1), __hadd2(a2, a3));
    return (int)(__low2float(t) + __high2float(t));
}

// (key >= cand) flags of one group of 8 keys, bit t = key t of the group
__device__ __forceinline__ uint32_t swar_flags8(const uint4& w, uint32_t c2) {
    // (key | 0x8000) - cand keeps bit 15 of each half iff key >= cand (keys, cand < 0x8000)
    const uint32_t x = ((((w.x | SW_H) - c2) & SW_H) >> 15) | ((((w.y | SW_H) - c2) & SW_H) >> 14) |
                       ((((w.z | SW_H) - c2) & SW_H) >> 13) | ((((w.w | SW_H) - c2) & SW_H) >> 12);
    return (x & 0xFu) | ((x >> 12) & 0xF0u);
}

// Generic path, warp-cooperative, one row: fp32 scores on order-preserving keys (any exponents).
template <int NB>
struct GenRow {
    uint32_t sq[NB];
    int ep[NB];
};

template <int NB>
__device__ __noinline__ void predict_row_generic(uint32_t* __restrict__ mask_out, int32_t* __restrict__ idx_out,
                                                 int Nk, int kk, int hd, int64_t row, GenRow<NB> gr,
                                                 const uint32_t* s_krec, const signed char* s_kexp, int nkp,
                                                 const float* kbias = nullptr) {
    constexpr int KPL = K1_MAX_KEYS / 32;
    const int lane = threadIdx.x & 31;
    uint32_t u[KPL];
    uint32_t aor = 0u, aand = 0xffffffffu;
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int j = r * 32 + lane;
        const bool valid = j < Nk;
        float s = 0.f;
        if (valid) {
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
                const float cnt = (float)(nbw - 2 * __popc(s_krec[(j * NB + b) * 2] ^ gr.sq[b]));
                const float t = exp2i((int)s_kexp[b * nkp + j]) * cnt;
                s = (b == 0) ? t * exp2i(gr.ep[0]) : fmaf(t, exp2i(gr.ep[b]), s);
            }
            if (kbias) s = __fadd_rn(s, __ldg(kbias + j));          // pred_scores + attn_bias, fp32
        }
        u[r] = valid ? ordered_key(s) : 0u;
        aor |= u[r];
        aand &= valid ? u[r] : 0xffffffffu;
    }
    aor = __reduce_or_sync(FULL, aor);
    aand = __reduce_and_sync(FULL, aand);
    uint32_t T = aand, vary = aor & ~aand;
    while (vary) {
        const uint32_t m1 = 1u << (31 - __clz(vary));
        vary ^= m1;
        const uint32_t cand = T | m1;
        int c = 0;
#pragma unroll
        for (int r = 0; r < KPL; ++r) c += (u[r] >= cand) ? 1 : 0;
        c = __reduce_add_sync(FULL, c);
        if (c >= kk) T = cand;
    }
    uint32_t ge[KPL], gt[KPL];
    int ngt = 0;
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        ge[r] = __ballot_sync(FULL, u[r] >= T);
        gt[r] = __ballot_sync(FULL, u[r] > T);
        ngt += __popc(gt[r]);
    }
    int rem = kk - ngt, base = 0;
    uint32_t myword = 0u;
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const uint32_t eq = ge[r] & ~gt[r];
        const int c = __popc(eq);
        uint32_t take;
        if (c <= rem) { take = eq; rem -= c; }
        else { take = keep_lowest_bits(eq, rem); rem = 0; }
        const uint32_t w = gt[r] | take;
        if (lane == r) myword = w;
        if (idx_out) {
            if ((w >> lane) & 1u) idx_out[row * kk + base + __popc(w & ((1u << lane) - 1u))] = r * 32 + lane;
            base += __popc(w);
        }
    }
    const int NW = (Nk + 31) >> 5;
    if (lane < NW) mask_out[row * NW + lane] = myword;
}

template <int NB>
__global__ void __launch_bounds__(K1T, (NB <= 2 ? 4 : 3))
k_predict_topk_rows(const PredParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Nk = p.Nk, Nq = p.Nq, hd = p.hd, kk = p.top_k;
    const K1Smem L = k1_smem_layout(NB, Nk);
    const int nkp = L.nkp, sstr = L.sstr, ng = nkp >> 3;
    uint32_t* s_krec = reinterpret_cast<uint32_t*>(smem_raw);
    signed char* s_kexp = reinterpret_cast<signed char*>(smem_raw + L.off_kexp);
    uint32_t* s_sc = reinterpret_cast<uint32_t*>(smem_raw + L.off_sc);
    int* s_kmin = reinterpret_cast<int*>(smem_raw + L.off_misc);
    int* s_kmax = s_kmin + 4;

    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int tid = threadIdx.x;
    const bool bf16 = p.bf16, flush = p.flush;
    const bool write_k = p.k_codes != nullptr && blockIdx.y == 0;
    const bool write_kop = p.k_op != nullptr && blockIdx.y == 0;
    const OpsLayout OL = ops_layout(Nq, Nk, hd);
    unsigned char* k_op = p.k_op ? p.k_op + (size_t)head * OL.k_head_bytes : nullptr;
    unsigned char* q_op = p.q_op ? p.q_op + (size_t)head * OL.q_head_bytes : nullptr;

    // ---------------- stage the keys of this head
    if (tid < 4) { s_kmin[tid] = 0x7fffffff; s_kmax[tid] = -0x7fffffff; }
    __syncthreads();
    {
        const float* kb = p.k.p + bb * p.k.sB + hh * p.k.sH;
        {   // first query row of this thread: in L2 by the time the keys are staged
            const int iq = blockIdx.y * K1T + tid;
            if (iq < Nq) prefetch_row_l2(p.q.p + bb * p.q.sB + hh * p.q.sH + (int64_t)iq * p.q.sN, hd);
        }
        for (int j = tid; j < nkp; j += K1T) {
            if (j + K1T < Nk) prefetch_row_l2(kb + (int64_t)(j + K1T) * p.k.sN, hd);
            if (j < Nk) {
                RowQ<NB> kq;
                const int64_t krow = (int64_t)head * Nk + j;
                quantize_row_thread<NB>(kb + (int64_t)j * p.k.sN, hd, bf16, flush, kq,
                                        write_k ? p.k_codes + krow * hd : nullptr,
                                        write_kop ? k_op + k_op_offset(OL, j, 0) : nullptr, OL.kb_rows * 16);
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    s_krec[(j * NB + b) * 2] = kq.sign[b];
                    s_kexp[b * nkp + j] = (signed char)kq.ep[b];
                    atomicMin(&s_kmin[b], kq.ep[b]);
                    atomicMax(&s_kmax[b], kq.ep[b]);
                    if (write_k) p.k_exps[krow * NB + b] = (int8_t)kq.e[b];
                }
            } else {
#pragma unroll
                for (int b = 0; b < NB; ++b) { s_krec[(j * NB + b) * 2] = 0u; s_kexp[b * nkp + j] = 0; }
            }
        }
        if (write_kop) {        // zero the padding of the operand image (key rows / head_dim up to 16)
            const int kch = OL.hdp >> 3, rows_pad = OL.nblk * OL.kb_rows;
            for (int t = tid; t < rows_pad * kch; t += K1T) {
                const int j = t % rows_pad, kc = t / rows_pad;
                if (j >= Nk || kc * 8 >= hd)
                    *reinterpret_cast<uint4*>(k_op + k_op_offset(OL, j, kc)) = make_uint4(0u, 0u, 0u, 0u);
            }
        }
    }
    __syncthreads();
    int kmin[NB], spread[NB];
    bool wide = false;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        kmin[b] = s_kmin[b];
        spread[b] = s_kmax[b] - kmin[b];
        wide |= spread[b] > K1_MAX_SPREAD;
    }
    for (int j = tid; j < nkp; j += K1T) {
#pragma unroll
        for (int b = 0; b < NB; ++b)
            s_krec[(j * NB + b) * 2 + 1] = (j < Nk && !wide) ? 1u << ((int)s_kexp[b * nkp + j] - kmin[b]) : 0u;
    }
    __syncthreads();

    const float* qb = p.q.p + bb * p.q.sB + hh * p.q.sH;
    const int NW = (Nk + 31) >> 5;
    uint32_t* my_sc = s_sc + tid * sstr;

    for (int i0 = blockIdx.y * K1T; i0 < Nq; i0 += K1T * gridDim.y) {
        const int i = i0 + tid;
        const bool valid = i < Nq;
        const int64_t row = (int64_t)head * Nq + (valid ? i : 0);
        RowQ<NB> rq;
        if (i + K1T * (int)gridDim.y < Nq) prefetch_row_l2(qb + (int64_t)(i + K1T * (int)gridDim.y) * p.q.sN, hd);
        if (q_op) {             // padding of the A-operand tile: rows past Nq, head_dim up to 16
            for (int kc = 0; kc < (OL.hdp >> 3); ++kc)
                if (!valid || kc * 8 >= hd)
                    *reinterpret_cast<uint4*>(q_op + q_op_offset(OL, i, kc)) = make_uint4(0u, 0u, 0u, 0u);
        }
        if (valid) {
            quantize_row_thread<NB>(qb + (int64_t)i * p.q.sN, hd, bf16, flush, rq,
                                    p.q_codes ? p.q_codes + row * hd : nullptr,
                                    q_op ? q_op + q_op_offset(OL, i, 0) : nullptr, K2T * 16);
            if (p.q_exps) {
#pragma unroll
                for (int b = 0; b < NB; ++b) p.q_exps[row * NB + b] = (int8_t)rq.e[b];
            }
        } else {
#pragma unroll
            for (int b = 0; b < NB; ++b) { rq.sign[b] = 0u; rq.e[b] = 0; rq.ep[b] = 0; }
        }
        // ---- integer-key parameters of this row
        int g = 0x7fffffff;
#pragma unroll
        for (int b = 0; b < NB; ++b) g = min(g, rq.ep[b] + kmin[b]);
        bool fast = valid && !wide && p.key_bias == nullptr;
        int mq[NB];
        long long M = 0;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            int sh = rq.ep[b] + kmin[b] - g;
            if (sh > K1_MAX_SPREAD) { fast = false; sh = K1_MAX_SPREAD; }
            mq[b] = 1 << sh;
            const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
            M += (long long)nbw << (sh + min(spread[b], K1_MAX_SPREAD));
        }
        if (M > K1_MAX_M) fast = false;
        if (!fast) {
            M = 0;
#pragma unroll
            for (int b = 0; b < NB; ++b) mq[b] = 0;
        }
        const int moff = ((int)M + 1) & ~1;

        // ---- pass 1: integer scores -> packed 15-bit keys in shared memory
        // (groups of 8 keys; only the last group can contain padding keys, which get key 0)
        for (int jg = 0; jg < ng; ++jg) {
            uint32_t us[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int j = jg * 8 + t;
                int S = moff;
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const uint2 rec = *reinterpret_cast<const uint2*>(s_krec + (j * NB + b) * 2);
                    const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
                    const int c = nbw - 2 * __popc(rq.sign[b] ^ rec.x);
                    S += (c * (int)rec.y) * mq[b];
                }
                us[t] = ((uint32_t)S >> 1) + 1u + K1_KEY_BIAS;
            }
            if (jg == ng - 1) {
#pragma unroll
                for (int t = 0; t < 8; ++t)
                    if (jg * 8 + t >= Nk) us[t] = 0u;
            }
            *reinterpret_cast<uint4*>(my_sc + jg * 4) =
                make_uint4(us[0] | (us[4] << 16), us[1] | (us[5] << 16), us[2] | (us[6] << 16),
                           us[3] | (us[7] << 16));
        }

        // ---- select: T = top_k-th largest key, bit-wise bisection (warp-uniform trip count)
        int wbits = 32 - __clz(moff + 1);
        wbits = __reduce_max_sync(FULL, wbits);
        uint32_t Tv = 0u;                                   // unbiased key value
        // the last rejected candidate is T + 1 (T's lowest zero bit set, the accepted ones below it cleared), so
        // its count is the number of keys > T; nothing rejected: T is all ones and no key lies above it
        int ngt = 0;
        for (int bit = wbits - 1; bit >= 0; --bit) {
            const uint32_t cand = Tv | (1u << bit);
            const int cnt = h2_count_ge(my_sc, ng, cand + K1_KEY_BIAS);
            if (cnt >= kk) Tv = cand; else ngt = cnt;
        }
        const uint32_t T = Tv + K1_KEY_BIAS;
        const bool has_gt = true;                           // T + 1 <= 0x7C00 - 1 by construction of K1_MAX_M

        // ---- emit the row bitmask (ties: ascending key index)
        {
            int rem = kk - ngt, pos = 0;
            uint32_t word = 0u;
            const uint32_t cT = T * 0x00010001u, cT1 = (T + 1u) * 0x00010001u;
            const bool store = valid && fast;
            for (int jg = 0; jg < ng; ++jg) {
                const uint4 w = *reinterpret_cast<const uint4*>(my_sc + jg * 4);
                const uint32_t ge8 = swar_flags8(w, cT);
                const uint32_t gt8 = has_gt ? swar_flags8(w, cT1) : 0u;
                const uint32_t eq8 = ge8 & ~gt8;
                const int c = __popc(eq8);
                uint32_t take;
                if (c <= rem) { take = eq8; rem -= c; }
                else { take = keep_lowest_bits(eq8, rem); rem = 0; }
                word |= (gt8 | take) << (8 * (jg & 3));
                if ((jg & 3) == 3 || jg == ng - 1) {
                    if (store) {
                        p.mask[row * NW + (jg >> 2)] = word;
                        if (p.idx) {
                            uint32_t w2 = word;
                            while (w2) {
                                const int bpos = __ffs(w2) - 1;
                                w2 &= w2 - 1u;
                                p.idx[row * kk + pos++] = (jg >> 2) * 32 + bpos;
                            }
                        }
                    }
                    word = 0u;
                }
            }
        }

        // ---- rows outside the integer-key window: warp-cooperative generic path
        unsigned todo = __ballot_sync(FULL, valid && !fast);
        while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1u;
            GenRow<NB> gr;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                gr.sq[b] = __shfl_sync(FULL, rq.sign[b], l);
                gr.ep[b] = __shfl_sync(FULL, rq.ep[b], l);
            }
            const int64_t grow = (int64_t)head * Nq + (i0 + (tid & ~31) + l);
            predict_row_generic<NB>(p.mask, p.idx, Nk, kk, hd, grow, gr, s_krec, s_kexp, nkp,
                                    p.key_bias ? p.key_bias + bb * p.kb_sB : nullptr);
        }
    }
}


// ==========================================================================================
// K1-long: the same fused quantizer + predictor + exact top-k for Nk > 256 (long-sequence sweep).
//
// A row's keys no longer fit in shared memory next to 127 other rows, so nothing per-row is
// stored: each thread re-derives its keys from the staged K records in every pass and the k-th
// largest is found by a most-significant-digit radix select over per-thread histograms
// (64 bins x 6 bits per level, [bin][thread] in shared memory => conflict-free, no atomics):
//   level 0..L-1   histogram of the current 6-bit digit among keys whose higher digits equal the
//                  prefix found so far; scan from the top bin to locate the digit of the k-th key
//   emit           keys > T kept, keys == T kept in ascending index until top_k
// Keys are the exact 15-bit integers of the short kernel when the exponent window allows
// (L = 3 levels) and order-preserving fp32 keys otherwise (L = 6) - chosen per row.
// K record per key: NB sign words + one word of per-block shifts (ek_b - kmin_b), 16 bytes.
// ==========================================================================================
constexpr int K1L_BINS = 64;

struct K1LSmem {
    int rw;                         // 32-bit words per key record
    size_t off_hist, off_misc, total;
};
__host__ __device__ inline K1LSmem k1l_smem_layout(int nb, int Nk) {
    K1LSmem L;
    L.rw = nb <= 3 ? 4 : 8;
    size_t o = (size_t)Nk * L.rw * 4;
    o = (o + 15) & ~(size_t)15;
    L.off_hist = o; o += (size_t)K1L_BINS * K1T * 4;
    L.off_misc = o; o += 64;
    L.total = o;
    return L;
}

template <int NB>
struct LongRow {
    uint32_t sign[NB];
    int mq[NB];          // fast: integer row multipliers 2^(eq_b + kmin_b - g)
    float wq[NB];        // slow: 2^eq_b
    int moff;
    bool fast;
};

template <int NB>
__device__ __forceinline__ uint32_t long_key(const LongRow<NB>& R, const uint32_t* rec, const int (&kmin)[NB], int hd) {
    const uint32_t shw = rec[NB];
    if (R.fast) {
        int S = R.moff;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
            const int c = nbw - 2 * __popc(R.sign[b] ^ rec[b]);
            S += (c << ((shw >> (8 * b)) & 0xffu)) * R.mq[b];
        }
        return ((uint32_t)S >> 1) + 1u;
    }
    float s = 0.f;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
        const float cnt = (float)(nbw - 2 * __popc(R.sign[b] ^ rec[b]));
        const float t = exp2i(kmin[b] + (int)((shw >> (8 * b)) & 0xffu)) * cnt;
        s = (b == 0) ? t * R.wq[0] : fmaf(t, R.wq[b], s);
    }
    return ordered_key(s);
}

// DT: element type of the q / k views (DT_*)
template <int NB, int DT = DT_F32>
__global__ void __launch_bounds__(K1T)
k_predict_topk_long(const PredParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Nk = p.Nk, Nq = p.Nq, hd = p.hd, kk = p.top_k;
    const K1LSmem L = k1l_smem_layout(NB, Nk);
    const int RW = L.rw;
    uint32_t* s_rec = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(smem_raw + L.off_hist);
    int* s_kmin = reinterpret_cast<int*>(smem_raw + L.off_misc);
    int* s_kmax = s_kmin + 4;
    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int tid = threadIdx.x;
    const bool bf16 = p.bf16, flush = p.flush;
    const bool write_k = p.k_codes != nullptr && blockIdx.y == 0;
    const bool write_kop = p.k_op != nullptr && blockIdx.y == 0;
    const OpsLayout OL = ops_layout(Nq, Nk, hd);
    unsigned char* k_op = p.k_op ? p.k_op + (size_t)head * OL.k_head_bytes : nullptr;
    unsigned char* q_op = p.q_op ? p.q_op + (size_t)head * OL.q_head_bytes : nullptr;

    if (p.row_filter) {              // only flagged rows are processed; nothing to do -> skip the K staging too
        int any = 0;
        for (int i = blockIdx.y * K1T + tid; i < Nq; i += K1T * gridDim.y) any |= p.row_filter[(int64_t)head * Nq + i];
        if (!__syncthreads_or(any)) return;
    }
    if (tid < 4) { s_kmin[tid] = 0x7fffffff; s_kmax[tid] = -0x7fffffff; }
    __syncthreads();
    {
        const float* kb = view_elem<DT>(p.k.p, bb * p.k.sB + hh * p.k.sH);
        for (int j = tid; j < Nk; j += K1T) {
            RowQ<NB> kq;
            const int64_t krow = (int64_t)head * Nk + j;
            quantize_row_thread<NB, DT>(view_elem<DT>(kb, (int64_t)j * p.k.sN), hd, bf16, flush, kq,
                                    write_k ? p.k_codes + krow * hd : nullptr,
                                    write_kop ? k_op + k_op_offset(OL, j, 0) : nullptr, OL.kb_rows * 16);
            uint32_t epw = 0u;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                s_rec[j * RW + b] = kq.sign[b];
                epw |= (uint32_t)(kq.ep[b] + 128) << (8 * b);        // provisional: biased exponent
                atomicMin(&s_kmin[b], kq.ep[b]);
                atomicMax(&s_kmax[b], kq.ep[b]);
                if (write_k) p.k_exps[krow * NB + b] = (int8_t)kq.e[b];
            }
            s_rec[j * RW + NB] = epw;
        }
        if (write_kop) {
            const int kch = OL.hdp >> 3, rows_pad = OL.nblk * OL.kb_rows;
            for (int t = tid; t < rows_pad * kch; t += K1T) {
                const int j = t % rows_pad, kc = t / rows_pad;
                if (j >= Nk || kc * 8 >= hd)
                    *reinterpret_cast<uint4*>(k_op + k_op_offset(OL, j, kc)) = make_uint4(0u, 0u, 0u, 0u);
            }
        }
    }
    __syncthreads();
    int kmin[NB], spread[NB];
    bool wide = false;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        kmin[b] = s_kmin[b];
        spread[b] = s_kmax[b] - kmin[b];
        wide |= spread[b] > K1_MAX_SPREAD;
    }
    for (int j = tid; j < Nk; j += K1T) {           // biased exponents -> shifts relative to kmin
        const uint32_t epw = s_rec[j * RW + NB];
        uint32_t shw = 0u;
#pragma unroll
        for (int b = 0; b < NB; ++b) shw |= (uint32_t)((int)((epw >> (8 * b)) & 0xffu) - 128 - kmin[b]) << (8 * b);
        s_rec[j * RW + NB] = shw;
    }
    __syncthreads();

    const float* qb = view_elem<DT>(p.q.p, bb * p.q.sB + hh * p.q.sH);
    const int NW = (Nk + 31) >> 5;
    uint32_t* my_hist = s_hist + tid;               // bin b at my_hist[b * K1T]

    for (int i0 = blockIdx.y * K1T; i0 < Nq; i0 += K1T * gridDim.y) {
        const int i = i0 + tid;
        const bool valid = i < Nq && (!p.row_filter || p.row_filter[(int64_t)head * Nq + i]);
        const int64_t row = (int64_t)head * Nq + (valid ? i : 0);
        RowQ<NB> rq;
        if (q_op) {
            for (int kc = 0; kc < (OL.hdp >> 3); ++kc)
                if (!valid || kc * 8 >= hd)
                    *reinterpret_cast<uint4*>(q_op + q_op_offset(OL, i, kc)) = make_uint4(0u, 0u, 0u, 0u);
        }
        if (valid) {
            quantize_row_thread<NB, DT>(view_elem<DT>(qb, (int64_t)i * p.q.sN), hd, bf16, flush, rq,
                                        p.q_codes ? p.q_codes + row * hd : nullptr,
                                        q_op ? q_op + q_op_offset(OL, i, 0) : nullptr, K2T * 16);
            if (p.q_exps) {
#pragma unroll
                for (int b = 0; b < NB; ++b) p.q_exps[row * NB + b] = (int8_t)rq.e[b];
            }
        } else {
#pragma unroll
            for (int b = 0; b < NB; ++b) { rq.sign[b] = 0u; rq.e[b] = 0; rq.ep[b] = 0; }
        }
        LongRow<NB> R;
        int g = 0x7fffffff;
#pragma unroll
        for (int b = 0; b < NB; ++b) g = min(g, rq.ep[b] + kmin[b]);
        R.fast = !wide;
        long long M = 0;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            int sh = rq.ep[b] + kmin[b] - g;
            if (sh > K1_MAX_SPREAD) { R.fast = false; sh = K1_MAX_SPREAD; }
            R.sign[b] = rq.sign[b];
            R.mq[b] = 1 << sh;
            R.wq[b] = exp2i(rq.ep[b]);
            const int nbw = (b < NB - 1) ? 32 : hd - 32 * (NB - 1);
            M += (long long)nbw << (sh + min(spread[b], K1_MAX_SPREAD));
        }
        if (M > 32766) R.fast = false;
        R.moff = R.fast ? (((int)M + 1) & ~1) : 0;
        const int wtot = R.fast ? 32 - __clz(R.moff + 1) : 32;       // key width in bits
        int nlev = (wtot + 5) / 6;
        nlev = __reduce_max_sync(FULL, nlev);

        // ---- MSD radix select over per-thread histograms
        uint32_t prefix = 0u;       // digits found so far (right-aligned)
        int krem = kk;
        for (int lev = 0; lev < nlev; ++lev) {
            const int my_lev = (wtot + 5) / 6;
            const int lo = 6 * (my_lev - 1 - lev);              // < 0: this row already has its full key
            for (int b = 0; b < K1L_BINS; ++b) my_hist[b * K1T] = 0u;
            if (lo >= 0) {
                for (int j = 0; j < Nk; ++j) {
                    const uint32_t u = long_key<NB>(R, s_rec + j * RW, kmin, hd);
                    const uint32_t hi = (lo + 6 >= 32) ? 0u : (u >> (lo + 6));
                    if (hi == prefix) my_hist[((u >> lo) & 63u) * K1T] += 1u;
                }
                int cum = 0, bin = K1L_BINS - 1;
                for (; bin > 0; --bin) {
                    const int h = (int)my_hist[bin * K1T];
                    if (cum + h >= krem) break;
                    cum += h;
                }
                krem -= cum;
                prefix = (prefix << 6) | (uint32_t)bin;
            }
        }
        const uint32_t T = prefix;

        // ---- emit: keys > T, then keys == T in ascending index until top_k (krem ties wanted)
        {
            int rem = krem, pos = 0;
            uint32_t word = 0u;
            for (int j = 0; j < Nk; ++j) {
                const uint32_t u = long_key<NB>(R, s_rec + j * RW, kmin, hd);
                bool keep = u > T;
                if (u == T && rem > 0) { keep = true; --rem; }
                word |= (keep ? 1u : 0u) << (j & 31);
                if ((j & 31) == 31 || j == Nk - 1) {
                    if (valid) {
                        p.mask[row * NW + (j >> 5)] = word;
                        if (p.idx) {
                            uint32_t w2 = word;
                            while (w2) {
                                const int bpos = __ffs(w2) - 1;
                                w2 &= w2 - 1u;
                                p.idx[row * kk + pos++] = (j & ~31) + bpos;
                            }
                        }
                    }
                    word = 0u;
                }
            }
        }
    }
}

}  // namespace mxp
