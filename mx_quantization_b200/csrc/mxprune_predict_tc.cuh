// K1-TC: fused MX quantizer + exponent-sign predictor + exact per-row top-k for Nk <= 256,
// scored on the tensor cores, selected in registers.
//
// The reference's predictor is a dense fp32 matmul of +-2^e operands
// (workloads/deit/scripts/main.py:118, funcs/exponent_based_prediction.py:44-94).  +-2^e is exact
// in bf16 and every partial sum of one (query, key) pair is an integer multiple of 2^g inside a
// 16-bit window, so tcgen05.mma kind::f16 with fp32 accumulators returns the reference's score
// bit for bit (tools/umma_exact_test.cu: exact up to a 20-bit window on B200).  XOR+POPC scoring on
// CUDA cores costs ~12 instructions per (row, key); the tensor core makes it free and leaves the
// CUDA cores to the quantizer and the selection.
//
// One CTA (256 threads) per (head, row split), two CTAs resident per SM (16 warps; TMEM - 256
// columns per CTA - and the register-resident keys are what bound the residency).
//   stage    Q/K fp32 rows arrive by TMA (cp.async.bulk.tensor) straight from the strided
//            (B,H,N,hd) view: tensor map dims {32 floats, N, hd/32, H, B}, box {32, 64 rows, hd/32},
//            SWIZZLE_128B, out-of-range rows zero-filled; a second, unswizzled map covers hd % 32.
//            A ring of slots (64 or 128 rows) keeps the next rows in flight while the current ones
//            are quantized.
//   quantize one thread per 32-wide MX block (conflict-free 128-bit reads of the swizzled slot):
//            A1 + A2 -> exact bf16 operand c*2^(e-6) for the attention kernel (HBM, MMA-ready),
//            predictor operand +-2^e (shared memory, MMA-ready), sign word + exponent (shared
//            memory, for the generic path), optional int8 codes / exponents (HBM).
//            No float<->int conversion instructions: floor() is an FADD.RM against 2^23 and the
//            bf16 value comes from one packed HFMA2.BF16 on the (128 + c) bit patterns.
//   score    S[128 x 32 NC] = Qp . Kp^T, hd/16 tcgen05.mma (M = 128), fp32 in TMEM
//   keys     a warp owns 16 query rows (TMEM lanes); lanes l and l + 16 share row l and split its key
//            columns in two halves - tcgen05.ld.16x32bx2 delivers exactly that.  score * 2^(-g-1) +
//            offset is the same 15-bit integer key as the CUDA-core kernel (mxprune_predict.cuh),
//            stored as an fp16 BIT PATTERN, two per register (<= 64 registers per thread)
//   select   bit-wise bisection for the top_k-th largest key: per step one HSET2.GE + one HADD2 per
//            two keys, no memory traffic; the two lanes of a row add their counts with one SHFL
//   emit     keys > T kept, keys == T kept in ascending key index until top_k (stable-sort rule)
// Rows outside the integer window (all-zero block, > 2^14 spread) take the same warp-cooperative
// fp32 path as the CUDA-core kernel, from the sign words kept in shared memory.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cuda_runtime.h>

#include "mxprune_host.cuh"
#include "mxprune_predict.cuh"

namespace mxp {

constexpr int K1C_T = 256;            // threads per CTA: two per query row of the tile
constexpr int K1C_TILE = 128;         // query rows per tile == TMEM lanes
constexpr int K1C_ROWS = 64;          // rows per TMA box
constexpr int K1C_MAXR = 4;           // ring slots

struct K1cSmem {
    int nfull, tail, nb, hdp, n_mma, tmem_cols, ring, G;
    size_t box_main, box_tail, slot_bytes;
    size_t off_kop, off_qop, off_ksign, off_kexp, off_qsign, off_qexp, off_misc, total;
};

// nc = number of 32-key chunks (the kernel's NC): the MMA covers 32 * nc key columns, rows past Nk
// of the predictor operand are zero so that padding keys score exactly 0.
// G = TMA boxes (of 64 rows) per ring slot == per quantize step.
// biased: two extra K columns carry the additive key bias through the MMA (see the kernel).
// opw = operand width multiplier: 2 when each side carries two operand parts [A | B] per row (K1-wide's
// two_step_leading_ones mode), chunk c of part B at chunk index (hdp >> 3) + c.
__host__ __device__ constexpr inline K1cSmem k1c_smem_layout(int hd, int nc, int ring, int G, bool biased = false, int opw = 1) {
    K1cSmem L{};
    L.nfull = hd >> 5;
    L.tail = hd & 31;
    L.nb = (hd + 31) >> 5;
    L.hdp = (hd + (biased ? 2 : 0) + 15) & ~15;
    L.n_mma = 32 * nc;
    int c = 32;
    while (c < 64 * ((nc + 1) / 2)) c <<= 1;              // both lane halves read (nc + 1) / 2 chunks
    L.tmem_cols = c;
    L.ring = ring;
    L.G = G;
    L.box_main = (size_t)K1C_ROWS * L.nfull * 128;
    L.box_tail = (size_t)K1C_ROWS * L.tail * 4;
    L.slot_bytes = (G * (L.box_main + L.box_tail) + 1023) & ~(size_t)1023;
    size_t o = L.slot_bytes * ring;
    L.off_kop = o;   o += (size_t)opw * (L.hdp >> 3) * L.n_mma * 16;
    L.off_qop = o;   o += (size_t)opw * (L.hdp >> 3) * K1C_TILE * 16;
    L.off_ksign = o; o += (size_t)L.nb * 256 * 4;
    L.off_kexp = o;  o += (size_t)L.nb * 256;
    L.off_qsign = o; o += (size_t)L.nb * K1C_TILE * 4;
    L.off_qexp = o;  o += (size_t)L.nb * K1C_TILE;
    L.off_misc = o;  o += 128;
    L.total = o;
    return L;
}

// Staging geometry of the stand-alone K1 launch as a function of (head_dim, key chunks): G = TMA boxes per ring slot
// (2 when a 64-row box gives fewer than 256 block tasks), ring = as many slots as fit with two CTAs per SM.
// constexpr: the launcher and the head_dim-specialised instantiations (template HD) evaluate the same rule.
constexpr size_t K1C_PER_CTA2 = 232448 / 2 - 1024, K1C_PER_CTA1 = 232448 - 1024;
__host__ __device__ constexpr inline int k1c_G(int hd, int nc, bool biased) {
    const int nb = (hd + 31) / 32;
    int G = nb <= 2 ? 2 : 1;
    if (k1c_smem_layout(hd, nc, 2, G, biased).total > K1C_PER_CTA2) G = 1;
    return G;
}
__host__ __device__ constexpr inline int k1c_ring(int hd, int nc, bool biased) {
    const int G = k1c_G(hd, nc, biased);
    int ring = K1C_MAXR;
    while (ring > 2 && k1c_smem_layout(hd, nc, ring, G, biased).total > K1C_PER_CTA2) --ring;
    return ring;
}

struct K1cMaps {
    CUtensorMap q_main, q_tail, k_main, k_tail;
};

// ---- K1-TC: tensor maps over the strided (B,H,N,hd) fp32 views + launch ----------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return (EncodeTiledFn)f;
    }();
    return fn;
}

// main map: dims {32 floats, N, hd/32, H, B}, box {32, 64, hd/32, 1, 1}, SWIZZLE_128B;
// tail map (hd % 32 floats at column 32*(hd/32)): dims {tail, N, H, B}, box {tail, 64, 1, 1}.
// dt (DT_*): element type of the view.  16-bit views: the same boxes in elements, 64-byte rows, SWIZZLE_64B (a box fills
// half of the space an fp32 box takes; slot geometry is the fp32 one).
inline bool make_view_maps(const View& v, int B, int H, int N, int hd, CUtensorMap* m_main, CUtensorMap* m_tail,
                           int dt = DT_F32) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const int nfull = hd >> 5, tail = hd & 31;
    const int es_b = dt == DT_F32 ? 4 : 2;
    const CUtensorMapDataType tdt = dt == DT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                  : dt == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const cuuint64_t sN = (cuuint64_t)v.sN * es_b, sH = (cuuint64_t)(H > 1 ? v.sH : hd) * es_b,
                     sB = (cuuint64_t)(B > 1 ? v.sB : (int64_t)N * v.sN) * es_b;
    if (!sN || !sH || !sB || (sN >> 40) || (sH >> 40) || (sB >> 40)) return false;
    if (nfull) {
        cuuint64_t dims[5] = {32, (cuuint64_t)N, (cuuint64_t)nfull, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t strides[4] = {sN, (cuuint64_t)(32 * es_b), sH, sB};
        cuuint32_t box[5] = {32, (cuuint32_t)K1C_ROWS, (cuuint32_t)nfull, 1, 1}, es[5] = {1, 1, 1, 1, 1};
        if (enc(m_main, tdt, 5, (void*)v.p, dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, dt == DT_F32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return false;
    }
    if (tail) {
        cuuint64_t dims[4] = {(cuuint64_t)tail, (cuuint64_t)N, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t strides[3] = {sN, sH, sB};
        cuuint32_t box[4] = {(cuuint32_t)tail, (cuuint32_t)K1C_ROWS, 1, 1}, es[4] = {1, 1, 1, 1};
        if (enc(m_tail, tdt, 4, (void*)((const char*)v.p + (size_t)32 * nfull * es_b), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return false;
    }
    return true;
}


// ---- TMA tensor loads (tile mode), completion counted on an mbarrier
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2,%3,%4,%5,%6}], [%7];" ::
        "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4),
        "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2,%3,%4,%5}], [%6];" ::
        "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
        "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

// One MX block of a staged 16-bit row as fp32 bit patterns (the fp32 kernels read their 128-byte SWIZZLE_128B rows
// inline).  Box g of the ring slot: main box at slot + g box_main - rows of 32 elements, block-major, 64 bytes per row,
// SWIZZLE_64B (16-byte chunk s of row r at s ^ ((r >> 1) & 3): conflict-free for consecutive rows on consecutive lanes);
// tail box at slot + tail_base + g box_tail - tail elements per row, unswizzled; rl6: row within the box.
template <int DT>
__device__ __forceinline__ void staged_block_bits_16(const unsigned char* slot, int g, uint32_t box_main,
                                                     uint32_t tail_base, uint32_t box_tail, int b, int rl6, bool full,
                                                     int tail, uint32_t (&xv)[32]) {
    if (full) {
        const unsigned char* src = slot + g * box_main + (b * 64 + rl6) * 64;
        const int sw = ((rl6 >> 1) & 3) << 4;
#pragma unroll
        for (int s = 0; s < 4; ++s) widen8<DT>(*reinterpret_cast<const uint4*>(src + ((s << 4) ^ sw)), &xv[8 * s]);
    } else {
        const unsigned char* src = slot + tail_base + g * box_tail + rl6 * tail * 2;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (8 * s < tail) v = *reinterpret_cast<const uint4*>(src + (s << 4));
            widen8<DT>(v, &xv[8 * s]);
        }
    }
}

// Results of quantizing one MX block (<= 32 elements) held by one thread.
struct BlockQ {
    int e, ep;              // A2 exponent, predictor exponent
    uint32_t sign;          // predictor sign bits, element (8c + 2p + h) at bit 4c + p + 16h
    uint4 op[4];            // exact operand  c * 2^(e-6), 8 bf16 per chunk
    uint4 pp[4];            // predictor operand +-2^ep
    uint32_t cw[8];         // int8 codes, 4 per word (only when CODES)
};

// xv: the block's 32 fp32 bit patterns (elements >= nd are zero).  A1 + A2 + operand formation.
// PRED = false skips the predictor operand and the sign word (callers that only need c * 2^(e-6)).
template <bool CODES, bool PRED = true>
__device__ __forceinline__ void quantize_block_thread(uint32_t (&xv)[32], int nd, bool bf16, bool flush, BlockQ& r) {
    if (bf16) {
#pragma unroll
        for (int t = 0; t < 32; ++t) xv[t] = bf16_half_away(xv[t]);
    }
    float mx4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < 32; ++t) mx4[t & 3] = fmaxf(mx4[t & 3], fabsf(__uint_as_float(xv[t])));
    const uint32_t mx = __float_as_uint(fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])));
    const int e = mx_shared_exp(mx);
    const bool dead = flush && e <= -127;
    r.e = e;
    r.ep = dead ? ZERO_BLOCK_EXP : e;
    const uint32_t e2 = bf16_pow2_bits(r.ep) * 0x00010001u;
    uint32_t sw = 0u;
    if (mx == 0u) {
        // all-zero block (also every out-of-range row the TMA zero-filled): codes 0, signs +
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            r.op[c] = make_uint4(0u, 0u, 0u, 0u);
            r.pp[c] = make_uint4(e2, e2, e2, e2);
        }
        if (CODES) {
#pragma unroll
            for (int v = 0; v < 8; ++v) r.cw[v] = 0u;
        }
    } else if (!dead && e >= -120 && e <= 126) {
        // floor(|x| * 2^(6-e) + 0.5) without F2I: RN add of 0.5 (as the reference rounds it), clamp,
        // then an add rounded toward -inf against 2^23 + 0x4300 leaves 0x4300 + c in the low 16
        // bits == the bf16 bit pattern of 128 + c;  (128 + c) * w - 128 * w = c * w exactly.
        const float s1 = exp2i(6 - e);
        const uint32_t wb = bf16_pow2_bits(e - 6) * 0x00010001u;
        const __nv_bfloat162 w2 = u32_as_bf2(wb);
        const __nv_bfloat162 nw2 = u32_as_bf2((bf16_pow2_bits(e + 1) | 0x8000u) * 0x00010001u);   // -128 * 2^(e-6)
        const __nv_bfloat162 zero2 = u32_as_bf2(0u);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t ow[4], pw[4], fl[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                float v = fmaf(fabsf(__uint_as_float(xv[8 * c + t])), s1, 0.5f);
                v = fminf(v, 127.0f);
                fl[t] = __float_as_uint(__fadd_rd(v, 8405760.0f));          // 2^23 + 0x4300
            }
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const uint32_t v2 = __byte_perm(fl[2 * p], fl[2 * p + 1], 0x5410);
                const uint32_t sx = __byte_perm(xv[8 * c + 2 * p], xv[8 * c + 2 * p + 1], 0x7632) & 0x80008000u;
                const uint32_t rr = bf2_as_u32(__hfma2(u32_as_bf2(v2), w2, nw2)) ^ sx;
                ow[p] = rr;
                if (PRED) {
                    const uint32_t m = __hlt2_mask(u32_as_bf2(rr), zero2);  // -0 is not < 0: zero codes count as +
                    pw[p] = (m & 0x80008000u) | e2;
                    sw |= m & (0x00010001u << (4 * c + p));
                } else {
                    pw[p] = 0u;
                }
            }
            r.op[c] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            r.pp[c] = make_uint4(pw[0], pw[1], pw[2], pw[3]);
            if (CODES) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t word = 0u;
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const int el = 8 * c + 4 * h + t;
                        const int cm = (int)(fl[4 * h + t] & 0x7fu);
                        const int sc = (xv[el] >> 31) ? -cm : cm;
                        word |= ((uint32_t)sc & 0xffu) << (8 * t);
                    }
                    r.cw[2 * c + h] = word;
                }
            }
        }
    } else {
        // rare: zero / flushed / extreme-exponent block - scalar arithmetic of mxprune_device.cuh
        const float wgt = exp2i(e - 6);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t ow[4], pw[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const int c0 = mx_code(xv[8 * c + 2 * p], e, dead), c1 = mx_code(xv[8 * c + 2 * p + 1], e, dead);
                ow[p] = pack_bf16_trunc((float)c0 * wgt, (float)c1 * wgt);
                const uint32_t m = (c0 < 0 ? 0x0000ffffu : 0u) | (c1 < 0 ? 0xffff0000u : 0u);
                pw[p] = (m & 0x80008000u) | e2;
                sw |= m & (0x00010001u << (4 * c + p));
                if (CODES) {
                    const uint32_t two = ((uint32_t)c0 & 0xffu) | (((uint32_t)c1 & 0xffu) << 8);
                    if (p & 1) r.cw[2 * c + (p >> 1)] |= two << 16;
                    else r.cw[2 * c + (p >> 1)] = two;
                }
            }
            r.op[c] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            r.pp[c] = make_uint4(pw[0], pw[1], pw[2], pw[3]);
        }
    }
    // padding lanes of a partial block carry no sign and no predictor weight
    if (nd < 32) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (8 * c >= nd) r.pp[c] = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    r.sign = sw;
}

// number of keys >= cand among NW2 register words (two fp16-pattern keys per word)
template <int NW2>
__device__ __forceinline__ int count_ge_regs(const uint32_t (&kw)[NW2], uint32_t cand) {
    const __half2 c2 = u32_as_h2(cand * 0x00010001u);
    __half2 a0 = u32_as_h2(0u), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
    for (int w = 0; w < NW2; w += 4) {
        a0 = __hadd2(a0, __hge2(u32_as_h2(kw[w]), c2));
        a1 = __hadd2(a1, __hge2(u32_as_h2(kw[w + 1]), c2));
        a2 = __hadd2(a2, __hge2(u32_as_h2(kw[w + 2]), c2));
        a3 = __hadd2(a3, __hge2(u32_as_h2(kw[w + 3]), c2));
    }
    const __half2 t = __hadd2(__hadd2(a0, a1), __hadd2(a2, a3));
    return (int)(__low2float(t) + __high2float(t));
}


// T = the kk-th largest key of a row whose keys sit in the registers of its two lanes (kw: two fp16-pattern keys per word),
// by bisection over the row's ACTUAL key range [lo, hi] (one packed min / max scan) instead of the worst-case window the
// integer-key parameters allow: measured ranges are 6 - 8 bits against 9 - 11, i.e. 2 - 3 fewer counting passes for the
// price of 0.8.  Candidates are lo + (Tv | 1 << bit), compared as bit patterns like the keys.
//   key0 / my_pad: padding columns (key index >= Nk) score exactly 0 -> key0; this lane holds my_pad of them
//   nvalid_m / nvalid_o: valid keys of this lane / of the partner lane
//   HAS_UNREAL: a lane may hold all-zero words (a key chunk past NC) - skipped by the range scan, below every candidate
// Returns T; nge_* = keys >= T, ngt_* = keys > T (mine / the partner's).  The counts of keys > T need no pass of their
// own: T + 1 is the last candidate the bisection rejected (T's lowest zero bit set, the accepted bits below it cleared).
template <int NWORDS, bool HAS_UNREAL>
__device__ __forceinline__ uint32_t select_kth_key(const uint32_t (&kw)[NWORDS], uint32_t key0, int my_pad, int kk,
                                                   int nvalid_m, int nvalid_o, int& nge_m, int& nge_o, int& ngt_m,
                                                   int& ngt_o) {
    __half2 mn2 = u32_as_h2(0x7bff7bffu), mx2 = u32_as_h2(0x04000400u);
#pragma unroll
    for (int w = 0; w < NWORDS; ++w) {
        const __half2 v = u32_as_h2(kw[w]);
        mx2 = __hmax2(mx2, v);
        if (HAS_UNREAL) mn2 = __hmin2(mn2, kw[w] == 0u ? mn2 : v);
        else mn2 = __hmin2(mn2, v);
    }
    uint32_t lo = min(h2_as_u32(mn2) & 0xffffu, h2_as_u32(mn2) >> 16);
    uint32_t hi = max(h2_as_u32(mx2) & 0xffffu, h2_as_u32(mx2) >> 16);
    lo = min(lo, __shfl_xor_sync(FULL, lo, 16));
    hi = max(hi, __shfl_xor_sync(FULL, hi, 16));
    const uint32_t range = hi > lo ? hi - lo : 0u;
    int wbits = 32 - __clz(range);
    wbits = __reduce_max_sync(FULL, wbits);                         // one loop count per warp (SHFL inside)
    uint32_t Tv = 0u;
    nge_m = nvalid_m; nge_o = nvalid_o;                             // every valid key is >= lo
    ngt_m = 0; ngt_o = 0;
#pragma unroll 1
    for (int bit = wbits - 1; bit >= 0; --bit) {
        const uint32_t cand = min(lo + (Tv | (1u << bit)), 0x7c00u);        // 0x7c00 (+inf): above every key
        const int mine = count_ge_regs<NWORDS>(kw, cand) - (key0 >= cand ? my_pad : 0);
        const int theirs = __shfl_xor_sync(FULL, mine, 16);
        if (mine + theirs >= kk) { Tv |= 1u << bit; nge_m = mine; nge_o = theirs; }
        else { ngt_m = mine; ngt_o = theirs; }
    }
    return lo + Tv;
}

// keep only the m lowest set bits of x (0 <= m <= 32), branch-free binary search
__device__ __forceinline__ uint32_t keep_lowest_bits_fast(uint32_t x, int m) {
    if (m <= 0) return 0u;
    if (m >= __popc(x)) return x;
    int pos = 0;                                    // bits [0, pos) hold fewer than m set bits
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int c = __popc(x & (((1u << s) - 1u) << pos));
        if (c < m) { m -= c; pos += s; }
    }
    // bit `pos` is the m-th remaining set bit's position or lower; include it
    return x & ((2u << pos) - 1u);
}

// Generic path (any exponents), warp-cooperative, one row: fp32 scores, same summation order as
// predict_row_generic in mxprune_predict.cuh.  s_ksign / s_kexp: [b][256].
static __device__ __noinline__ void predict_row_generic_tc(uint32_t* __restrict__ mask_out, int32_t* __restrict__ idx_out,
                                                    int Nk, int kk, int hd, int nb, int64_t row, const uint32_t* sq,
                                                    const int* ep, const uint32_t* s_ksign,
                                                    const signed char* s_kexp, const float* kbias) {
    constexpr int KPL = 8;
    const int lane = threadIdx.x & 31;
    uint32_t u[KPL];
    uint32_t aor = 0u, aand = 0xffffffffu;
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int j = r * 32 + lane;
        const bool valid = j < Nk;
        float s = 0.f;
        if (valid) {
            for (int b = 0; b < nb; ++b) {
                const int nbw = min(32, hd - 32 * b);
                const float cnt = (float)(nbw - 2 * __popc(s_ksign[b * 256 + j] ^ sq[b]));
                const float t = exp2i((int)s_kexp[b * 256 + j]) * cnt;
                s = (b == 0) ? t * exp2i(ep[0]) : fmaf(t, exp2i(ep[b]), s);
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

// 16 TMEM lanes x 16 consecutive columns, twice: lanes 0-15 of the warp get columns [c, c+16) of
// TMEM lanes L..L+15, lanes 16-31 get columns [c + SPLIT, c + SPLIT + 16) of the same TMEM lanes.
template <int SPLIT>
__device__ __forceinline__ void tmem_ld_16x32bx2_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x32bx2.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16], %17;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr), "n"(SPLIT));
}

template <int SPLIT>
__device__ __forceinline__ void tmem_ld_16x32bx2_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x32bx2.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr), "n"(SPLIT));
}

// NC = number of 32-key TMEM chunks a row's keys occupy (Nk <= 32 * NC); the MMA's N is 32 * NC.
// BIASED: an additive key bias (cross-attention text mask) is present; compiled separately so that the
// unbiased kernel carries none of its code.
// HG != 0: the two lanes of a row split the key columns at 8 HG instead of at a multiple of 32 - lane half 0 owns
// columns [0, 8 HG), half 1 [8 HG, 16 HG) - so that a key count just above a multiple of 32 (DeiT's 197 -> 2 x 104)
// does not cost a whole extra 32-key chunk of selection work per lane; the row mask is then written byte-wise
// (8 HG is a byte boundary of the bitmask).  HG = 0: halves of NCH 32-key chunks, mask written in words.
// HD: head_dim at compile time (0 = run time) - staging geometry and operand offsets fold; BF: A1 rounding at compile
// time (-1 = run time, 0 = bfloat 32, 1 = bfloat 16); DT: element type of the q / k views (DT_*)
template <int NC, bool CODES, bool BIASED, int HG = 0, int HD = 0, int BF = -1, int DT = DT_F32>
__global__ void __launch_bounds__(K1C_T, 2)
k_predict_topk_tc(const PredParams p, const __grid_constant__ K1cMaps maps, const int ring_arg, const int G_arg) {
    extern __shared__ __align__(1024) unsigned char smem_k1c[];     // 1024-byte aligned: SWIZZLE_128B boxes
    unsigned char* const smem = smem_k1c;
    constexpr int NMMA = 32 * NC;
    constexpr int NCH = (NC + 1) / 2;                               // key chunks per thread
    constexpr int HW = HG ? 8 * HG : NCH * 32;                      // key columns per lane
    constexpr int NPAIR = HW / 32, REM = HW - 32 * NPAIR;           // full 32-column chunks + an 8- or 16-column rest
    constexpr int NWORDS = HW / 2;                                  // packed key words per lane
    constexpr int NLW = (HW + 31) / 32;                             // bitmask words per lane (lane-local bit order)
    static_assert(HG == 0 || (!BIASED && !CODES && (REM == 8 || REM == 16) && 16 * HG <= 32 * NC && NWORDS % 4 == 0),
                  "tight split: unbiased kernel, rest of 8 or 16 columns");
    const int Nk = p.Nk, Nq = p.Nq, hd = HD ? HD : p.hd, kk = p.top_k;
    constexpr bool biased = BIASED;
    const int ring = HD ? k1c_ring(HD, NC, BIASED) : ring_arg, G = HD ? k1c_G(HD, NC, BIASED) : G_arg;
    const K1cSmem L = k1c_smem_layout(hd, NC, ring, G, biased);
    const int nfull = L.nfull, tail = L.tail, nb = L.nb;
    const int kch = L.hdp >> 3;                                     // 16-byte chunks per predictor-operand row
    // operand chunks the partial block owns: in the HBM exact operand (its zero padding included) and in
    // the shared-memory predictor operand (with a bias, the chunks past the data belong to the bias columns)
    const int tail_chunks_hbm = (((hd + 15) & ~15) >> 3) - 4 * nfull;
    const int tail_chunks = biased ? (tail + 7) >> 3 : kch - 4 * nfull;
    unsigned char* s_kop = smem + L.off_kop;
    unsigned char* s_qop = smem + L.off_qop;
    uint32_t* s_ksign = reinterpret_cast<uint32_t*>(smem + L.off_ksign);
    signed char* s_kexp = reinterpret_cast<signed char*>(smem + L.off_kexp);
    uint32_t* s_qsign = reinterpret_cast<uint32_t*>(smem + L.off_qsign);
    signed char* s_qexp = reinterpret_cast<signed char*>(smem + L.off_qexp);
    int* s_kmin = reinterpret_cast<int*>(smem + L.off_misc);        // [4]
    int* s_kmax = s_kmin + 4;                                       // [4]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_kmax + 4);
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + L.off_misc + 64);   // [K1C_MAXR]
    uint64_t* bar_mma = bar_full + K1C_MAXR;
    int* s_bmeta = reinterpret_cast<int*>(bar_mma + 1);            // [3] bias: min 2-adic exponent, max |bias| bits, inexact flag

    const int head = blockIdx.x, bb = head / p.H, hh = head - bb * p.H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // selection mapping: warp w owns TMEM lanes [32 (w & 3) + 16 (w >> 2), +16); lanes l and l + 16
    // of the warp share query row l of those and take the lower / upper half of its key columns
    const int lane_base = 32 * (warp & 3) + 16 * (warp >> 2);
    const int rr = lane_base + (lane & 15);                         // row of the tile
    const int part = lane >> 4;
    const bool bf16 = BF < 0 ? (p.bf16 != 0) : (BF != 0), flush = p.flush;
    const bool write_k = CODES && p.k_codes != nullptr && blockIdx.y == 0;
    const bool write_q = CODES && p.q_codes != nullptr;
    const bool write_kop = p.k_op != nullptr && blockIdx.y == 0;
    const OpsLayout OL = ops_layout(Nq, Nk, hd);
    unsigned char* k_op = p.k_op ? p.k_op + (size_t)head * OL.k_head_bytes : nullptr;
    unsigned char* q_op = p.q_op ? p.q_op + (size_t)head * OL.q_head_bytes : nullptr;
    const int kb_rows = OL.kb_rows;
    const float* kbias = biased ? p.key_bias + bb * p.kb_sB : nullptr;

    // ---- step schedule of this CTA: CR = 64 G rows per step; K steps first, then the Q tiles
    const int CR = K1C_ROWS * G, cr_shift = G == 2 ? 7 : 6;
    const int nks = (NMMA + CR - 1) / CR;                           // every MMA row of the K operand is written
    const int qsteps = K1C_TILE / CR;                               // steps per query tile (2 or 1)
    const int tiles = (Nq + K1C_TILE - 1) / K1C_TILE;
    const int my_tiles = (tiles - (int)blockIdx.y + (int)gridDim.y - 1) / (int)gridDim.y;
    const int nsteps = nks + qsteps * my_tiles;
    const uint32_t box_main = (uint32_t)L.box_main, box_tail = (uint32_t)L.box_tail;
    const uint32_t slot_tx = (uint32_t)G * (box_main + box_tail) / (DT == DT_F32 ? 1 : 2);   // 16-bit: half-filled slots
    const uint32_t slot_bytes = (uint32_t)L.slot_bytes;
    const uint32_t tail_base = (uint32_t)G * box_main;

    auto issue = [&](int c, int slot_i) {                           // one thread
        unsigned char* slot = smem + (size_t)slot_i * slot_bytes;
        uint64_t* bar = &bar_full[slot_i];
        const bool is_k = c < nks;
        int row0;
        if (is_k) row0 = c * CR;
        else {
            const int qc = c - nks;
            row0 = ((int)blockIdx.y + (qc / qsteps) * (int)gridDim.y) * K1C_TILE + (qc % qsteps) * CR;
        }
        mbar_expect_tx(bar, slot_tx);
        for (int g = 0; g < G; ++g) {
            if (nfull) tma_load_5d(slot + g * box_main, is_k ? &maps.k_main : &maps.q_main, 0, row0 + g * K1C_ROWS, 0, hh, bb, bar);
            if (tail) tma_load_4d(slot + tail_base + g * box_tail, is_k ? &maps.k_tail : &maps.q_tail, 0, row0 + g * K1C_ROWS, hh, bb, bar);
        }
    };

    if (tid == 0) {
        for (int r = 0; r < ring; ++r) mbar_init(&bar_full[r], 1);
        mbar_init(bar_mma, 1);
        prefetch_tmap(&maps.k_main); prefetch_tmap(&maps.q_main);
        if (tail) { prefetch_tmap(&maps.k_tail); prefetch_tmap(&maps.q_tail); }
    }
    if (tid < 4) { s_kmin[tid] = 0x7fffffff; s_kmax[tid] = -0x7fffffff; }
    if (tid == 4) { s_bmeta[0] = 0x7fffffff; s_bmeta[1] = 0; s_bmeta[2] = 0; }
    if (warp == 0) tmem_alloc(s_tmem, (uint32_t)L.tmem_cols);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    const uint32_t tmem = *s_tmem;
    const uint32_t my_tmem = tmem + ((uint32_t)lane_base << 16);
    if (tid == 0) {
        const int pre = min(ring, nsteps);
        for (int c = 0; c < pre; ++c) issue(c, c);
    }
    const uint32_t idesc = umma_idesc_bf16_f32(128, NMMA);
    const int NW = (Nk + 31) >> 5;
    // padding key columns (index >= Nk, score exactly 0) among THIS thread's chunks [part NCH, part NCH + NCH)
    const int my_cols_end = HG ? (part + 1) * HW : min(NC, (part + 1) * NCH) * 32, my_cols_beg = part * HW;
    const int my_pad = max(0, my_cols_end - max(Nk, my_cols_beg));
    uint32_t ph_mma = 0;
    int slot_i = 0;
    uint32_t slot_par = 0;
    int tile = (int)blockIdx.y - (int)gridDim.y;                    // advanced at the first step of every tile
    int qstep = qsteps - 1;                                         // step within the tile

    for (int c = 0; c < nsteps; ++c) {
        const bool is_k = c < nks;
        if (!is_k) {
            if (++qstep == qsteps) { qstep = 0; tile += (int)gridDim.y; }
        }
        const int row0 = is_k ? c * CR : tile * K1C_TILE + qstep * CR;
        const int nrows = is_k ? Nk : Nq;
        const unsigned char* slot = smem + (size_t)slot_i * slot_bytes;
        mbar_wait(&bar_full[slot_i], slot_par);

        // -------- quantize the step's rows: one thread per MX block, block-major task order
        // (consecutive lanes <-> consecutive rows of one block index: conflict-free reads of the
        //  swizzled boxes, conflict-free / coalesced operand stores)
        const int ntask = CR * nb;
        for (int t = tid; t < ntask; t += K1C_T) {
            const int b = t >> cr_shift, rl = t & (CR - 1);
            const int g = rl >> 6, rl6 = rl & 63;
            const int row = row0 + rl;
            const bool in_range = row < nrows;
            const bool full = b < nfull;
            uint32_t xv[32];
            if constexpr (DT != DT_F32) {
                staged_block_bits_16<DT>(slot, g, box_main, tail_base, box_tail, b, rl6, full, tail, xv);
            } else if (full) {
                const unsigned char* src = slot + g * box_main + (b * 64 + rl6) * 128;
                const int sw7 = (rl6 & 7) << 4;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const uint4 v = *reinterpret_cast<const uint4*>(src + ((s << 4) ^ sw7));
                    xv[4 * s] = v.x; xv[4 * s + 1] = v.y; xv[4 * s + 2] = v.z; xv[4 * s + 3] = v.w;
                }
            } else {
                const unsigned char* src = slot + tail_base + g * box_tail + rl6 * tail * 4;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    uint4 v = make_uint4(0u, 0u, 0u, 0u);
                    if (4 * s < tail) v = *reinterpret_cast<const uint4*>(src + (s << 4));
                    xv[4 * s] = v.x; xv[4 * s + 1] = v.y; xv[4 * s + 2] = v.z; xv[4 * s + 3] = v.w;
                }
            }
            BlockQ r;
            quantize_block_thread<CODES>(xv, full ? 32 : tail, bf16, flush, r);
            const int nchunk = full ? 4 : tail_chunks, nchunk_hbm = full ? 4 : tail_chunks_hbm;
            if (is_k) {
                if (row < NMMA) {
                    unsigned char* dst = s_kop + ((4 * b) * NMMA + row) * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch)
                        if (ch < nchunk)
                            *reinterpret_cast<uint4*>(dst + ch * (NMMA * 16)) =
                                in_range ? r.pp[ch] : make_uint4(0u, 0u, 0u, 0u);
                }
                s_ksign[b * 256 + row] = r.sign;
                s_kexp[b * 256 + row] = (signed char)r.ep;
                {   // b is warp-uniform (>= 64 tasks per block index): one shared-memory atomic per warp
                    const int lo = __reduce_min_sync(FULL, in_range ? r.ep : 0x7fffffff);
                    const int hi = __reduce_max_sync(FULL, in_range ? r.ep : -0x7fffffff);
                    if (lane == 0) { atomicMin(&s_kmin[b], lo); atomicMax(&s_kmax[b], hi); }
                }
                if (write_kop && row < kb_rows) {
                    unsigned char* dst = k_op + ((size_t)(4 * b) * kb_rows + row) * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch)
                        if (ch < nchunk_hbm) *reinterpret_cast<uint4*>(dst + (size_t)ch * kb_rows * 16) = r.op[ch];
                }
                if (CODES && write_k && in_range) {
                    const int64_t krow = (int64_t)head * Nk + row;
                    p.k_exps[krow * nb + b] = (int8_t)r.e;
                    uint32_t* dst = reinterpret_cast<uint32_t*>(p.k_codes + krow * hd + 32 * b);
#pragma unroll
                    for (int v = 0; v < 8; ++v)
                        if (4 * v < (full ? 32 : tail)) dst[v] = r.cw[v];
                }
            } else {
                const int rt = qstep * CR + rl;                     // row within the tile
                unsigned char* dst = s_qop + ((4 * b) * K1C_TILE + rt) * 16;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch)
                    if (ch < nchunk) *reinterpret_cast<uint4*>(dst + ch * (K1C_TILE * 16)) = r.pp[ch];
                s_qsign[b * K1C_TILE + rt] = r.sign;
                s_qexp[b * K1C_TILE + rt] = (signed char)r.ep;
                if (q_op) {
                    unsigned char* gdst = q_op + (size_t)tile * OL.q_tile_bytes + ((size_t)(4 * b) * K1C_TILE + rt) * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch)
                        if (ch < nchunk_hbm) *reinterpret_cast<uint4*>(gdst + ch * (K1C_TILE * 16)) = r.op[ch];
                }
                if (CODES && write_q && in_range) {
                    const int64_t qrow = (int64_t)head * Nq + row;
                    p.q_exps[qrow * nb + b] = (int8_t)r.e;
                    uint32_t* dst2 = reinterpret_cast<uint32_t*>(p.q_codes + qrow * hd + 32 * b);
#pragma unroll
                    for (int v = 0; v < 8; ++v)
                        if (4 * v < (full ? 32 : tail)) dst2[v] = r.cw[v];
                }
            }
        }
        if (biased) {
            // The additive key bias rides through the MMA: two extra K columns hold bias_j split into
            // two bf16 terms (exact when the bias has <= 16 significant bits) on the key side and 1.0 on
            // the query side, so the accumulator is pred + bias_j - exact whenever both are multiples of
            // 2^(g+1) inside the integer window, which is when fl32(pred + bias) is exact as well.
            const int cb = hd >> 3;                                 // first chunk past the data
            for (int t = tid; t < CR; t += K1C_T) {
                const int row = row0 + t;
                if (is_k) {
                    uint32_t w0 = 0u;
                    int ex = 0x7fffffff;
                    uint32_t mag = 0u, inexact = 0u;
                    if (row < nrows) {
                        const float bj = __ldg(kbias + row);
                        const uint32_t bits = __float_as_uint(bj);
                        const uint32_t hi = bits & 0xffff0000u;
                        const uint32_t lo = __float_as_uint(bj - __uint_as_float(hi));     // exact
                        w0 = (hi >> 16) | (lo & 0xffff0000u);
                        inexact = (lo & 0xffffu) ? 1u : 0u;
                        mag = bits & 0x7fffffffu;
                        if (mag) ex = (int)(mag >> 23) - 150 + (__ffs((int)((mag & 0x7fffffu) | 0x800000u)) - 1);
                        if ((mag != 0u && (mag >> 23) == 0u) || (mag >> 23) == 255u) inexact = 1u;   // subnormal / inf / nan: fp32 path
                    }
                    if (row < NMMA) {
                        *reinterpret_cast<uint4*>(s_kop + ((size_t)cb * NMMA + row) * 16) = make_uint4(w0, 0u, 0u, 0u);
                        for (int ch = cb + 1; ch < kch; ++ch)
                            *reinterpret_cast<uint4*>(s_kop + ((size_t)ch * NMMA + row) * 16) = make_uint4(0u, 0u, 0u, 0u);
                    }
                    ex = __reduce_min_sync(FULL, ex);
                    mag = __reduce_max_sync(FULL, mag);
                    inexact = __reduce_or_sync(FULL, inexact);
                    if (lane == 0) { atomicMin(&s_bmeta[0], ex); atomicMax(&s_bmeta[1], (int)mag); atomicOr(&s_bmeta[2], (int)inexact); }
                } else {
                    const int rt = qstep * CR + t;
                    *reinterpret_cast<uint4*>(s_qop + ((size_t)cb * K1C_TILE + rt) * 16) = make_uint4(0x3F803F80u, 0u, 0u, 0u);
                    for (int ch = cb + 1; ch < kch; ++ch)
                        *reinterpret_cast<uint4*>(s_qop + ((size_t)ch * K1C_TILE + rt) * 16) = make_uint4(0u, 0u, 0u, 0u);
                }
            }
        }
        fence_proxy_async_smem();                                   // operand stores -> visible to the MMA
        __syncthreads();                                            // slot consumed; operands complete
        if (tid == 0 && c + ring < nsteps) issue(c + ring, slot_i);
        if (++slot_i == ring) { slot_i = 0; slot_par ^= 1u; }
        if (is_k || qstep != qsteps - 1) continue;

        // =============== a full query tile is quantized: score, select, emit
        if (kk >= Nk) {
            // dense attention (the reference's top_k=False blocks, e.g. DeiT block 11 / DiT block 27:
            // workloads/deit/scripts/main.py:282-296): every key is kept, nothing to score or select
            const int i = tile * K1C_TILE + rr;
            if (i < Nq) {
                const int64_t row = (int64_t)head * Nq + i;
                for (int w = part; w < NW; w += 2) {
                    const int nv = Nk - 32 * w;
                    p.mask[row * NW + w] = nv >= 32 ? 0xffffffffu : (1u << nv) - 1u;
                }
                if (p.idx && part == 0)
                    for (int j = 0; j < Nk; ++j) p.idx[row * kk + j] = j;
            }
            continue;
        }
        if (tid == 0) {
            tcgen05_fence_after_sync();
            for (int ks = 0; ks < (L.hdp >> 4); ++ks) {
                const uint64_t da = umma_smem_desc(smem_u32(s_qop + (size_t)(2 * ks) * K1C_TILE * 16), K1C_TILE * 16, 128);
                const uint64_t db = umma_smem_desc(smem_u32(s_kop + (size_t)(2 * ks) * NMMA * 16), NMMA * 16, 128);
                umma_bf16_ss(tmem, da, db, idesc, ks > 0);
            }
            umma_commit(bar_mma);
        }
        // ---- integer-key parameters of this thread's row (same window rules as mxprune_predict.cuh)
        const int i = tile * K1C_TILE + rr;
        const bool valid = i < Nq;
        const int64_t row = (int64_t)head * Nq + (valid ? i : 0);
        int kmin[4], spread[4], epq[4];
        uint32_t sq[4];
        bool wide = false;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            kmin[b] = b < nb ? s_kmin[b] : 0;
            spread[b] = b < nb ? s_kmax[b] - kmin[b] : 0;
            wide |= spread[b] > K1_MAX_SPREAD;
            epq[b] = b < nb ? (int)s_qexp[b * K1C_TILE + rr] : 0;
            sq[b] = b < nb ? s_qsign[b * K1C_TILE + rr] : 0u;
        }
        int g = 0x7fffffff;
#pragma unroll
        for (int b = 0; b < 4; ++b)
            if (b < nb) g = min(g, epq[b] + kmin[b]);
        bool fast = valid && !wide && g >= -100 && g <= 80;
        long long M = 0;
        if (biased) {
            // integer keys carry the bias when every bias_j is an even multiple of 2^g (then pred + bias
            // is exact in fp32, as the reference adds it); its magnitude widens the key window
            if (s_bmeta[2] != 0 || g + 1 > s_bmeta[0]) fast = false;
            const float bm = __uint_as_float((uint32_t)s_bmeta[1]) * (fast ? exp2i(-g) : 0.f);
            if (bm > 40000.f) fast = false; else M = (long long)bm;
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            if (b < nb) {
                int sh = epq[b] + kmin[b] - g;
                if (sh > K1_MAX_SPREAD) { fast = false; sh = K1_MAX_SPREAD; }
                const int nbw = min(32, hd - 32 * b);
                M += (long long)nbw << (sh + min(spread[b], K1_MAX_SPREAD));
            }
        }
        if (M > K1_MAX_M) fast = false;
        if (!fast) M = 0;
        const int moff = ((int)M + 1) & ~1;
        const float scl = fast ? exp2i(-g - 1) : 0.f;
        const uint32_t key0 = (uint32_t)((moff >> 1) + 1) + K1_KEY_BIAS;    // key of a score of exactly 0
        const float cadd = 8388608.0f + (float)key0;

        mbar_wait(bar_mma, ph_mma);
        ph_mma ^= 1u;
        tcgen05_fence_after_sync();

        // ---- scores -> fp16-pattern keys in registers.  This thread's chunk w is key columns
        // [32 (part NCH + w), +32); word 16w + t = keys (base + t, base + 16 + t).  Padding columns
        // (key index >= Nk) score exactly 0 -> key0; they are discounted below.  A chunk past NC
        // (odd NC, upper half) holds zeros, which no candidate reaches.
        uint32_t kw[NWORDS];
#pragma unroll
        for (int w = 0; w < NPAIR; ++w) {
            // chunk index part * NCH + w < NC (always, with the tight split)
            const bool real = HG != 0 || (w < NCH - 1) || (NC % 2 == 0) || part == 0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t r[16];
                tmem_ld_16x32bx2_x16<HW>(my_tmem + w * 32 + h * 16, r);
                tmem_ld_wait();
                // r[t] = key column 16h + t of the chunk: low halves come from h = 0, high halves from h = 1
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const uint32_t f = __float_as_uint(fmaf(__uint_as_float(r[t]), scl, cadd));
                    if (h == 0) kw[16 * w + t] = f;
                    else kw[16 * w + t] = real ? __byte_perm(kw[16 * w + t], f, 0x5410) : 0u;
                }
            }
        }
        if constexpr (REM == 16) {                                  // word 16 NPAIR + t = keys (base + t, base + 8 + t)
            uint32_t r[16];
            tmem_ld_16x32bx2_x16<HW>(my_tmem + NPAIR * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int t = 0; t < 8; ++t)
                kw[16 * NPAIR + t] = __byte_perm(__float_as_uint(fmaf(__uint_as_float(r[t]), scl, cadd)),
                                                 __float_as_uint(fmaf(__uint_as_float(r[t + 8]), scl, cadd)), 0x5410);
        }
        if constexpr (REM == 8) {                                   // word 16 NPAIR + t = keys (base + t, base + 4 + t)
            uint32_t r[8];
            tmem_ld_16x32bx2_x8<HW>(my_tmem + NPAIR * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int t = 0; t < 4; ++t)
                kw[16 * NPAIR + t] = __byte_perm(__float_as_uint(fmaf(__uint_as_float(r[t]), scl, cadd)),
                                                 __float_as_uint(fmaf(__uint_as_float(r[t + 4]), scl, cadd)), 0x5410);
        }
        // every thread has its row parameters and its keys in registers: TMEM and the Q-side shared
        // memory may be reused by the next tile from here on (warps run the selection unsynchronised)
        tcgen05_fence_before_sync();
        __syncthreads();

        // ---- select: T = top_k-th largest key; the row's two lanes add their counts
        int nge_m, nge_o, ngt_m, ngt_o;
        const int nvalid_m = min(my_cols_end, max(Nk, my_cols_beg)) - my_cols_beg;
        const uint32_t T = select_kth_key<NWORDS, (HG == 0 && (NC & 1))>(kw, key0, my_pad, kk, nvalid_m, Nk - nvalid_m,
                                                                       nge_m, nge_o, ngt_m, ngt_o);

        // ---- emit the row bitmask (ties: ascending key index; the lower lane owns the lower columns)
        {
            const int rem_all = kk - (ngt_m + ngt_o);               // ties to keep in the whole row
            const int ties0 = part == 0 ? nge_m - ngt_m : nge_o - ngt_o;
            const int ngt0 = part == 0 ? ngt_m : ngt_o;
            int rem = part == 0 ? rem_all : rem_all - min(rem_all, ties0);
            int pos = part == 0 ? 0 : ngt0 + min(rem_all, ties0);   // kept keys below this thread's columns
            const __half2 t2 = u32_as_h2(T * 0x00010001u);
            const bool store = valid && fast;
            uint32_t lw[NLW];                                       // tight split: this lane's words, lane-local bit order
#pragma unroll
            for (int w = 0; w < NLW; ++w) {
                uint32_t gt = 0u, eq = 0u;                          // lane-local bit i <-> key column my_cols_beg + 32 w + i
                if (w < NPAIR) {
#pragma unroll
                    for (int t = 0; t < 16; ++t) {
                        const __half2 kv = u32_as_h2(kw[16 * w + t]);
                        gt |= __hgt2_mask(kv, t2) & (0x00010001u << t);
                        eq |= __heq2_mask(kv, t2) & (0x00010001u << t);
                    }
                } else if constexpr (REM != 0) {                    // the rest: REM / 2 words of keys (t, REM / 2 + t)
#pragma unroll
                    for (int t = 0; t < REM / 2; ++t) {
                        const __half2 kv = u32_as_h2(kw[16 * NPAIR + t]);
                        gt |= __hgt2_mask(kv, t2) & (0x00010001u << t);
                        eq |= __heq2_mask(kv, t2) & (0x00010001u << t);
                    }
                    // high halves sit at bit 16 + t: move them down to bit REM / 2 + t
                    gt = (gt & 0xffffu) | ((gt >> 16) << (REM / 2));
                    eq = (eq & 0xffffu) | ((eq >> 16) << (REM / 2));
                }
                const int nv = Nk - (my_cols_beg + 32 * w);         // valid key columns in this word
                const uint32_t vm = nv >= 32 ? 0xffffffffu : (nv <= 0 ? 0u : (1u << nv) - 1u);
                gt &= vm;
                eq &= vm;
                const int cnt = __popc(eq);
                uint32_t take = eq;
                if (cnt > rem) take = keep_lowest_bits_fast(eq, rem);
                rem -= min(cnt, rem);
                const uint32_t word = gt | take;
                if (HG == 0) {
                    const int gw = part * NCH + w;
                    if (store && gw < NW) p.mask[row * NW + gw] = word;
                } else {
                    lw[w] = word;
                }
                if (store && p.idx) {
                    uint32_t w2 = word;
                    while (w2) {
                        const int bpos = __ffs(w2) - 1;
                        w2 &= w2 - 1u;
                        p.idx[row * kk + pos++] = my_cols_beg + 32 * w + bpos;
                    }
                }
            }
            if constexpr (HG != 0) {
                // tight split: the upper lane's bits start REM bits into global word NPAIR.  The lower lane stores
                // words 0 .. NPAIR (the shared word completed with the partner's first bits), the upper lane the
                // funnel-shifted rest - aligned 32-bit stores, 16 consecutive rows per instruction
                const uint32_t other0 = __shfl_xor_sync(FULL, lw[0], 16);
                if (store) {
                    uint32_t* mrow = p.mask + row * NW;
                    if (part == 0) {
#pragma unroll
                        for (int w = 0; w < NPAIR; ++w) mrow[w] = lw[w];
                        mrow[NPAIR] = lw[NPAIR] | (other0 << REM);
                    } else {
#pragma unroll
                        for (int w = 0; w < NPAIR; ++w)
                            if (NPAIR + 1 + w < NW) mrow[NPAIR + 1 + w] = __funnelshift_l(lw[w], lw[w + 1], REM);
                    }
                }
            }
        }

        // ---- rows outside the integer-key window: warp-cooperative generic path (16 rows per warp)
        unsigned todo = __ballot_sync(FULL, valid && !fast) & 0xffffu;
        while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1u;
            uint32_t gsq[4];
            int gep[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                gsq[b] = __shfl_sync(FULL, sq[b], l);
                gep[b] = __shfl_sync(FULL, epq[b], l);
            }
            const int64_t grow = (int64_t)head * Nq + (tile * K1C_TILE + lane_base + l);
            predict_row_generic_tc(p.mask, p.idx, Nk, kk, hd, nb, grow, gsq, gep, s_ksign, s_kexp, kbias);
        }
    }
    tcgen05_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, (uint32_t)L.tmem_cols);
}

// ---- K1-TC launch: which instantiation serves a call (host side; maps, layout L, dyn and grid set by the caller) ----
template <int NC, bool CODES, bool BIASED, int HG = 0, int HD = 0, int BF = -1, int DT = DT_F32>
static int launch_predict_topk_tc_one(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn,
                                      dim3 grid, cudaStream_t st) {
    MXP_ENSURE_DYN_SMEM((k_predict_topk_tc<NC, CODES, BIASED, HG, HD, BF, DT>), 227 * 1024);
    k_predict_topk_tc<NC, CODES, BIASED, HG, HD, BF, DT><<<grid, K1C_T, dyn, st>>>(p, maps, L.ring, L.G);
    return check_launch("k_predict_topk_tc");
}
// the workload head shapes get instantiations with head_dim and the A1 switch folded at compile time
template <int NC, int HG, int HD, int DT>
static int launch_predict_topk_tc_hd(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn,
                                     dim3 grid, cudaStream_t st) {
    return p.bf16 ? launch_predict_topk_tc_one<NC, false, false, HG, HD, 1, DT>(p, maps, L, dyn, grid, st)
                  : launch_predict_topk_tc_one<NC, false, false, HG, HD, 0, DT>(p, maps, L, dyn, grid, st);
}
// nc = key chunks; q / k of element type DT (== p.dt).  Key bias and code outputs are never requested together.
template <int DT>
static int launch_predict_topk_tc_dt(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn, dim3 grid,
                                     int nc, cudaStream_t st) {
    const bool biased = p.key_bias != nullptr, codes = p.q_codes != nullptr || p.k_codes != nullptr;
#define MXP_TC(NC_)                                                                                        \
    return biased ? launch_predict_topk_tc_one<NC_, false, true, 0, 0, -1, DT>(p, maps, L, dyn, grid, st)     \
         : codes  ? launch_predict_topk_tc_one<NC_, true, false, 0, 0, -1, DT>(p, maps, L, dyn, grid, st)     \
                  : launch_predict_topk_tc_one<NC_, false, false, 0, 0, -1, DT>(p, maps, L, dyn, grid, st)
    switch (nc) {
        case 1: MXP_TC(1);
        case 2: MXP_TC(2);
        case 4: MXP_TC(4);
        case 7:
            // 193 .. 224 keys: the two lanes of a row split the columns at 104 / 112 instead of 128 (no dummy chunk)
            if (!biased && !codes && p.Nk > 192 && p.Nk <= 208 && p.hd == 64)       // DeiT / ViT-224 heads
                return launch_predict_topk_tc_hd<7, 13, 64, DT>(p, maps, L, dyn, grid, st);
            if (!biased && !codes && p.Nk > 192 && p.Nk <= 208)
                return launch_predict_topk_tc_one<7, false, false, 13, 0, -1, DT>(p, maps, L, dyn, grid, st);
            if (!biased && !codes && p.Nk > 208)
                return launch_predict_topk_tc_one<7, false, false, 14, 0, -1, DT>(p, maps, L, dyn, grid, st);
            MXP_TC(7);
        default:
            if (!biased && !codes && p.hd == 72)                                      // DiT / PixArt heads
                return launch_predict_topk_tc_hd<8, 0, 72, DT>(p, maps, L, dyn, grid, st);
            MXP_TC(8);
    }
#undef MXP_TC
}

// launch_predict_topk_tc_dt for 16-bit q / k (p.dt), compiled in mxprune_predict16.cu
int launch_predict_topk_tc_16(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn, dim3 grid, int nc,
                              cudaStream_t st);

}  // namespace mxp
