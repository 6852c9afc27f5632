// K2: exact MXINT8 attention over the kept keys on the Blackwell tensor cores - the MMA-ready operand layout every
// exact-attention kernel reads, and the one-key-block kernel k_attend_pair (Nk <= 256).
//
// Key fact: every MXINT8 value c * 2^(e-6) (|c| <= 127) is EXACTLY representable in bf16 (8
// significant bits, fp32 exponent range).  So both contractions of the reference,
//     true_scores = mx.matmul(q, k^T)            microxscaling/mx/matmul.py:68-88
//     x           = mx.matmul(attn, v)           workloads/deit/scripts/main.py:152
// are products of exact bf16 operands accumulated in fp32 - which is precisely
// tcgen05.mma kind::f16 with bf16 inputs and fp32 accumulators in tensor memory.  No product is
// altered; only the fp32 summation order differs from MKL's (as between any two BLAS).
//
// Operands arrive "MMA-ready" in HBM (OpsLayout below): K1 writes the dequantised Q and K as bf16
// in the exact shared-memory image the MMA wants (K-major, no swizzle, 16-byte chunks of 8
// consecutive K elements; chunk (row r, k-chunk c) at c*(ROWS*16) + r*16  =>  SBO = 128 B,
// LBO = ROWS*16 B), k_prep_v does the same for V^T after quantising V along TOKENS
// (matmul.py:76-83).  K2 therefore stages with TMA bulk copies (cp.async.bulk + mbarrier
// complete_tx) and spends its instructions on the softmax / P-quantisation epilogue only.
//
// Nk <= 256 (k_attend_pair): one key block, the head's K and V operands resident in shared memory.  Per query tile
// S = Q.K^T (hd/16 MMAs, N = Nk) -> TMEM; pass A max over the kept keys; pass B E = exp(t - max) (0 where pruned)
// written back over S, row sum; pass C P = E/sum -> A1 -> MXINT8 per 32-key window -> bf16 A operand, O += P_w.V_w
// (O reuses the TMEM columns of windows already consumed).  k_attend_sparse (mxprune_attend_sparse.cuh) runs the same
// stages on compacted row lists when top_k is small; Nk > 256 streams key blocks of 128 through k_attend_long_pair
// (mxprune_attend_long.cuh).
#pragma once
#include "mxprune_device.cuh"
#include "mxprune_umma.cuh"

namespace mxp {

constexpr int K2T = 128;
constexpr int K2_P_BYTES = 4 * 4 * K2T * 16;       // P operand of one MMA group of four 32-key windows: 32 KiB
constexpr int K2_SINGLE_MAX = 256;                 // largest Nk handled as one key block

struct AttnParams {
    const unsigned char *q_op, *k_op, *v_op;       // MMA-ready bf16 operands (OpsLayout)
    const uint32_t* mask;
    int B, H, Nq, Nk, hd;
    float scale;
    int bf16, flush;
    float* out;                 // element type out_dt
    int64_t o_sB, o_sH, o_sN;
    int out_dt;                 // DT_* (host side: selects the kernel instantiation)
    const float* key_bias;      // optional additive bias per (batch, key), added to score * scale (fp32)
    int64_t kb_sB;
};

// Layout of the MMA-ready operand buffers of one head (all sizes in bytes).
struct OpsLayout {
    int hdp, nw, single, kb_rows, nblk, wpb, q_tiles;
    size_t q_tile_bytes, k_blk_bytes, v_blk_bytes, q_head_bytes, k_head_bytes, v_head_bytes;
};

__host__ __device__ inline OpsLayout ops_layout(int Nq, int Nk, int hd) {
    OpsLayout L;
    L.hdp = (hd + 15) & ~15;
    L.nw = (Nk + 31) >> 5;
    L.single = Nk <= K2_SINGLE_MAX;
    L.kb_rows = L.single ? ((Nk + 15) & ~15) : 128;            // key rows per block (MMA N)
    L.nblk = L.single ? 1 : (Nk + 127) / 128;
    L.wpb = L.single ? L.nw : 4;                                // 32-key windows per block
    L.q_tiles = (Nq + K2T - 1) / K2T;
    L.q_tile_bytes = (size_t)(L.hdp / 8) * K2T * 16;
    L.k_blk_bytes = (size_t)(L.hdp / 8) * L.kb_rows * 16;
    L.v_blk_bytes = (size_t)(L.wpb * 4) * L.hdp * 16;
    L.q_head_bytes = L.q_tile_bytes * L.q_tiles;
    L.k_head_bytes = L.k_blk_bytes * L.nblk;
    L.v_head_bytes = L.v_blk_bytes * L.nblk;
    return L;
}
// byte offset (within a head) of the 16-byte chunk holding dims [8kc, 8kc+8) of query row i
__host__ __device__ inline size_t q_op_offset(const OpsLayout& L, int i, int kc) {
    return (size_t)(i / K2T) * L.q_tile_bytes + ((size_t)kc * K2T + (i % K2T)) * 16;
}
// ... of key row j
__host__ __device__ inline size_t k_op_offset(const OpsLayout& L, int j, int kc) {
    const int blk = L.single ? 0 : j / 128, jl = L.single ? j : j % 128;
    return (size_t)blk * L.k_blk_bytes + ((size_t)kc * L.kb_rows + jl) * 16;
}
// ... holding tokens [8tc, 8tc+8) of V column d
__host__ __device__ inline size_t v_op_offset(const OpsLayout& L, int tc, int d) {
    const int blk = L.single ? 0 : tc / 16, tl = L.single ? tc : tc % 16;
    return (size_t)blk * L.v_blk_bytes + ((size_t)tl * L.hdp + d) * 16;
}

// shared memory of the one-key-block kernels: the head's K and V operands, then the P window group
struct K2Smem {
    size_t off_v, off_p, total;
};
__host__ __device__ inline K2Smem k2_smem_layout(const OpsLayout& O) {
    K2Smem L;
    size_t o = O.k_blk_bytes;
    L.off_v = o; o += O.v_blk_bytes;
    L.off_p = o; o += K2_P_BYTES;                    // P window group; also the Q tile (<= 32 KiB)
    L.total = o;
    return L;
}

// ---- TMA bulk copy global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ------------------------------------------------------------------------------------------
// k_attend_pair: the single-key-block case (Nk <= 256) with TWO LANES PER QUERY ROW.
// 256 threads per CTA, 16 warps per SM.  A warp owns 16 query rows (TMEM lanes); lanes l and l + 16
// share row l.  Key windows (32 keys) are dealt in pairs: lane half h takes windows 4g + 2h and
// 4g + 2h + 1 of every group g of four - tcgen05.ld/st.16x32bx2 with a column split of 64 reads and
// writes exactly that.  Row maximum and row sum are combined with one SHFL each; every other step of
// the epilogue is per window and needs no exchange.  The next window's tcgen05.ld is in flight
// while the current one is processed.
// ------------------------------------------------------------------------------------------
constexpr int K2P_T = 256;

__device__ __forceinline__ void tmem_ld_16x32bx2_s64_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x32bx2.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32], 64;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_st_16x32bx2_s64_x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.16x32bx2.x32.b32 [%0], 64, {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

// TMEM columns the pair kernel allocates: the S tile plus whatever the 64-column split reads past it
__host__ __device__ inline int k2p_tmem_cols(const OpsLayout& O) {
    const int need = 128 * ((O.nw + 3) / 4);
    int c = 32;
    while (c < need || c < O.hdp) c <<= 1;
    return c;
}

// A 256-thread group of a CTA: its thread index, named barrier, shared-memory window, mbarriers, TMEM columns.
// The exact-attention bodies below are GROUP functions: the stand-alone kernels run them as a whole CTA (barrier 0),
// the fused kernel (mxprune_fused.cuh) as one of the two groups of a CTA.
struct GroupCtx {
    int tid;                            // 0..255 within the group
    int bar_id;                         // named barrier of the group (0 when the group is the whole CTA)
    unsigned char* smem;                // 1024-byte aligned window of the dynamic shared memory
    uint64_t* bar_ld;                   // mbarriers (count 1), initialised by the caller; phases below
    uint64_t* bar_s;
    uint64_t* bar_o;
    uint32_t tmem;                      // base of the group's TMEM columns
    uint32_t ph_ld, ph_s, ph_o;
    unsigned long long* prof;           // debug: per-phase cycle accumulators of the group's thread 0 (null = off)
    long long t_last;
};
// debug phase accounting (mxp_debug_fused_timing): thread 0 of the group adds the cycles since its last mark to slot i
#ifdef MXP_FUSED_TIMING
#define MXP_PROF(gc, i)                                                     \
    do {                                                                    \
        if ((gc).prof != nullptr && (gc).tid == 0) {                        \
            const long long now_ = clock64();                               \
            (gc).prof[i] += (unsigned long long)(now_ - (gc).t_last);       \
            (gc).t_last = now_;                                             \
        }                                                                   \
        __syncwarp(); /* tcgen05 .sync.aligned instructions need the warp converged again */ \
    } while (0)
#else
#define MXP_PROF(gc, i) do { } while (0)
#endif
__device__ __forceinline__ void group_sync(const GroupCtx& g) {
    asm volatile("bar.sync %0, 256;" ::"r"(g.bar_id) : "memory");
}

// O tile (TMEM lanes = query rows of the tile, columns [0, hdp)) -> A1 -> global memory.  Warp w reads the TMEM lanes of
// quarter w & 3 and the column half w >> 2; 32 x 32 blocks are transposed through the warp's private 4 KiB of shared
// memory (stage_base + 4096 w; conflict-free 16-byte chunks, chunk q of row l at position q ^ (l & 7)) so that 8 lanes
// store 128 contiguous bytes of one output row: 4 full lines per store instruction instead of 32 partial ones.
// OT (DT_*): a 16-bit output type the tile may be stored in - when out16, the fp32 values are rounded to nearest even at
// the store (64 contiguous bytes per 8 lanes); OT = DT_F32 stores fp32 only.
template <bool BF16, int OT = DT_F32>
__device__ __forceinline__ void store_o_tile(uint32_t tmem, unsigned char* stage_base, int warp, int lane, int tile,
                                             int Nq, int hd, int hdp, float* out_head, int64_t o_sN, bool out16 = false) {
    const int half_cols = hdp >> 1;                                 // multiple of 8
    const uint32_t ot = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    unsigned char* const stg = stage_base + warp * 4096;
    const int row0 = tile * K2T + 32 * (warp & 3);
    const int cbeg = (warp >> 2) * half_cols, cend = cbeg + half_cols;
    for (int c0 = cbeg; c0 < cend; c0 += 32) {
        const int nc = min(32, cend - c0);                          // columns of this block (multiple of 8)
#pragma unroll
        for (int h = 0; h < 4; ++h) {                               // 8 columns at a time: few live registers
            if (8 * h < nc) {
                uint32_t r[8];
                tmem_ld_32x32b_x8(ot + c0 + 8 * h, r);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    uint4 v = make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
                    if (BF16) { v.x = bf16_half_away(v.x); v.y = bf16_half_away(v.y); v.z = bf16_half_away(v.z); v.w = bf16_half_away(v.w); }
                    *reinterpret_cast<uint4*>(stg + lane * 128 + (((2 * h + q) ^ (lane & 7)) << 4)) = v;
                }
            }
        }
        __syncwarp();
        const int ch = lane & 7;
        const int col = c0 + 4 * ch;
        if (4 * ch < nc && col < hd) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int rl = (lane >> 3) + 4 * it;
                const uint4 v = *reinterpret_cast<const uint4*>(stg + rl * 128 + ((ch ^ (rl & 7)) << 4));
                if (row0 + rl < Nq) {
                    if (OT != DT_F32 && out16) store_out4<OT>(out_head, (int64_t)(row0 + rl) * o_sN + col, v);
                    else store_out4<DT_F32>(out_head, (int64_t)(row0 + rl) * o_sN + col, v);
                }
            }
        }
        __syncwarp();
    }
}

// One head (query tiles tile_begin, tile_begin + tile_step, ...) through the dense-epilogue exact attention.
// q_op / k_op / v_op: this head's MMA-ready operands; mask_head: its [Nq][NW] mask words; out_head: its output rows;
// bias_b: the batch's additive key bias (BIAS only); s_bias: 256 floats of shared memory (BIAS only).
// OT / out16: output type (store_o_tile)
template <bool BF16, bool BIAS, int OT = DT_F32>
__device__ __forceinline__ void attend_pair_head(GroupCtx& gc, const OpsLayout& O, int Nq, int Nk, int hd, float scale,
                                                 bool flush, const unsigned char* q_op, const unsigned char* k_op,
                                                 const unsigned char* v_op, const uint32_t* mask_head, float* out_head,
                                                 int64_t o_sN, const float* bias_b, float* s_bias, int tile_begin,
                                                 int tile_step, bool out16 = false) {
    constexpr bool bf16 = BF16;
    const K2Smem L = k2_smem_layout(O);
    const int hdp = O.hdp, NW = O.nw, kbr = O.kb_rows;
    const int NG = (NW + 3) >> 2;                                   // groups of four windows
    unsigned char* const smem = gc.smem;
    unsigned char* sK = smem;
    unsigned char* sV = smem + L.off_v;
    unsigned char* sP = smem + L.off_p;
    const int tid = gc.tid, warp = tid >> 5, lane = tid & 31;
    const int lane_base = 32 * (warp & 3) + 16 * (warp >> 2);
    const int rr = lane_base + (lane & 15);                         // row of the tile
    const int part = lane >> 4;                                     // which window pair of each group
    uint64_t& bar_ld = *gc.bar_ld;
    uint64_t& bar_s = *gc.bar_s;
    uint64_t& bar_o = *gc.bar_o;
    uint32_t& ph_ld = gc.ph_ld;
    uint32_t& ph_s = gc.ph_s;
    uint32_t& ph_o = gc.ph_o;
    if (BIAS) {
        s_bias[tid] = tid < Nk ? __ldg(bias_b + tid) : 0.f;
        group_sync(gc);
    }
    const uint32_t tmem = gc.tmem;
    const uint32_t my_tmem = tmem + ((uint32_t)lane_base << 16);
    const uint32_t idesc_s = umma_idesc_bf16_f32(128, kbr);
    const uint32_t idesc_o = umma_idesc_bf16_f32(128, hdp);

    if (tid == 0) {                                                 // the head's K and V operands stay resident
        mbar_expect_tx(&bar_ld, (uint32_t)(O.k_blk_bytes + O.v_blk_bytes));
        tma_bulk_g2s(sK, k_op, (uint32_t)O.k_blk_bytes, &bar_ld);
        tma_bulk_g2s(sV, v_op, (uint32_t)O.v_blk_bytes, &bar_ld);
    }
    mbar_wait(&bar_ld, ph_ld);
    ph_ld ^= 1u;

    for (int tile = tile_begin; tile < O.q_tiles; tile += tile_step) {
        const int i = tile * K2T + rr;
        const bool valid = i < Nq;
        const uint32_t* mrow = mask_head + (size_t)(valid ? i : 0) * NW;

        if (tid == 0) {                                             // Q tile (A operand) -> the P buffer region
            mbar_expect_tx(&bar_ld, (uint32_t)O.q_tile_bytes);
            tma_bulk_g2s(sP, q_op + (size_t)tile * O.q_tile_bytes, (uint32_t)O.q_tile_bytes, &bar_ld);
        }
        // this lane's windows: 4g + 2 part + j, g < 2, j < 2  ->  mask words mw[2g + j]
        uint32_t mw[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int w = 4 * (t >> 1) + 2 * part + (t & 1);
            mw[t] = (valid && w < NW) ? mrow[w] : 0u;
        }
        mbar_wait(&bar_ld, ph_ld);
        ph_ld ^= 1u;
        if (tid == 0) {
            tcgen05_fence_after_sync();
            for (int ks = 0; ks < (hdp >> 4); ++ks) {
                const uint64_t da = umma_smem_desc(smem_u32(sP + (size_t)(2 * ks) * K2T * 16), K2T * 16, 128);
                const uint64_t db = umma_smem_desc(smem_u32(sK + (size_t)(2 * ks) * kbr * 16), kbr * 16, 128);
                umma_bf16_ss(tmem, da, db, idesc_s, ks > 0);
            }
            umma_commit(&bar_s);
        }
        mbar_wait(&bar_s, ph_s);
        ph_s ^= 1u;
        tcgen05_fence_after_sync();
        const int nwin = 2 * NG;                                    // window slots per lane (some may be empty)

        // ---- pass A: row max of bf16?(s) * scale over the kept keys
        float mb4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        {
            uint32_t ra[32], rb[32];
            tmem_ld_16x32bx2_s64_x32(my_tmem, ra);
#pragma unroll 1
            for (int t = 0; t < nwin; t += 2) {
                tmem_ld_wait();
                tmem_ld_16x32bx2_s64_x32(my_tmem + 128 * (t >> 1) + 32, rb);
                {
                    const uint32_t m0 = mw[t & 3];
                    const int kb0 = 128 * (t >> 1) + 64 * part;     // key index of column c
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        float s = __uint_as_float(ra[c]);
                        if (bf16) s = bf16_half_away(s);
                        float tv = __fmul_rn(s, scale);
                        if (BIAS) tv = __fadd_rn(tv, s_bias[kb0 + c]);
                        mb4[c & 3] = fmaxf(mb4[c & 3], ((m0 >> c) & 1u) ? tv : -INFINITY);
                        ra[c] = __float_as_uint(tv);
                    }
                    tmem_st_16x32bx2_s64_x32(my_tmem + 128 * (t >> 1), ra);     // pass B reads t, not s
                }
                tmem_ld_wait();
                if (t + 2 < nwin) tmem_ld_16x32bx2_s64_x32(my_tmem + 128 * ((t >> 1) + 1), ra);
                {
                    const uint32_t m1 = mw[(t + 1) & 3];
                    const int kb1 = 128 * (t >> 1) + 32 + 64 * part;
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        float s = __uint_as_float(rb[c]);
                        if (bf16) s = bf16_half_away(s);
                        float tv = __fmul_rn(s, scale);
                        if (BIAS) tv = __fadd_rn(tv, s_bias[kb1 + c]);
                        mb4[c & 3] = fmaxf(mb4[c & 3], ((m1 >> c) & 1u) ? tv : -INFINITY);
                        rb[c] = __float_as_uint(tv);
                    }
                    tmem_st_16x32bx2_s64_x32(my_tmem + 128 * (t >> 1) + 32, rb);
                }
            }
        }
        tmem_st_wait();
        float m = fmaxf(fmaxf(mb4[0], mb4[1]), fmaxf(mb4[2], mb4[3]));
        m = fmaxf(m, __shfl_xor_sync(FULL, m, 16));
        const float m_use = (m == -INFINITY) ? 0.f : m;             // no kept key

        // ---- pass B: E = exp(t - m) on kept keys (0 where pruned), written back over S; row sum
        float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
        for (int t = 0; t < nwin; ++t) {
            const uint32_t mwt = mw[t & 3];
            const uint32_t col = 128 * (t >> 1) + 32 * (t & 1);
            uint32_t r[32];
            tmem_ld_16x32bx2_s64_x32(my_tmem + col, r);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const float tv = __uint_as_float(r[c]);             // bf16?(s) * scale (+ bias), from pass A
                const float ex = exp_nonpos(__fsub_rn(tv, m_use));
                const float ev = ((mwt >> c) & 1u) ? ex : 0.f;
                sum4[c & 3] += ev;
                r[c] = __float_as_uint(ev);
            }
            tmem_st_16x32bx2_s64_x32(my_tmem + col, r);
        }
        tmem_st_wait();
        float l = (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
        l += __shfl_xor_sync(FULL, l, 16);
        const float inv = l > 0.f ? 1.0f / l : 0.f;

        // ---- pass C: P = E/sum -> A1 -> MXINT8 per window -> bf16 A operand; O += P_w . V_w per group
        bool first_mma = true;
        for (int g = 0; g < NG; ++g) {
            if (g > 0) {                                            // previous group's MMAs have finished reading sP
                mbar_wait(&bar_o, ph_o);
                ph_o ^= 1u;
            }
#pragma unroll 1
            for (int j = 0; j < 2; ++j) {
                const int wl = 2 * part + j;                        // window slot within the group
                uint32_t r[32];
                tmem_ld_16x32bx2_s64_x32(my_tmem + 128 * g + 32 * j, r);
                tmem_ld_wait();
                uint32_t mx4[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int c = 0; c < 32; ++c) {
                    uint32_t pb = __float_as_uint(__uint_as_float(r[c]) * inv);
                    if (bf16) pb = bf16_half_away(pb);
                    r[c] = pb;
                }
#pragma unroll
                for (int c = 0; c < 32; c += 8) {                   // p >= 0: bit patterns order like the values;
#pragma unroll
                    for (int q = 0; q < 4; ++q)                     // three-input max: one VIMNMX3 per two elements
                        mx4[q] = __vimax3_u32(mx4[q], r[c + 2 * q], r[c + 2 * q + 1]);
                }
                const uint32_t mx = max(max(mx4[0], mx4[1]), max(mx4[2], mx4[3]));
                const int e = mx_shared_exp(mx);
                const bool dead = (flush && e <= -127) || mx == 0u;
                unsigned char* pdst = sP + ((size_t)(wl * 4) * K2T + rr) * 16;
                if (dead || e >= -120) {
                    // code = min(127, floor(p * 2^(6-e) + 0.5)) without F2I / I2F (see K1); a dead
                    // window (no kept key / flushed) runs the same code with scale 0: code 0
                    const int ec = max(e, -120);
                    const float s1 = dead ? 0.f : exp2i(6 - ec);
                    const __nv_bfloat162 w2 = u32_as_bf2(bf16_pow2_bits(ec - 6) * 0x00010001u);
                    const __nv_bfloat162 nw2 = u32_as_bf2((bf16_pow2_bits(ec + 1) | 0x8000u) * 0x00010001u);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        uint32_t ow[4];
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            const float v0 = fminf(fmaf(__uint_as_float(r[q * 8 + 2 * h]), s1, 0.5f), 127.0f);
                            const float v1 = fminf(fmaf(__uint_as_float(r[q * 8 + 2 * h + 1]), s1, 0.5f), 127.0f);
                            const uint32_t v2 = __byte_perm(__float_as_uint(__fadd_rd(v0, 8405760.0f)),
                                                            __float_as_uint(__fadd_rd(v1, 8405760.0f)), 0x5410);
                            ow[h] = bf2_as_u32(__hfma2(u32_as_bf2(v2), w2, nw2));
                        }
                        *reinterpret_cast<uint4*>(pdst + (size_t)q * K2T * 16) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
                    }
                } else {
                    const float s1 = exp2i(-e), wgt = exp2i(e - 6);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float f[8];
#pragma unroll
                        for (int t = 0; t < 8; ++t) {
                            const float rq = __uint_as_float(r[q * 8 + t]) * s1 * 64.0f + 0.5f;
                            f[t] = (float)min(__float2int_rz(rq), 127) * wgt;
                        }
                        *reinterpret_cast<uint4*>(pdst + (size_t)q * K2T * 16) =
                            make_uint4(pack_bf16_trunc(f[0], f[1]), pack_bf16_trunc(f[2], f[3]),
                                       pack_bf16_trunc(f[4], f[5]), pack_bf16_trunc(f[6], f[7]));
                    }
                }
            }
            fence_proxy_async_smem();
            tcgen05_fence_before_sync();
            group_sync(gc);
            if (tid == 0) {
                tcgen05_fence_after_sync();
                for (int wl = 0; wl < 4; ++wl) {
                    const int w = 4 * g + wl;
                    if (w >= NW) break;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint64_t da = umma_smem_desc(smem_u32(sP + (size_t)(wl * 4 + 2 * h) * K2T * 16), K2T * 16, 128);
                        const uint64_t db = umma_smem_desc(smem_u32(sV + (size_t)(w * 4 + 2 * h) * hdp * 16), hdp * 16, 128);
                        umma_bf16_ss(tmem, da, db, idesc_o, !first_mma);
                        first_mma = false;
                    }
                }
                umma_commit(&bar_o);
            }
        }
        mbar_wait(&bar_o, ph_o);
        ph_o ^= 1u;
        tcgen05_fence_after_sync();

        // ---- O -> A1 -> global (coalesced through the P region, which the finished MMAs no longer read)
        store_o_tile<BF16, OT>(tmem, sP, warp, lane, tile, Nq, hd, hdp, out_head, o_sN, out16);
        fence_proxy_async_smem();               // P writes (generic proxy) before the next TMA into the region
        tcgen05_fence_before_sync();
        group_sync(gc);                          // every lane has read O before TMEM / sP are reused
        tcgen05_fence_after_sync();
    }
}

// OT: output element type (DT_*)
template <bool BF16, bool BIAS, int OT = DT_F32>
__global__ void __launch_bounds__(K2P_T, 2)
k_attend_pair(const AttnParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[3];
    __shared__ uint32_t tmem_base_s;
    __shared__ float s_bias[BIAS ? 256 : 1];                        // PixArt cross-attention text mask (:794-803)
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int tid = threadIdx.x;
    const uint32_t tcols = (uint32_t)k2p_tmem_cols(O);
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1); }
    if ((tid >> 5) == 0) tmem_alloc(&tmem_base_s, tcols);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    GroupCtx g{tid, 0, smem, &bars[0], &bars[1], &bars[2], tmem_base_s, 0u, 0u, 0u, nullptr, 0};
    attend_pair_head<BF16, BIAS, OT>(g, O, p.Nq, p.Nk, p.hd, p.scale, p.flush != 0, p.q_op + (size_t)head * O.q_head_bytes,
                                     p.k_op + (size_t)head * O.k_head_bytes, p.v_op + (size_t)head * O.v_head_bytes,
                                     p.mask + (size_t)head * p.Nq * O.nw, out_elem(p.out, bb * p.o_sB + hh * p.o_sH, OT != DT_F32), p.o_sN,
                                     BIAS ? p.key_bias + bb * p.kb_sB : nullptr, s_bias, (int)blockIdx.y, (int)gridDim.y,
                                     OT != DT_F32);
    if ((tid >> 5) == 0) tmem_dealloc(g.tmem, tcols);
}


// ------------------------------------------------------------------------------------------
// V -> A1 -> MXINT8 along TOKENS (32-token windows per column) -> bf16 MMA-ready V^T operand.
// grid (heads, groups of 4 windows); thread <-> (window, column) pairs, consecutive threads on
// consecutive columns (coalesced loads, conflict-free 16-byte stores).
// ------------------------------------------------------------------------------------------
struct VPrepParams {
    View v;
    int H, Nq, Nk, hd, bf16, flush;
    unsigned char* v_op;
};

// DT: element type of the V view (DT_*)
template <int DT = DT_F32>
static __global__ void __launch_bounds__(K2T)
k_prep_v(const VPrepParams p) {
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int hdp = O.hdp, Nk = p.Nk, hd = p.hd;
    const int nw_pad = O.nblk * O.wpb;                         // windows incl. block padding
    const float* vb = view_elem<DT>(p.v.p, bb * p.v.sB + hh * p.v.sH);
    unsigned char* dst = p.v_op + (size_t)head * O.v_head_bytes;
    const int w0 = blockIdx.y * 4, w1 = min(w0 + 4, nw_pad);
    for (int t = threadIdx.x; t < (w1 - w0) * hdp; t += K2T) {
        const int w = w0 + t / hdp, d = t % hdp;
        uint32_t xb[32];
        uint32_t mx = 0u;
        const float* vp = view_elem<DT>(vb, (int64_t)(w * 32) * p.v.sN + d);
        const int nvalid = (d < hd) ? max(0, min(32, Nk - w * 32)) : 0;
#pragma unroll
        for (int tt = 0; tt < 32; ++tt) {
            uint32_t b = 0u;
            if (tt < nvalid) b = load_elem_bits<DT>(vp, 0);
            vp = view_elem<DT>(vp, p.v.sN);
            if (p.bf16) b = bf16_half_away(b);
            xb[tt] = b;
            mx = max(mx, b & 0x7fffffffu);
        }
        const int e = mx_shared_exp(mx);
        const bool dead = p.flush && e <= -127;
        if (mx != 0u && !dead && e >= -120 && e <= 126) {
            // codes without F2I / I2F (same arithmetic as the K1 quantizer): FFMA, clamp, FADD.RM against
            // 2^23 + 0x4300 -> bf16 pattern of 128 + c in the low half; (128 + c) * w - 128 * w = c * w
            const float s1 = exp2i(6 - e);
            const __nv_bfloat162 w2 = u32_as_bf2(bf16_pow2_bits(e - 6) * 0x00010001u);
            const __nv_bfloat162 nw2 = u32_as_bf2((bf16_pow2_bits(e + 1) | 0x8000u) * 0x00010001u);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t ow[4];
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const uint32_t x0 = xb[q * 8 + 2 * h], x1 = xb[q * 8 + 2 * h + 1];
                    const float v0 = fminf(fmaf(fabsf(__uint_as_float(x0)), s1, 0.5f), 127.0f);
                    const float v1 = fminf(fmaf(fabsf(__uint_as_float(x1)), s1, 0.5f), 127.0f);
                    const uint32_t v2 = __byte_perm(__float_as_uint(__fadd_rd(v0, 8405760.0f)),
                                                    __float_as_uint(__fadd_rd(v1, 8405760.0f)), 0x5410);
                    const uint32_t sx = __byte_perm(x0, x1, 0x7632) & 0x80008000u;
                    ow[h] = bf2_as_u32(__hfma2(u32_as_bf2(v2), w2, nw2)) ^ sx;
                }
                *reinterpret_cast<uint4*>(dst + v_op_offset(O, w * 4 + q, d)) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            }
        } else {
            const float wgt = exp2i(e - 6);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float f[8];
#pragma unroll
                for (int tt = 0; tt < 8; ++tt) f[tt] = (float)mx_code(xb[q * 8 + tt], e, dead) * wgt;
                *reinterpret_cast<uint4*>(dst + v_op_offset(O, w * 4 + q, d)) =
                    make_uint4(pack_bf16_trunc(f[0], f[1]), pack_bf16_trunc(f[2], f[3]), pack_bf16_trunc(f[4], f[5]),
                               pack_bf16_trunc(f[6], f[7]));
            }
        }
    }
}

// 8 int8 codes (two words) of one MX block with exponent weight w = 2^(e-6) -> 8 bf16 in a uint4
__device__ __forceinline__ uint4 dequant8_bf16(uint32_t lo, uint32_t hi, float w) {
    float f[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        f[t] = (float)(int)(signed char)((lo >> (8 * t)) & 0xff) * w;
        f[4 + t] = (float)(int)(signed char)((hi >> (8 * t)) & 0xff) * w;
    }
    return make_uint4(pack_bf16_trunc(f[0], f[1]), pack_bf16_trunc(f[2], f[3]), pack_bf16_trunc(f[4], f[5]),
                      pack_bf16_trunc(f[6], f[7]));
}

// ------------------------------------------------------------------------------------------
// Compact codes/exps -> MMA-ready operands (public mxp_sparse_attention entry, which receives
// codes).  which = 0: query rows (tiles of 128), 1: key rows (key blocks).  Also zero-fills padding.
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
k_codes_to_ops(const int8_t* __restrict__ codes, const int8_t* __restrict__ exps, unsigned char* __restrict__ ops,
               int heads, int Nq, int Nk, int hd, int which) {
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const int NB = (hd + 31) >> 5, kch = O.hdp >> 3;
    const int rows = which == 0 ? Nq : Nk;
    const int rows_pad = which == 0 ? O.q_tiles * K2T : O.nblk * O.kb_rows;
    const size_t head_bytes = which == 0 ? O.q_head_bytes : O.k_head_bytes;
    const int64_t total = (int64_t)heads * rows_pad * kch;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(t % rows_pad);
        const int kc = (int)((t / rows_pad) % kch);
        const int64_t head = t / ((int64_t)rows_pad * kch);
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (r < rows && kc * 8 < hd) {
            const int64_t grow = head * rows + r;
            const uint2 c = __ldg(reinterpret_cast<const uint2*>(codes + grow * hd + kc * 8));
            v = dequant8_bf16(c.x, c.y, exp2i((int)__ldg(exps + grow * NB + (kc >> 2)) - 6));
        }
        const size_t off = which == 0 ? q_op_offset(O, r, kc) : k_op_offset(O, r, kc);
        *reinterpret_cast<uint4*>(ops + head * head_bytes + off) = v;
    }
}

// ---- launchers defined in mxprune_fused.cu (second translation unit of libmxprune)
// Exact attention with the cost following top_k (mxprune_attend_sparse.cuh).  Returns 1 when the shape is outside
// that kernel's domain (the caller then launches the dense-epilogue kernel), else 0 with the launch status in *rc_out.
// top_k: every row of the mask holds at most top_k kept keys (masks written by the selection kernels).
int attend_sparse_try(const AttnParams& p, int top_k, cudaStream_t st, int* rc_out);

// The fused kernel (mxprune_fused.cuh): the whole path q,k,v -> out as one persistent launch.  Returns 1 when the
// call is outside its domain (the caller then runs the three-kernel path), else 0 with the launch status in *rc_out.
struct FusedArgs {
    View q, k, v;
    int dt, out_dt;                  // element types (DT_*) of q / k / v and of out
    int B, H, Nq, Nk, hd, top_k, bf16, flush;
    float scale;
    float* out;
    int64_t o_sB, o_sH, o_sN;
    uint32_t* mask_out;              // optional: where the caller wants the row masks
    unsigned char* slots;            // workspace for the per-group operand slots (256-byte aligned)
    size_t slots_bytes;
};
struct FusedSlotLayout { size_t k, v, mask, bytes; };
FusedSlotLayout fused_slot_layout(int Nq, int Nk, int hd);
size_t fused_workspace_bytes(int Nq, int Nk, int hd);
int fused_try(const FusedArgs& a, cudaStream_t st, int* rc_out);
void fused_set_pingpong(int on);
void fused_set_timing_buffer(unsigned long long* buf);   // debug: [2 * 160][32] u64 device buffer, or null

}  // namespace mxp
