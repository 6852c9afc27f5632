// K2-sparse: exact MXINT8 attention over the kept keys for SMALL top_k / Nk (Nk <= 256), cost following k.
//
// The reference only ever uses the k gathered entries of a row (workloads/deit/scripts/main.py:124,
// 147-152: gather -> softmax over k values -> scatter into zeros -> mx.matmul).  k_attend_pair evaluates
// its epilogue (scale, exp, P quantizer) for every key POSITION under a mask predicate, because a
// thread cannot index its TMEM registers dynamically; at DeiT's k / N = 15 % that is 85 % discarded
// work.  Here the dense part of the epilogue is only a copy:
//   S = Q.K^T on the tensor core (as before)  ->  each lane stages its 32-column TMEM window in shared
//   memory (8 x 16-byte stores, private to the thread) and walks the set bits of its mask word: the
//   kept scores are appended, scaled, to the row's LIST in shared memory (ascending key order, the
//   two lanes of a row at offsets derived from the mask popcounts), together with the key index; the
//   walk also yields the per-window maximum.
// Everything after that runs on the list, the row's two lanes splitting it by RANK (entries t = part,
// part + 2, ...: exactly top_k / 2 iterations for every thread - no divergence, two entries in flight):
//   pass B   e = exp(t - max), row sum
//   exps     window exponent from the window maximum: floor(log2(bf16?(exp(tmax_w - max) * inv))) - the
//            same arithmetic, on the same inputs, as the entry that attains the maximum
//   pass C   p = e * inv -> A1 -> MXINT8 code with the window's exponent -> one bf16 element scattered
//            into the (zero-filled) P operand of its 4-window group;  O += P_g . V_g on the tensor core.
// The list overlays the K operand (dead once S is complete; K is re-fetched per query tile, from L2).
// Masks must hold at most top_k kept keys per row (guaranteed for masks produced by the selection kernels).
//
// The body is a GROUP function (256 threads, one named barrier, its own shared-memory window, mbarriers
// and 256 TMEM columns): k_attend_sparse runs it as a whole CTA, the fused kernel (mxprune_fused.cuh) as
// one of the two groups of a CTA.
#pragma once
#include "mxprune_attend.cuh"

namespace mxp {

constexpr int K2S_LSTR = 144;          // list stride in entries: 128 rows + 16 (odd / even ranks hit disjoint banks)

struct K2sSmem {
    int cap;                            // list entries per row
    size_t off_lj, off_ew, off_v, off_p, total;
};
__host__ __device__ inline K2sSmem k2s_smem_layout(const OpsLayout& O, int top_k) {
    K2sSmem L;
    L.cap = top_k;
    size_t o = (size_t)L.cap * K2S_LSTR * 4;                    // list of fp32 values, [t][K2S_LSTR]
    L.off_lj = o; o += ((size_t)L.cap * K2S_LSTR + 15) & ~(size_t)15;   // key index per entry, u8
    L.off_ew = o; o += 8 * K2T * 8;                              // per (window, row): {2^(6-e) fp32, bf16 2^(e-6) | -128 * 2^(e-6) << 16}
    if (o < O.k_blk_bytes) o = O.k_blk_bytes;                    // the region first stages the K operand
    o = (o + 127) & ~(size_t)127;
    L.off_v = o; o += O.v_blk_bytes;
    L.off_p = o; o += K2_P_BYTES;                                // Q tile / window staging / P group
    L.total = o;
    return L;
}

// exp(x - m) for the list passes (x <= m)
__device__ __forceinline__ float exp_sub(float x, float m) { return exp_nonpos(__fsub_rn(x, m)); }

// One head (all its query tiles) through the sparse exact-attention epilogue.  q_op / k_op / v_op: this head's
// MMA-ready operands (global memory); mask_head: this head's [Nq][NW] mask words (global or shared memory);
// out_head: the head's output rows (row stride o_sN); OT / out16: output type (store_o_tile).
template <bool BF16, int OT = DT_F32>
__device__ __forceinline__ void attend_sparse_head(GroupCtx& g, const OpsLayout& O, const K2sSmem& L, int Nq, int Nk,
                                                   int hd, float scale, bool flush, const unsigned char* q_op,
                                                   const unsigned char* k_op, const unsigned char* v_op,
                                                   const uint32_t* mask_head, float* out_head, int64_t o_sN,
                                                   int tile_begin, int tile_step, bool out16 = false) {
    constexpr bool bf16 = BF16;
    const int hdp = O.hdp, NW = O.nw, kbr = O.kb_rows;
    const int NG = (NW + 3) >> 2;
    const int cap = L.cap;
    unsigned char* const smem = g.smem;
    unsigned char* sK = smem;
    float* s_list = reinterpret_cast<float*>(smem);
    unsigned char* s_lj = smem + L.off_lj;
    uint2* s_ew = reinterpret_cast<uint2*>(smem + L.off_ew);
    unsigned char* sV = smem + L.off_v;
    unsigned char* sP = smem + L.off_p;
    const int tid = g.tid, warp = tid >> 5, lane = tid & 31;
    const int lane_base = 32 * (warp & 3) + 16 * (warp >> 2);
    const int rr = lane_base + (lane & 15);                         // row of the tile
    const int part = lane >> 4;
    const uint32_t tmem = g.tmem;
    const uint32_t my_tmem = tmem + ((uint32_t)lane_base << 16);
    const uint32_t idesc_s = umma_idesc_bf16_f32(128, kbr);
    const uint32_t idesc_o = umma_idesc_bf16_f32(128, hdp);
    bool v_loaded = false;
    // this thread's private staging area for one 32-column window: 128 bytes at tid * 128, the 16-byte chunk q
    // stored at position q ^ (tid & 7) (conflict-free 128-bit stores); element c lives at byte (4 c) ^ stg_sw
    unsigned char* const stg = sP + tid * 128;
    const uint32_t stg_sw = (uint32_t)(tid & 7) << 4;

    for (int tile = tile_begin; tile < O.q_tiles; tile += tile_step) {
        const int i = tile * K2T + rr;
        const bool valid = i < Nq;
        const uint32_t* mrow = mask_head + (size_t)(valid ? i : 0) * NW;

        if (tid == 0) {     // Q tile -> the P region, K -> the list region; V once per head
            mbar_expect_tx(g.bar_ld, (uint32_t)(O.q_tile_bytes + O.k_blk_bytes + (v_loaded ? 0 : O.v_blk_bytes)));
            tma_bulk_g2s(sP, q_op + (size_t)tile * O.q_tile_bytes, (uint32_t)O.q_tile_bytes, g.bar_ld);
            tma_bulk_g2s(sK, k_op, (uint32_t)O.k_blk_bytes, g.bar_ld);
            if (!v_loaded) tma_bulk_g2s(sV, v_op, (uint32_t)O.v_blk_bytes, g.bar_ld);
        }
        v_loaded = true;
        // this lane's window slots t = 0..3: window w(t) = 4 (t >> 1) + 2 part + (t & 1)
        uint32_t mw[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int w = 4 * (t >> 1) + 2 * part + (t & 1);
            mw[t] = (valid && w < NW) ? mrow[w] : 0u;
        }
        // list offsets in ascending key order: windows 0,1 (part 0), 2,3 (part 1), 4,5 (part 0), 6,7 (part 1)
        const uint32_t pack = (uint32_t)__popc(mw[0]) | ((uint32_t)__popc(mw[1]) << 8) | ((uint32_t)__popc(mw[2]) << 16) |
                              ((uint32_t)__popc(mw[3]) << 24);
        const uint32_t opack = __shfl_xor_sync(FULL, pack, 16);
        const uint32_t pa = part ? opack : pack, pb = part ? pack : opack;     // part 0's / part 1's counts
        const int a0 = pa & 0xff, a1 = (pa >> 8) & 0xff, a2 = (pa >> 16) & 0xff, a3 = pa >> 24;
        const int b0 = pb & 0xff, b1 = (pb >> 8) & 0xff, b2 = (pb >> 16) & 0xff, b3 = pb >> 24;
        const int n0 = a0 + a1 + b0 + b1;                            // kept keys in windows 0..3
        const int ntot = min(n0 + a2 + a3 + b2 + b3, cap);           // all kept keys of the row (<= top_k by contract)
        int off[4];
        off[0] = part ? a0 + a1 : 0;
        off[1] = part ? a0 + a1 + b0 : a0;
        off[2] = part ? n0 + a2 + a3 : n0;
        off[3] = part ? n0 + a2 + a3 + b2 : n0 + a2;

        MXP_PROF(g, 10);
        mbar_wait(g.bar_ld, g.ph_ld);
        g.ph_ld ^= 1u;
        MXP_PROF(g, 11);
        if (tid == 0) {
            tcgen05_fence_after_sync();
            for (int ks = 0; ks < (hdp >> 4); ++ks) {
                const uint64_t da = umma_smem_desc(smem_u32(sP + (size_t)(2 * ks) * K2T * 16), K2T * 16, 128);
                const uint64_t db = umma_smem_desc(smem_u32(sK + (size_t)(2 * ks) * kbr * 16), kbr * 16, 128);
                umma_bf16_ss(tmem, da, db, idesc_s, ks > 0);
            }
            umma_commit(g.bar_s);
        }
        mbar_wait(g.bar_s, g.ph_s);                                 // S complete: the Q tile and K are consumed
        g.ph_s ^= 1u;
        tcgen05_fence_after_sync();
        MXP_PROF(g, 12);

        // ---- compaction: kept scores -> list (value = bf16?(s) * scale, key index), window maxima
        float wmax[4];
        {
            uint32_t r[32];
            tmem_ld_16x32bx2_s64_x32(my_tmem, r);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                wmax[t] = -INFINITY;
                if ((t >> 1) < NG) {                                // slot exists (uniform)
                    tmem_ld_wait();
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<uint4*>(stg + ((uint32_t)(q << 4) ^ stg_sw)) =
                            make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
                    if (t + 1 < 4 && ((t + 1) >> 1) < NG)
                        tmem_ld_16x32bx2_s64_x32(my_tmem + 128 * ((t + 1) >> 1) + 32 * ((t + 1) & 1), r);
                    const int wbase = 32 * (4 * (t >> 1) + 2 * part + (t & 1));
                    uint32_t m = mw[t];
                    // entries beyond the list's capacity (never with a selection-kernel mask) are dropped
                    if (off[t] + __popc(m) > cap) m = 0u;
                    float* pl = s_list + off[t] * K2S_LSTR + rr;
                    unsigned char* pj = s_lj + off[t] * K2S_LSTR + rr;
                    float wm = -INFINITY;
                    while (m) {                                     // two kept keys per iteration
                        const int c0 = __ffs((int)m) - 1;
                        m &= m - 1u;
                        const bool two = m != 0u;
                        const int c1 = two ? __ffs((int)m) - 1 : c0;
                        m &= m - 1u;
                        float s0 = *reinterpret_cast<const float*>(stg + ((uint32_t)(c0 << 2) ^ stg_sw));
                        float s1 = *reinterpret_cast<const float*>(stg + ((uint32_t)(c1 << 2) ^ stg_sw));
                        if (bf16) { s0 = bf16_half_away(s0); s1 = bf16_half_away(s1); }
                        const float t0 = __fmul_rn(s0, scale), t1 = __fmul_rn(s1, scale);
                        wm = fmaxf(wm, fmaxf(t0, t1));
                        pl[0] = t0;
                        pj[0] = (unsigned char)(wbase + c0);
                        if (two) {                                  // (the next slot may belong to the partner lane)
                            pl[K2S_LSTR] = t1;
                            pj[K2S_LSTR] = (unsigned char)(wbase + c1);
                        }
                        pl += two ? 2 * K2S_LSTR : K2S_LSTR;
                        pj += two ? 2 * K2S_LSTR : K2S_LSTR;
                    }
                    wmax[t] = wm;
                }
            }
        }
        float m = fmaxf(fmaxf(wmax[0], wmax[1]), fmaxf(wmax[2], wmax[3]));
        m = fmaxf(m, __shfl_xor_sync(FULL, m, 16));
        const float m_use = (m == -INFINITY) ? 0.f : m;             // no kept key
        __syncwarp();                                               // the partner lane's list entries
        MXP_PROF(g, 13);

        // ---- pass B: e = exp(t - max) over the row's list, the two lanes alternating; row sum
        const int nmine = (ntot - part + 1) >> 1;                   // entries part, part + 2, ...
        float sum0 = 0.f, sum1 = 0.f;
        {
            float* pl = s_list + part * K2S_LSTR + rr;
            int it = 0;
            for (; it + 2 <= nmine; it += 2) {
                const float x0 = pl[0], x1 = pl[2 * K2S_LSTR];
                const float e0 = exp_sub(x0, m_use), e1 = exp_sub(x1, m_use);
                sum0 += e0;
                sum1 += e1;
                pl[0] = e0;
                pl[2 * K2S_LSTR] = e1;
                pl += 4 * K2S_LSTR;
            }
            if (it < nmine) {
                const float e0 = exp_sub(pl[0], m_use);
                sum0 += e0;
                pl[0] = e0;
            }
        }
        float sum = sum0 + sum1;
        sum += __shfl_xor_sync(FULL, sum, 16);
        const float inv = sum > 0.f ? 1.0f / sum : 0.f;

        // ---- window exponents (A8: P blocks are 32 consecutive ORIGINAL key positions)
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int w = 4 * (t >> 1) + 2 * part + (t & 1);
            float s1 = 0.f;
            uint32_t wb = 0x3f80u | (0xc300u << 16);                // 1.0 | -128.0 (unused: no entries)
            if (wmax[t] != -INFINITY) {
                uint32_t pbits = __float_as_uint(exp_sub(wmax[t], m_use) * inv);
                if (bf16) pbits = bf16_half_away(pbits);
                const int e = mx_shared_exp(pbits);
                const bool dead = (flush && e <= -127) || pbits == 0u;
                if (dead || e >= -120) {
                    const int ec = max(e, -120);
                    s1 = dead ? 0.f : exp2i(6 - ec);
                    wb = bf16_pow2_bits(ec - 6) | ((bf16_pow2_bits(ec + 1) | 0x8000u) << 16);
                } else {
                    s1 = (float)e;                                  // negative: the slow path, exponent itself
                }
            }
            s_ew[w * K2T + rr] = make_uint2(__float_as_uint(s1), wb);
        }

        // ---- pass C: P = e * inv -> A1 -> MXINT8 with the window's exponent -> bf16 element of the A operand
        // (the P operand overlays the staging areas of ALL threads: every warp must have finished its walk)
        MXP_PROF(g, 14);
        group_sync(g);
        MXP_PROF(g, 15);
        bool first_mma = true;
        unsigned char* const prow = sP + rr * 16;
        const unsigned char* const erow = reinterpret_cast<const unsigned char*>(s_ew + rr);
        for (int gi = 0; gi < NG; ++gi) {
            if (gi > 0) {                                           // previous group's MMAs have finished reading sP
                mbar_wait(g.bar_o, g.ph_o);
                g.ph_o ^= 1u;
            }
            // zero this lane's two windows of its row, then scatter
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    *reinterpret_cast<uint4*>(prow + (size_t)((2 * part + j) * 4 + q) * K2T * 16) = make_uint4(0u, 0u, 0u, 0u);
            __syncwarp();
            const int tbeg = gi ? n0 : 0, tend = gi ? ntot : min(n0, ntot);
            // One list entry -> one bf16 element of the P operand.  The window's exponent record is a dependent shared-memory
            // load (entry -> key index -> window -> record), so two entries are processed together with ONE branch for the
            // rare slow exponent path (both chains in flight), and the next pair's entry is fetched before the current pair
            // is converted.
            auto window_rec = [&](int j) { return *reinterpret_cast<const uint2*>(erow + ((j & 0xe0) << 5)); };   // (j >> 5) * 128 * 8
            auto p_bits = [&](float ev) {
                uint32_t pbits = __float_as_uint(ev * inv);
                if (bf16) pbits = bf16_half_away(pbits);
                return pbits;
            };
            auto fast_val = [&](uint32_t pbits, const uint2& ew) {
                // code = min(127, floor(p * 2^(6-e) + 0.5)) without F2I / I2F (see K1)
                const float v = fminf(fmaf(__uint_as_float(pbits), __uint_as_float(ew.x), 0.5f), 127.0f);
                const uint32_t cb = __float_as_uint(__fadd_rd(v, 8405760.0f)) & 0xffffu;         // bf16 pattern of 128 + code
                return bf2_as_u32(__hfma2(u32_as_bf2(cb), u32_as_bf2(ew.y), u32_as_bf2(ew.y >> 16)));
            };
            auto any_val = [&](uint32_t pbits, const uint2& ew) {
                const float s1 = __uint_as_float(ew.x);
                if (s1 >= 0.f) return fast_val(pbits, ew);
                const int e = (int)s1;
                const float rq = __uint_as_float(pbits) * exp2i(-e) * 64.0f + 0.5f;
                return __float_as_uint((float)min(__float2int_rz(rq), 127) * exp2i(e - 6)) >> 16;
            };
            auto put = [&](int j, uint32_t val) {
                // element (window j >> 5 & 3, key j & 31): chunk (j & 127) >> 3 of the group, 2-byte slot j & 7
                *reinterpret_cast<unsigned short*>(prow + ((((uint32_t)j & 127u) * 0x102u) & 0x780eu)) = (unsigned short)val;
            };
            const int first = tbeg + ((part ^ tbeg) & 1);           // this lane's parity class: t = part (mod 2)
            const int nmy = (tend - first + 1) >> 1;
            const float* pl = s_list + first * K2S_LSTR + rr;
            const unsigned char* pj = s_lj + first * K2S_LSTR + rr;
            int it = 0;
            int j0 = 0, j1 = 0;
            float e0 = 0.f, e1 = 0.f;
            if (nmy >= 2) { j0 = pj[0]; j1 = pj[2 * K2S_LSTR]; e0 = pl[0]; e1 = pl[2 * K2S_LSTR]; }
            for (; it + 2 <= nmy; it += 2) {
                const uint2 w0 = window_rec(j0), w1 = window_rec(j1);
                const int cj0 = j0, cj1 = j1;
                const uint32_t pb0 = p_bits(e0), pb1 = p_bits(e1);
                pl += 4 * K2S_LSTR;
                pj += 4 * K2S_LSTR;
                if (it + 4 <= nmy) { j0 = pj[0]; j1 = pj[2 * K2S_LSTR]; e0 = pl[0]; e1 = pl[2 * K2S_LSTR]; }
                uint32_t v0, v1;
                if (__uint_as_float(w0.x) >= 0.f && __uint_as_float(w1.x) >= 0.f) {
                    v0 = fast_val(pb0, w0);
                    v1 = fast_val(pb1, w1);
                } else {
                    v0 = any_val(pb0, w0);
                    v1 = any_val(pb1, w1);
                }
                put(cj0, v0);
                put(cj1, v1);
            }
            if (it < nmy) {
                const int j = pj[0];
                put(j, any_val(p_bits(pl[0]), window_rec(j)));
            }
            MXP_PROF(g, 16);
            fence_proxy_async_smem();
            tcgen05_fence_before_sync();
            group_sync(g);
            MXP_PROF(g, 17);
            if (tid == 0) {
                tcgen05_fence_after_sync();
                for (int wl = 0; wl < 4; ++wl) {
                    const int w = 4 * gi + wl;
                    if (w >= NW) break;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint64_t da = umma_smem_desc(smem_u32(sP + (size_t)(wl * 4 + 2 * h) * K2T * 16), K2T * 16, 128);
                        const uint64_t db = umma_smem_desc(smem_u32(sV + (size_t)(w * 4 + 2 * h) * hdp * 16), hdp * 16, 128);
                        umma_bf16_ss(tmem, da, db, idesc_o, !first_mma);
                        first_mma = false;
                    }
                }
                umma_commit(g.bar_o);
            }
        }
        mbar_wait(g.bar_o, g.ph_o);
        g.ph_o ^= 1u;
        tcgen05_fence_after_sync();
        MXP_PROF(g, 18);

        // ---- O -> A1 -> global (coalesced through the P region, which the finished MMAs no longer read)
        store_o_tile<BF16, OT>(tmem, sP, warp, lane, tile, Nq, hd, hdp, out_head, o_sN, out16);
        MXP_PROF(g, 19);
        fence_proxy_async_smem();               // list / P writes (generic proxy) before the next tile's TMA overwrites them
        tcgen05_fence_before_sync();
        group_sync(g);                          // every lane has read O before TMEM / sP / the list are reused
        tcgen05_fence_after_sync();
        MXP_PROF(g, 20);
    }
}

template <bool BF16, int OT = DT_F32>
__global__ void __launch_bounds__(K2P_T, 2)
k_attend_sparse(const AttnParams p, const int top_k) {
    extern __shared__ __align__(128) unsigned char smem_k2s[];
    __shared__ uint64_t bars[3];
    __shared__ uint32_t tmem_base_s;
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    const K2sSmem L = k2s_smem_layout(O, top_k);
    const int head = blockIdx.x, bb = head / p.H, hh = head % p.H;
    const int tid = threadIdx.x;
    const uint32_t tcols = (uint32_t)k2p_tmem_cols(O);
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1); }
    if ((tid >> 5) == 0) tmem_alloc(&tmem_base_s, tcols);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    GroupCtx g{tid, 0, smem_k2s, &bars[0], &bars[1], &bars[2], tmem_base_s, 0u, 0u, 0u, nullptr, 0};
    attend_sparse_head<BF16, OT>(g, O, L, p.Nq, p.Nk, p.hd, p.scale, p.flush != 0,
                                 p.q_op + (size_t)head * O.q_head_bytes, p.k_op + (size_t)head * O.k_head_bytes,
                                 p.v_op + (size_t)head * O.v_head_bytes, p.mask + (size_t)head * p.Nq * O.nw,
                                 out_elem(p.out, bb * p.o_sB + hh * p.o_sH, OT != DT_F32), p.o_sN, (int)blockIdx.y,
                                 (int)gridDim.y, OT != DT_F32);
    if ((tid >> 5) == 0) tmem_dealloc(g.tmem, tcols);
}

}  // namespace mxp
