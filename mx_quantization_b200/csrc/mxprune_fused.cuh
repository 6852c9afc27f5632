// The fused kernel: quantizer + exponent-sign predictor + top-k + V preparation + exact attention over the
// kept keys of workloads/deit/scripts/main.py:101-152 as ONE persistent launch (Nk <= 256).
//
// One CTA of 512 threads per SM = two independent GROUPS of 256 threads.  A group owns a 113 KiB window of
// shared memory, 256 TMEM columns, one named barrier and its own mbarriers, and walks a static list of heads;
// per head it runs two phases back to back:
//   phase 1 (predict_topk_head)  TMA-stage K, V and Q rows of the strided fp32 views; MX-quantize them (one
//       thread per 32-wide block along head_dim for Q / K, per 32-TOKEN window and column for V); score the
//       +-2^e operands on the tensor core; select the top_k keys of every query row in registers (the code of
//       k_predict_topk_tc, mxprune_predict_tc.cuh).  The exact bf16 operands of Q, K and V^T and the row masks
//       go to the group's private WORKSPACE SLOT in global memory - ~95 KB that the same SM re-reads a few
//       microseconds later and overwrites for its next head, so it lives in L2 and never needs to reach HBM.
//   phase 2 (attend_sparse_head / attend_pair_head)  exact MXINT8 attention over the kept keys, operands
//       fetched from the slot with TMA bulk copies, shared memory and TMEM of phase 1 reused.
// The two groups of an SM run unsynchronised, so one group's ALU-bound selection overlaps the other's
// latency-bound attention epilogue - the overlap two separate kernels (each filling the SM with its own
// kind of work) cannot have - and q/k/v operands and masks make no HBM round trip.
#pragma once
#include "mxprune_predict_tc.cuh"
#include "mxprune_attend_sparse.cuh"

namespace mxp {

constexpr int FUSED_T = 512;
constexpr size_t FUSED_GROUP_SMEM = 113 * 1024;           // per-group window (multiple of 1024: SWIZZLE_128B boxes)

// Phase-1 staging geometry of the fused kernel as a function of (head_dim, key chunks): TMA boxes per ring slot (G) and
// ring depth, the largest that fit the group's window.  constexpr: the launcher and the head_dim-specialised kernel
// instantiations (template HD) evaluate the same rule.
__host__ __device__ constexpr inline int fused_G(int hd, int nc) {
    const int nb = (hd + 31) / 32;
    int G = nb <= 2 ? 2 : 1;
    if (k1c_smem_layout(hd, nc, 2, G).total > FUSED_GROUP_SMEM - 256) G = 1;
    return G;
}
__host__ __device__ constexpr inline int fused_ring(int hd, int nc) {
    const int G = fused_G(hd, nc);
    int ring = K1C_MAXR;
    while (ring > 2 && k1c_smem_layout(hd, nc, ring, G).total > FUSED_GROUP_SMEM - 256) --ring;
    return ring;
}

struct FusedMaps {
    CUtensorMap q_main, q_tail, k_main, k_tail, v_main, v_tail;
};

struct FusedParams {
    int B, H, Nq, Nk, hd, top_k, bf16, flush;
    float scale;
    float* out;                  // fp32, or the kernel's 16-bit input type when out16
    int64_t o_sB, o_sH, o_sN;
    uint32_t* mask_out;          // optional [B*H][Nq][NW]: when given, the masks are written there instead of the slot
    unsigned char* slots;        // workspace: one slot per group
    size_t slot_bytes, slot_k, slot_v, slot_mask;    // byte offsets of the k / v operands and the mask inside a slot
    int ring, G;                 // TMA ring of phase 1
    int sparse;                  // phase 2: 1 = cost-follows-k epilogue, 0 = dense epilogue
    int pingpong;                // 1: at most one group of a CTA inside phase 1 at a time (drives the groups into anti-phase)
    unsigned long long* timing;  // debug: [2 * gridDim][32] per-phase cycle sums of each group's thread 0 (null = off)
    int out16;                   // 16-bit input kernels: out holds the input type instead of fp32
};

struct K1State {                 // phase-1 pipeline state carried from head to head
    int slot_i;
    uint32_t slot_par, ph_mma;
};

// ---- phase 1 for one head.  bar_full[ring], bar_mma: the group's mbarriers (count 1).
// HD: head_dim as a compile-time constant (0 = run time): with it every staging / operand offset of the quantize steps folds
// (The token count folded as well - 197 - gave no smaller code and 116 bytes of spills at the 128-register cap:
// 5.40 -> 5.92 ms per DeiT-base step.  Not a template parameter.)
template <int NC, int HG, bool BF16, int HD, int DT>
__device__ __forceinline__ void predict_topk_head(GroupCtx& gc, K1State& st, uint64_t* bar_full, uint64_t* bar_mma,
                                                  const FusedParams& p, const FusedMaps& maps, const K1cSmem& L,
                                                  const OpsLayout& OL, int head, unsigned char* q_op, unsigned char* k_op,
                                                  unsigned char* v_op, uint32_t* mask_head, int tile_begin, int tile_step) {
    unsigned char* const smem = gc.smem;
    constexpr int NMMA = 32 * NC;
    constexpr int NCH = (NC + 1) / 2;                               // key chunks per thread
    constexpr int HW = HG ? 8 * HG : NCH * 32;                      // key columns per lane
    constexpr int NPAIR = HW / 32, REM = HW - 32 * NPAIR;           // full 32-column chunks + an 8- or 16-column rest
    constexpr int NWORDS = HW / 2;                                  // packed key words per lane
    constexpr int NLW = (HW + 31) / 32;                             // bitmask words per lane (lane-local bit order)
    static_assert(HG == 0 || ((REM == 8 || REM == 16) && 16 * HG <= 32 * NC && NWORDS % 4 == 0), "tight split");
    const int Nk = p.Nk, Nq = p.Nq, hd = HD ? HD : p.hd, kk = p.top_k;
    const int G = L.G, ring = L.ring;
    const int nfull = L.nfull, tail = L.tail, nb = L.nb;
    const int kch = L.hdp >> 3;                                     // 16-byte chunks per predictor-operand row
    const int tail_chunks_hbm = (((hd + 15) & ~15) >> 3) - 4 * nfull;
    const int tail_chunks = kch - 4 * nfull;
    unsigned char* s_kop = smem + L.off_kop;
    unsigned char* s_qop = smem + L.off_qop;
    uint32_t* s_ksign = reinterpret_cast<uint32_t*>(smem + L.off_ksign);
    signed char* s_kexp = reinterpret_cast<signed char*>(smem + L.off_kexp);
    uint32_t* s_qsign = reinterpret_cast<uint32_t*>(smem + L.off_qsign);
    signed char* s_qexp = reinterpret_cast<signed char*>(smem + L.off_qexp);
    int* s_kmin = reinterpret_cast<int*>(smem + L.off_misc);        // [4]
    int* s_kmax = s_kmin + 4;                                       // [4]

    const int bb = head / p.H, hh = head - bb * p.H;
    const int tid = gc.tid, warp = tid >> 5, lane = tid & 31;
    const int lane_base = 32 * (warp & 3) + 16 * (warp >> 2);
    const int rr = lane_base + (lane & 15);                         // row of the tile
    const int part = lane >> 4;
    constexpr bool bf16 = BF16;
    const bool flush = p.flush;
    const int kb_rows = OL.kb_rows;
    const int hdp_v = OL.hdp, NWk = OL.nw;

    // ---- step schedule: CR = 64 G rows per step; K steps, then V steps, then the Q tiles
    const int CR = K1C_ROWS * G, cr_shift = G == 2 ? 7 : 6;
    const int nks = (NMMA + CR - 1) / CR;                           // every MMA row of the K operand is written
    const int nvs = (32 * NWk + CR - 1) / CR;                       // every token window of V
    const int qsteps = K1C_TILE / CR;                               // steps per query tile (2 or 1)
    const int tiles_all = (Nq + K1C_TILE - 1) / K1C_TILE;
    const int tiles = tiles_all > tile_begin ? (tiles_all - tile_begin + tile_step - 1) / tile_step : 0;   // this group's query tiles
    const int nsteps = nks + nvs + qsteps * tiles;
    const uint32_t box_main = (uint32_t)L.box_main, box_tail = (uint32_t)L.box_tail;
    const uint32_t slot_tx = (uint32_t)G * (box_main + box_tail) / (DT == DT_F32 ? 1 : 2);
    const uint32_t slot_bytes = (uint32_t)L.slot_bytes;
    const uint32_t tail_base = (uint32_t)G * box_main;

    auto issue = [&](int c, int slot_i) {                           // one thread
        unsigned char* slot = smem + (size_t)slot_i * slot_bytes;
        uint64_t* bar = &bar_full[slot_i];
        const CUtensorMap *mm, *mt;
        int row0;
        if (c < nks) { mm = &maps.k_main; mt = &maps.k_tail; row0 = c * CR; }
        else if (c < nks + nvs) { mm = &maps.v_main; mt = &maps.v_tail; row0 = (c - nks) * CR; }
        else {
            const int qc = c - nks - nvs, qt = qc / qsteps;
            mm = &maps.q_main; mt = &maps.q_tail;
            row0 = (tile_begin + qt * tile_step) * K1C_TILE + (qc - qt * qsteps) * CR;
        }
        mbar_expect_tx(bar, slot_tx);
        for (int g = 0; g < G; ++g) {
            if (nfull) tma_load_5d(slot + g * box_main, mm, 0, row0 + g * K1C_ROWS, 0, hh, bb, bar);
            if (tail) tma_load_4d(slot + tail_base + g * box_tail, mt, 0, row0 + g * K1C_ROWS, hh, bb, bar);
        }
    };

    if (tid < 4) { s_kmin[tid] = 0x7fffffff; s_kmax[tid] = -0x7fffffff; }
    if (tid == 0) {
        const int pre = min(ring, nsteps);
        int s = st.slot_i;
        for (int c = 0; c < pre; ++c) {
            issue(c, s);
            if (++s == ring) s = 0;
        }
    }
    group_sync(gc);                                                 // kmin / kmax initialised
    const uint32_t tmem = gc.tmem;
    const uint32_t my_tmem = tmem + ((uint32_t)lane_base << 16);
    const uint32_t idesc = umma_idesc_bf16_f32(128, NMMA);
    const int NW = (Nk + 31) >> 5;
    const int my_cols_end = HG ? (part + 1) * HW : min(NC, (part + 1) * NCH) * 32, my_cols_beg = part * HW;
    const int my_pad = max(0, my_cols_end - max(Nk, my_cols_beg));
    int slot_i = st.slot_i;
    uint32_t slot_par = st.slot_par, ph_mma = st.ph_mma;
    int tile = tile_begin - tile_step;
    int qstep = qsteps - 1;

    for (int c = 0; c < nsteps; ++c) {
        const bool is_k = c < nks;
        const bool is_v = !is_k && c < nks + nvs;
        if (!is_k && !is_v) {
            if (++qstep == qsteps) { qstep = 0; tile += tile_step; }
        }
        const int row0 = is_k ? c * CR : is_v ? (c - nks) * CR : tile * K1C_TILE + qstep * CR;
        const int nrows = is_k ? Nk : Nq;
        const unsigned char* slot = smem + (size_t)slot_i * slot_bytes;
        MXP_PROF(gc, 0);
        mbar_wait(&bar_full[slot_i], slot_par);
        MXP_PROF(gc, 1);

        if (is_v) {
            // -------- V: A1 + MXINT8 along TOKENS (32-token windows per column, matmul.py:76-83) -> bf16 V^T operand.
            // task = (window of the step, column): consecutive lanes read consecutive columns of one staged row
            // (one 128-byte line of the swizzled box: conflict-free) and store consecutive 16-byte chunks.
            const int ntask = (CR >> 5) * hdp_v;
            for (int t = tid; t < ntask; t += K2P_T) {
                const int wl = t / hdp_v, d = t - wl * hdp_v;
                const int w = (row0 >> 5) + wl;
                if (w >= NWk) continue;
                uint32_t xv[32];
                if (DT != DT_F32 && d < 32 * nfull) {             // 64-byte rows, SWIZZLE_64B (staged_block_bits)
                    const int b = d >> 5, dd = d & 31;
                    const unsigned char* src = slot + ((wl >> 1) * box_main) + (size_t)(b * 64 + (wl & 1) * 32) * 64 + ((dd & 7) << 1);
                    const int ch = dd >> 3;
#pragma unroll
                    for (int tt = 0; tt < 32; ++tt)
                        xv[tt] = widen1<DT>(*reinterpret_cast<const uint16_t*>(src + tt * 64 + ((ch ^ ((tt >> 1) & 3)) << 4)));
                } else if (DT != DT_F32 && d < hd) {
                    const unsigned char* src = slot + tail_base + (wl >> 1) * box_tail + (size_t)((wl & 1) * 32) * tail * 2 + (d - 32 * nfull) * 2;
#pragma unroll
                    for (int tt = 0; tt < 32; ++tt) xv[tt] = widen1<DT>(*reinterpret_cast<const uint16_t*>(src + tt * tail * 2));
                } else if (d < 32 * nfull) {
                    const int b = d >> 5, dd = d & 31;
                    const unsigned char* src = slot + ((wl >> 1) * box_main) + (size_t)(b * 64 + (wl & 1) * 32) * 128 + ((dd & 3) << 2);
                    const int ch = dd >> 2;
#pragma unroll
                    for (int tt = 0; tt < 32; ++tt)
                        xv[tt] = *reinterpret_cast<const uint32_t*>(src + tt * 128 + ((ch ^ (tt & 7)) << 4));
                } else if (d < hd) {
                    const unsigned char* src = slot + tail_base + (wl >> 1) * box_tail + (size_t)((wl & 1) * 32) * tail * 4 + (d - 32 * nfull) * 4;
#pragma unroll
                    for (int tt = 0; tt < 32; ++tt) xv[tt] = *reinterpret_cast<const uint32_t*>(src + tt * tail * 4);
                } else {
#pragma unroll
                    for (int tt = 0; tt < 32; ++tt) xv[tt] = 0u;
                }
                BlockQ r;
                quantize_block_thread<false, false>(xv, 32, bf16, flush, r);
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    *reinterpret_cast<uint4*>(v_op + ((size_t)(w * 4 + q) * hdp_v + d) * 16) = r.op[q];
            }
        } else {
            // -------- quantize the step's rows: one thread per MX block, block-major task order
            const int ntask = CR * nb;
            for (int t = tid; t < ntask; t += K2P_T) {
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
                quantize_block_thread<false>(xv, full ? 32 : tail, bf16, flush, r);
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
                    if (row < kb_rows) {
                        unsigned char* dst = k_op + ((size_t)(4 * b) * kb_rows + row) * 16;
#pragma unroll
                        for (int ch = 0; ch < 4; ++ch)
                            if (ch < nchunk_hbm) *reinterpret_cast<uint4*>(dst + (size_t)ch * kb_rows * 16) = r.op[ch];
                    }
                } else {
                    const int rt = qstep * CR + rl;                     // row within the tile
                    unsigned char* dst = s_qop + ((4 * b) * K1C_TILE + rt) * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch)
                        if (ch < nchunk) *reinterpret_cast<uint4*>(dst + ch * (K1C_TILE * 16)) = r.pp[ch];
                    s_qsign[b * K1C_TILE + rt] = r.sign;
                    s_qexp[b * K1C_TILE + rt] = (signed char)r.ep;
                    unsigned char* gdst = q_op + (size_t)tile * OL.q_tile_bytes + ((size_t)(4 * b) * K1C_TILE + rt) * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch)
                        if (ch < nchunk_hbm) *reinterpret_cast<uint4*>(gdst + ch * (K1C_TILE * 16)) = r.op[ch];
                }
            }
        }
        MXP_PROF(gc, 2);
        fence_proxy_async_smem();                                   // operand stores -> visible to the MMA
        group_sync(gc);                                             // slot consumed; operands complete
        MXP_PROF(gc, 3);
        if (tid == 0 && c + ring < nsteps) issue(c + ring, slot_i);
        if (++slot_i == ring) { slot_i = 0; slot_par ^= 1u; }
        if (is_k || is_v || qstep != qsteps - 1) continue;

        // =============== a full query tile is quantized: score, select, emit
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

        MXP_PROF(gc, 4);
        mbar_wait(bar_mma, ph_mma);
        ph_mma ^= 1u;
        tcgen05_fence_after_sync();
        MXP_PROF(gc, 5);

        // ---- scores -> fp16-pattern keys in registers (see k_predict_topk_tc)
        uint32_t kw[NWORDS];
#pragma unroll
        for (int w = 0; w < NPAIR; ++w) {
            const bool real = HG != 0 || (w < NCH - 1) || (NC % 2 == 0) || part == 0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t r[16];
                tmem_ld_16x32bx2_x16<HW>(my_tmem + w * 32 + h * 16, r);
                tmem_ld_wait();
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
        MXP_PROF(gc, 6);
        tcgen05_fence_before_sync();
        group_sync(gc);
        MXP_PROF(gc, 7);

        // ---- select: T = top_k-th largest key; the row's two lanes add their counts
        int nge_m, nge_o, ngt_m, ngt_o;
        const int nvalid_m = min(my_cols_end, max(Nk, my_cols_beg)) - my_cols_beg;
        const uint32_t T = select_kth_key<NWORDS, (HG == 0 && (NC & 1))>(kw, key0, my_pad, kk, nvalid_m, Nk - nvalid_m,
                                                                       nge_m, nge_o, ngt_m, ngt_o);
        MXP_PROF(gc, 8);

        // ---- emit the row bitmask (ties: ascending key index; the lower lane owns the lower columns)
        {
            const int rem_all = kk - (ngt_m + ngt_o);               // ties to keep in the whole row
            const int ties0 = part == 0 ? nge_m - ngt_m : nge_o - ngt_o;
            int rem = part == 0 ? rem_all : rem_all - min(rem_all, ties0);
            const __half2 t2 = u32_as_h2(T * 0x00010001u);
            const bool store = valid && fast;
            uint32_t* mrow32 = mask_head + (size_t)(valid ? i : 0) * NW;
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
                    if (store && gw < NW) mrow32[gw] = word;
                } else {
                    lw[w] = word;
                }
            }
            if constexpr (HG != 0) {                                // aligned word stores (see k_predict_topk_tc)
                const uint32_t other0 = __shfl_xor_sync(FULL, lw[0], 16);
                if (store) {
                    if (part == 0) {
#pragma unroll
                        for (int w = 0; w < NPAIR; ++w) mrow32[w] = lw[w];
                        mrow32[NPAIR] = lw[NPAIR] | (other0 << REM);
                    } else {
#pragma unroll
                        for (int w = 0; w < NPAIR; ++w)
                            if (NPAIR + 1 + w < NW) mrow32[NPAIR + 1 + w] = __funnelshift_l(lw[w], lw[w + 1], REM);
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
            const int64_t grow = tile * K1C_TILE + lane_base + l;
            predict_row_generic_tc(mask_head, nullptr, Nk, kk, hd, nb, grow, gsq, gep, s_ksign, s_kexp, nullptr);
        }
        MXP_PROF(gc, 9);
    }
    st.slot_i = slot_i;
    st.slot_par = slot_par;
    st.ph_mma = ph_mma;
}

// The two phases of a head.  (Inlined: as separate functions the call ABI's callee-saved registers cost 0.5 - 1.2 KB
// of spills per thread; inlined the kernel stays at the 128-register cap with a handful of spilled loop invariants.
// Keep an eye on `-Xptxas -v`: spills next to in-flight tcgen05.ld results are not something to live with.)
template <int NC, int HG, bool BF16, int HD, int DT>
__device__ __forceinline__ void fused_phase1(GroupCtx& gc, K1State& st, uint64_t* bars, const FusedParams& p, const FusedMaps& maps,
                                          int head, unsigned char* slot, uint32_t* mask_head, int tile_begin, int tile_step) {
    const K1cSmem L1 = HD ? k1c_smem_layout(HD, NC, fused_ring(HD, NC), fused_G(HD, NC)) : k1c_smem_layout(p.hd, NC, p.ring, p.G);
    const OpsLayout O = ops_layout(p.Nq, p.Nk, HD ? HD : p.hd);
    predict_topk_head<NC, HG, BF16, HD, DT>(gc, st, &bars[0], &bars[K1C_MAXR], p, maps, L1, O, head, slot, slot + p.slot_k, slot + p.slot_v,
                              mask_head, tile_begin, tile_step);
}
// HD != 0: head_dim at compile time; such instantiations carry the cost-follows-k epilogue only (the launcher sends
// dense-epilogue calls to the HD = 0 kernels); so do the KMAX != 0 ones (launched for sparse calls only)
template <bool BF16, int HD, int DT, int KMAX>
__device__ __forceinline__ void fused_phase2(GroupCtx& gc, const FusedParams& p, int head, const unsigned char* slot,
                                          const uint32_t* mask_head, int tile_begin, int tile_step) {
    const int hd = HD ? HD : p.hd, Nq = p.Nq, Nk = p.Nk;
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const int bb = head / p.H, hh = head - bb * p.H;
    const bool out16 = DT != DT_F32 && p.out16 != 0;
    float* out_head = out16 ? out_elem(p.out, bb * p.o_sB + hh * p.o_sH, true) : p.out + bb * p.o_sB + hh * p.o_sH;
    if (HD != 0 || KMAX != 0 || p.sparse) {
        const K2sSmem L2 = k2s_smem_layout(O, p.top_k);
        attend_sparse_head<BF16, DT, KMAX>(gc, O, L2, Nq, Nk, hd, p.scale, p.flush != 0, slot, slot + p.slot_k, slot + p.slot_v,
                                           mask_head, out_head, p.o_sN, tile_begin, tile_step, out16);
    } else {
        attend_pair_head<BF16, false, DT>(gc, O, Nq, Nk, hd, p.scale, p.flush != 0, slot, slot + p.slot_k, slot + p.slot_v,
                                          mask_head, out_head, p.o_sN, nullptr, nullptr, tile_begin, tile_step, out16);
    }
}

// NC, HG: key-column geometry of phase 1 (see k_predict_topk_tc); BF16: A1 rounding on (bfloat 16); HD: head_dim at
// compile time (0 = any); DT: element type of q / k / v (DT_*) - the output is fp32 or, with p.out16, that type;
// KMAX: register bound of the cost-follows-k epilogue (0: list path; != 0: register path, sparse epilogue only)
template <int NC, int HG, bool BF16, int HD, int DT = DT_F32, int KMAX = 0>
__global__ void __launch_bounds__(FUSED_T, 1)
k_fused_pruned_attention(const __grid_constant__ FusedParams p, const __grid_constant__ FusedMaps maps) {
    extern __shared__ __align__(1024) unsigned char smem_fused[];
    __shared__ uint64_t s_bars[2][K1C_MAXR + 4];                    // per group: ring, mma, ld, s, o
    __shared__ uint32_t s_tmem[2];
    __shared__ int s_lock;                                          // phase-1 token of the CTA's two groups
    const int grp = threadIdx.x >> 8;
    const int tid = threadIdx.x & 255;
    uint64_t* bars = s_bars[grp];
    const int heads = p.B * p.H;
    const int Nq_ = p.Nq, Nk_ = p.Nk;
    const int NW = (Nk_ + 31) >> 5;
    const bool has_tail = (p.hd & 31) != 0;

    if (threadIdx.x == 0) s_lock = 0;
    if (tid == 0) {
        for (int r = 0; r < K1C_MAXR + 4; ++r) mbar_init(&bars[r], 1);
        prefetch_tmap(&maps.k_main); prefetch_tmap(&maps.q_main); prefetch_tmap(&maps.v_main);
        if (has_tail) { prefetch_tmap(&maps.k_tail); prefetch_tmap(&maps.q_tail); prefetch_tmap(&maps.v_tail); }
    }
    if ((threadIdx.x >> 5) == 0) tmem_alloc(&s_tmem[0], 512u);        // the SM's whole tensor memory: 256 columns per group
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    GroupCtx gc{tid, 1 + grp, smem_fused + (size_t)grp * FUSED_GROUP_SMEM, &bars[K1C_MAXR + 1], &bars[K1C_MAXR + 2],
                &bars[K1C_MAXR + 3], s_tmem[0] + 256u * (uint32_t)grp, 0u, 0u, 0u, nullptr, 0};
    // debug accounting lives in the last 256 bytes of the group's window (beyond every layout's footprint)
    unsigned long long* const s_prof = reinterpret_cast<unsigned long long*>(gc.smem + FUSED_GROUP_SMEM - 256);
    if (p.timing) {
        if (tid < 32) s_prof[tid] = 0ull;
        gc.prof = s_prof;
        gc.t_last = clock64();
    }
    K1State st{0, 0u, 0u};
    const int gslot = 2 * (int)blockIdx.x + grp;
    unsigned char* const slot = p.slots + (size_t)gslot * p.slot_bytes;

    // Heads are dealt round-robin to the chip's groups.  The last, partial round would leave most groups idle for a whole
    // head time (3072 heads over 296 groups: 10 full rounds + 112 heads); when at most half of the groups have a head
    // left and a head has two query tiles, the two groups of a CTA share one head of that round instead - each
    // quantizes K and V for itself and takes one of the query tiles (no phase-1 token: they start together).
    const int ngroups = 2 * (int)gridDim.x;
    const int full = heads / ngroups, rem = heads - full * ngroups;
    const bool tail_split = rem > 0 && 2 * rem <= ngroups && (Nq_ + K1C_TILE - 1) / K1C_TILE == 2;
    const int nrounds = full + (rem > 0 ? 1 : 0);
    for (int r = 0; r < nrounds; ++r) {
        int head = r * ngroups + gslot, tile_begin = 0, tile_step = 1;
        bool lock = p.pingpong != 0;
        if (r == full) {
            if (tail_split) {
                if (gslot >= 2 * rem) break;
                head = r * ngroups + (gslot >> 1);
                tile_begin = gslot & 1;
                tile_step = 2;
                lock = false;
            } else if (gslot >= rem) {
                break;
            }
        }
        uint32_t* mask_head = p.mask_out ? p.mask_out + (size_t)head * Nq_ * NW
                                         : reinterpret_cast<uint32_t*>(slot + p.slot_mask);
        if (lock) {                                                 // take the phase-1 token
            if (tid == 0) {
                while (atomicCAS(&s_lock, 0, 1) != 0) __nanosleep(64);
            }
            group_sync(gc);
        }
        fused_phase1<NC, HG, BF16, HD, DT>(gc, st, bars, p, maps, head, slot, mask_head, tile_begin, tile_step);
        // phase 1 -> phase 2: the slot's operands (generic-proxy global stores) are read back by TMA bulk copies
        // (async proxy), the masks by ordinary loads of other threads of the group; phase 2 also re-purposes the
        // shared memory that phase 1 wrote with generic stores as TMA destinations
        asm volatile("fence.proxy.async;" ::: "memory");
        __threadfence_block();
        tcgen05_fence_before_sync();
        group_sync(gc);
        tcgen05_fence_after_sync();
        if (lock && tid == 0) atomicExch(&s_lock, 0);               // every thread of the group has left phase 1
        MXP_PROF(gc, 21);
        fused_phase2<BF16, HD, DT, KMAX>(gc, p, head, slot, mask_head, tile_begin, tile_step);
        // phase 2 ends with fence.proxy.async + group barrier: its shared memory and TMEM may be reused, and its TMA
        // reads of the slot have completed (every copy was waited for), so the next head may overwrite the slot
    }
    if (p.timing && tid == 0) {
        MXP_PROF(gc, 22);
        for (int i = 0; i < 32; ++i) p.timing[(size_t)gslot * 32 + i] = s_prof[i];
    }
    tcgen05_fence_before_sync();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) tmem_dealloc(s_tmem[0], 512u);
}

}  // namespace mxp
