// K1-long-TC: the fused quantizer + exponent-sign predictor + exact top-k for Nk > 256 (the
// long-sequence sweep, config C5) with the scores on the tensor cores.
//
// A row's keys no longer fit in registers or shared memory, so the selection RE-SCORES the row in every pass - which is
// what the tensor core makes cheap: a pass streams the head's predictor operand Kp (bf16 +-2^e, MMA-ready, written once per
// head by k_quantize_ops) through shared memory in blocks of 128 keys, one tcgen05.mma per block and query tile into one of
// two TMEM buffers, and the threads read their scores back with tcgen05.ld.16x32bx2: a warp owns 16 query rows, lanes l and
// l + 16 share row l and take keys [0,64) / [64,128) of the block.  Per-lane u16 histograms in shared memory ([bin][thread]:
// conflict-free, no atomics); the two lanes of a row add their columns when they scan from the top bin.
//   fine window   (default) a sample of the row predicts its threshold; ONE pass with 126 exact bins around the prediction
//                 (bins of 2^fs keys + one level for the digit inside the bin when the sample spreads wide) - see
//                 k_select_long_tc
//   radix levels  64 bins x 6 bits per level over the key's static width, most significant digit first: the fallback when
//                 the threshold misses the window, and the whole selection under mxp_set_fused_path(0)
//   emit          keys > T kept, keys == T kept in ascending index until top_k
// Keys are exact integers (score * 2^(-g-1) + offset, read from the low mantissa bits of one FFMA) of up to 22 bits; rows
// beyond that window are flagged and left to the CUDA-core kernel (k_predict_topk_long, row-filtered), which handles any
// exponents.  Pipeline per pass: TMA bulk copy of block j+2 and the MMA of block j+1 run while the threads count block j.
#pragma once
#include "mxprune_predict_tc.cuh"

namespace mxp {

constexpr int KL_T = 512;             // threads per CTA: a pair of query tiles, two lanes per query row
constexpr int KL_TILE = 128;          // query rows per tile
constexpr int KL_BINS = 64;           // bins of a radix level
constexpr int KL_FBINS = 128;         // bins of the fine window (adaptive front end)
constexpr int KL_MAX_RANGE = 1400;    // widest sample key range the fine window takes on
constexpr int KL_WIDE_M = 1 << 21;    // largest |S| bound (in key units) of a row this kernel ranks: every partial sum of the
                                      // score is an integer below 2^22 - exact in fp32 in any order, and the products span
                                      // <= 16 bits, inside the tensor core's measured exact window (profiles/r01_umma_exactness)

// ------------------------------------------------------------------------------------------
// k_quantize_ops: fp32 (B,H,N,hd) view -> MMA-ready bf16 operands in HBM, one thread per MX block.
//   op   exact operand  c * 2^(e-6)   (for the attention kernel; may be null)
//   pp   predictor operand +-2^e
//   ep   predictor exponents  int8 [heads][rows_pad][4]        (query side: row parameters)
//   head_meta u32 [heads][8]: min over keys of (ep_b + 200) and of (200 - ep_b)   (key side)
// which = 0: query layout (tiles of 128 rows), 1: key layout (blocks of OL.kb_rows rows).
// ------------------------------------------------------------------------------------------
struct QuantOpsParams {
    View x;
    int H, N, rows_pad, hd, bf16, flush, which, Nq, Nk;
    unsigned char *op, *pp;
    int8_t* ep;
    uint32_t* head_meta;
    int8_t *codes, *exps;
};

// DT: element type of the view (DT_*)
template <bool CODES, int DT = DT_F32>
__global__ void __launch_bounds__(256)
k_quantize_ops(const QuantOpsParams p) {
    const OpsLayout OL = ops_layout(p.Nq, p.Nk, p.hd);
    const int head = blockIdx.x, bb = head / p.H, hh = head - bb * p.H;
    const int hd = p.hd, nb = (hd + 31) >> 5, nfull = hd >> 5, tail = hd & 31;
    const int kch = OL.hdp >> 3, tail_chunks = kch - 4 * nfull;
    const float* xb = DT == DT_F32 ? p.x.p + bb * p.x.sB + hh * p.x.sH : view_elem<DT>(p.x.p, bb * p.x.sB + hh * p.x.sH);
    const size_t head_bytes = p.which == 0 ? OL.q_head_bytes : OL.k_head_bytes;
    unsigned char* op = p.op ? p.op + (size_t)head * head_bytes : nullptr;
    unsigned char* pp = p.pp + (size_t)head * head_bytes;
    const int ntask = p.rows_pad * nb;                  // rows_pad is a multiple of 128: b is warp-uniform
    for (int t = blockIdx.y * blockDim.x + threadIdx.x; t < ntask; t += gridDim.y * blockDim.x) {
        const int b = t / p.rows_pad, row = t - b * p.rows_pad;
        const bool in_range = row < p.N;
        const bool full = b < nfull;
        const int nd = full ? 32 : tail;
        uint32_t xv[32];
        if constexpr (DT == DT_F32) {
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
                if (in_range && 4 * s < nd) f = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)row * p.x.sN + 32 * b) + s);
                xv[4 * s] = __float_as_uint(f.x); xv[4 * s + 1] = __float_as_uint(f.y);
                xv[4 * s + 2] = __float_as_uint(f.z); xv[4 * s + 3] = __float_as_uint(f.w);
            }
        } else {
            load_block_bits<DT>(view_elem<DT>(xb, (int64_t)row * p.x.sN + 32 * b), nd, in_range, xv);
        }
        BlockQ r;
        quantize_block_thread<CODES>(xv, nd, p.bf16, p.flush, r);
        const int nchunk = full ? 4 : tail_chunks;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            if (ch < nchunk) {
                const size_t off = p.which == 0 ? q_op_offset(OL, row, 4 * b + ch) : k_op_offset(OL, row, 4 * b + ch);
                *reinterpret_cast<uint4*>(pp + off) = in_range ? r.pp[ch] : make_uint4(0u, 0u, 0u, 0u);
                if (op) *reinterpret_cast<uint4*>(op + off) = r.op[ch];
            }
        }
        if (p.ep) p.ep[((size_t)head * p.rows_pad + row) * 4 + b] = (int8_t)r.ep;
        if (p.head_meta) {
            const uint32_t lo = __reduce_min_sync(FULL, in_range ? (uint32_t)(r.ep + 200) : 0xffffffffu);
            const uint32_t hi = __reduce_min_sync(FULL, in_range ? (uint32_t)(200 - r.ep) : 0xffffffffu);
            if ((threadIdx.x & 31) == 0) {
                atomicMin(&p.head_meta[head * 8 + b], lo);
                atomicMin(&p.head_meta[head * 8 + 4 + b], hi);
            }
        }
        if (CODES && p.codes && in_range) {
            const int64_t grow = (int64_t)head * p.N + row;
            p.exps[grow * nb + b] = (int8_t)r.e;
            uint32_t* dst = reinterpret_cast<uint32_t*>(p.codes + grow * hd + 32 * b);
#pragma unroll
            for (int v = 0; v < 8; ++v)
                if (4 * v < nd) dst[v] = r.cw[v];
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_select_long_tc
// ------------------------------------------------------------------------------------------
struct LongSelParams {
    const unsigned char *q_pp, *k_pp;
    const int8_t* q_ep;             // [heads][q_rows_pad][4]
    const uint32_t* head_meta;      // [heads][8]
    uint8_t* flags;                 // [heads][Nq]: 1 = row left to the CUDA-core kernel
    uint32_t* mask;
    int32_t* idx;
    int H, Nq, Nk, hd, top_k;
    int adaptive;                   // 1: sampled fine window in front of the radix levels (see below)
    int splits;                     // CTAs per head (linear grid, a head's CTAs adjacent: its Kp operand stays in L2)
    const float* key_bias;          // BIAS: additive key bias key_bias[b * kb_sB + j] (see k_select_long_tc)
    int64_t kb_sB;
};

struct KLSmem {
    size_t off_k, off_bias, off_hist, off_misc, total;
    int bins;
};
__host__ __device__ inline KLSmem kl_smem_layout(const OpsLayout& O, bool bias = false) {
    KLSmem L;
    size_t o = 2 * O.q_tile_bytes;
    L.off_k = o;    o += 2 * O.k_blk_bytes;
    L.off_bias = o; if (bias) o += 2 * 128 * 4;     // BIAS: bias_j - bmax of two key blocks
    // the fine window wants 128 counters per lane; head dims whose operand tiles leave no room keep 64
    L.bins = (o + (size_t)KL_FBINS * KL_T * 2 + 128 <= (size_t)227 * 1024) ? KL_FBINS : KL_BINS;
    L.off_hist = o; o += (size_t)L.bins * KL_T * 2;
    L.off_misc = o; o += 128;
    L.total = o;
    return L;
}

// gt / eq bit masks of one 32-key window against the row's threshold: keys (c, c + 16) packed per register and compared as
// fp16 bit patterns (one HSET2 per two keys).  Narrow rows (|S| bound <= K1_MAX_M): the key itself, biased into the
// normal fp16 range.  WIDE: the key re-centred on the threshold and clamped, max(min(u - T + 0x4000, 0x7BFF), 0) - one
// VIADDMNMX more per key; the clamp only moves keys that are far from T, so the classification is exact for any width.
template <bool WIDE>
__device__ __forceinline__ void kl_compare_window(const uint32_t (&r)[32], float scl, float cadd, int aw, __half2 t2,
                                                  uint32_t& gt_out, uint32_t& eq_out) {
    uint32_t gt = 0u, eq = 0u;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        uint32_t fl = __float_as_uint(fmaf(__uint_as_float(r[c]), scl, cadd));
        uint32_t fh = __float_as_uint(fmaf(__uint_as_float(r[c + 16]), scl, cadd));
        if (WIDE) {
            fl = (uint32_t)__viaddmin_s32_relu((int)fl, aw, 0x7BFF);
            fh = (uint32_t)__viaddmin_s32_relu((int)fh, aw, 0x7BFF);
        }
        const __half2 kv = u32_as_h2(__byte_perm(fl, fh, 0x5410));
        gt |= __hgt2_mask(kv, t2) & (0x00010001u << c);
        eq |= __heq2_mask(kv, t2) & (0x00010001u << c);
    }
    gt_out = gt;
    eq_out = eq;
}

// BIAS: the 32 scores of one TMEM read (this lane's keys sd[0..31]) -> score + (bias_j - bmax), clamped below at xfloor
// (the value of key 0): keys below the row's window all land on key 0
__device__ __forceinline__ void kl_add_bias(uint32_t (&r)[32], const float* sd, float xfloor) {
#pragma unroll
    for (int c = 0; c < 32; c += 4) {
        const float4 d = *reinterpret_cast<const float4*>(sd + c);
        r[c] = __float_as_uint(fmaxf(__fadd_rn(__uint_as_float(r[c]), d.x), xfloor));
        r[c + 1] = __float_as_uint(fmaxf(__fadd_rn(__uint_as_float(r[c + 1]), d.y), xfloor));
        r[c + 2] = __float_as_uint(fmaxf(__fadd_rn(__uint_as_float(r[c + 2]), d.z), xfloor));
        r[c + 3] = __float_as_uint(fmaxf(__fadd_rn(__uint_as_float(r[c + 3]), d.w), xfloor));
    }
}

// lowest power of two of which the fp32 value x != 0 is a multiple
__device__ __forceinline__ int kl_unit_exp(float x) {
    const uint32_t b = __float_as_uint(x) & 0x7fffffffu;
    const int e = (int)(b >> 23);
    const uint32_t m = e ? ((b & 0x7fffffu) | 0x800000u) : b;
    return (e ? e - 150 : -149) + __ffs((int)m) - 1;
}

// One CTA = one PAIR of 128-row query tiles of one head (16 warps: warps 0-7 the even tile, 8-15 the odd
// one; 512 TMEM columns = two score buffers per tile) sharing every K block it streams.
//
// Adaptive front end (p.adaptive): a radix level resolves 6 bits of a key whose STATIC width is 11-13 bits (up to 22), while a
// row's keys really spread over a few hundred values around a threshold that a sample predicts well.  So: (1) score the first
// 256 keys once (128 below 2048 keys) into the TMEM buffers, take their min / max and a 128-bin histogram, and read off the
// sample's top_k/Nk quantile c; (2) ONE pass over all keys with 126 exact bins for the keys c-63 .. c+62 and two clamp bins;
// if the k-th largest key falls into an exact bin the row has its threshold and tie count, and the emit pass follows: two
// passes instead of three or four.  A row whose sample spreads over more than KL_MAX_RANGE values takes bins of 2^fs keys
// (fs <= 6) and ONE radix level for the fs bits inside the bin (three passes for its pair).  A row whose threshold lands in a
// clamp bin, or whose sample is wider still, sends its tile pair through the radix levels - same result, the old cost.
//
// BIAS (additive key bias, ranked value fl32(pred + bias_j)): the bias is added on the CUDA cores to every score read
// from TMEM, as x = score + d_j with d_j = fl32(bias_j - bmax) (bmax: the batch's largest bias), so the keys stay
// integers of the row's unit 2^(g+1) below the unbiased window's top.  With 2^u the unit of every bias, 2^du that of
// every d_j and m = min(g, u), a row keeps the fast path when du >= g + 1 (integer keys), g <= u + 1 or every d_j is 0
// (the d_j of keys inside the window are exact), and |bmax| and the window's span (2^(g+1) times key 0's offset) are
// <= 2^(23+m) (the reference's pred + bias_j is exact inside the window).  Then every key inside the window equals the
// reference's value up to the constant bmax, and every key below it (x below the value of key 0, e.g. PixArt's -10000
// mask) is also below every key inside it in the reference.  Those keys are clamped to key 0.  A row whose threshold lands on key 0 (fewer than
// top_k keys inside the window) is flagged in the emit pass and re-ranked by the CUDA-core kernel, as rows outside the
// window are.
template <bool BIAS = false>
__global__ void __launch_bounds__(KL_T, 1)
k_select_long_tc(const LongSelParams p) {
    extern __shared__ __align__(1024) unsigned char smem_kl[];
    unsigned char* const smem = smem_kl;
    const int Nk = p.Nk, Nq = p.Nq, hd = p.hd, kk = p.top_k;
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const KLSmem L = kl_smem_layout(O, BIAS);
    const int nb = (hd + 31) >> 5, nblk = O.nblk;
    unsigned char* sQ = smem;
    unsigned char* sK = smem + L.off_k;
    unsigned short* s_hist = reinterpret_cast<unsigned short*>(smem + L.off_hist);
    uint64_t* bar_k = reinterpret_cast<uint64_t*>(smem + L.off_misc);       // [2]
    uint64_t* bar_mma = bar_k + 2;                                          // [2]
    uint64_t* bar_q = bar_k + 4;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_k + 5);
    int* s_nlev = reinterpret_cast<int*>(s_tmem + 1);
    int* s_gen = s_nlev + 1;                            // 1: this tile pair takes the radix levels
    int* s_wide = s_nlev + 2;                           // 1: some row of the pair has keys wider than 15 bits
    int* s_l2 = s_nlev + 3;                             // 1: some row's fine bins hold more than one key value
    uint32_t* s_bmax = reinterpret_cast<uint32_t*>(s_nlev + 4);    // BIAS: order-preserving bits of the largest bias
    int* s_bunit = s_nlev + 5;                          // BIAS: exponent of the coarsest unit every bias is a multiple of
    int* s_dunit = s_nlev + 6;                          // BIAS: the same for every bias_j - bmax
    float* s_d = reinterpret_cast<float*>(smem + L.off_bias);      // BIAS: [2][128] bias_j - bmax of key blocks

    const int head = blockIdx.x / p.splits;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int half = warp >> 3, w8 = warp & 7;          // which tile of the pair; warp within the tile
    const int lane_base = 32 * (w8 & 3) + 16 * (w8 >> 2);
    const int rr = lane_base + (lane & 15);             // row of the tile
    const int part = lane >> 4;                         // keys [64 part, 64 part + 64) of every block
    const unsigned char* q_pp = p.q_pp + (size_t)head * O.q_head_bytes;
    const unsigned char* k_pp = p.k_pp + (size_t)head * O.k_head_bytes;
    const int q_rows_pad = O.q_tiles * KL_TILE;
    const int n_pairs = (O.q_tiles + 1) >> 1;

    if (tid == 0) {
        mbar_init(&bar_k[0], 1); mbar_init(&bar_k[1], 1);
        mbar_init(&bar_mma[0], 1); mbar_init(&bar_mma[1], 1);
        mbar_init(bar_q, 1);
        if (BIAS) { *s_bmax = 0u; *s_bunit = 0x7fffffff; *s_dunit = 0x7fffffff; }
    }
    if (warp == 0) tmem_alloc(s_tmem, 512u);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    const uint32_t tmem = *s_tmem;
    const float* const bias_b = BIAS ? p.key_bias + (head / p.H) * p.kb_sB : nullptr;
    float bmax = 0.f;
    int bunit = 0x7fffffff, dunit = 0x7fffffff;
    if (BIAS) {                                          // the batch's largest bias and the units of the biases / d_j
        uint32_t mx = 0u;
        int un = 0x7fffffff;
        for (int j = tid; j < Nk; j += KL_T) {
            const float b = __ldg(bias_b + j);
            const uint32_t u = __float_as_uint(b);
            mx = max(mx, (u & 0x80000000u) ? ~u : u | 0x80000000u);
            if (b != 0.f) un = min(un, kl_unit_exp(b));
        }
        mx = __reduce_max_sync(FULL, mx);
        un = __reduce_min_sync(FULL, un);
        if (lane == 0) { atomicMax(s_bmax, mx); atomicMin(s_bunit, un); }
        __syncthreads();
        const uint32_t m = *s_bmax;
        bmax = __uint_as_float((m & 0x80000000u) ? m & 0x7fffffffu : ~m);
        bunit = *s_bunit;
        int du = 0x7fffffff;
        for (int j = tid; j < Nk; j += KL_T) {
            const float d = __fsub_rn(__ldg(bias_b + j), bmax);
            if (d != 0.f) du = min(du, kl_unit_exp(d));
        }
        du = __reduce_min_sync(FULL, du);
        if (lane == 0) atomicMin(s_dunit, du);
        __syncthreads();
        dunit = *s_dunit;
    }
    // BIAS: bias_j - bmax of key block blk -> s_d[(blk & 1) * 128 ..] (keys past Nk: 0, the score of Kp's zero rows)
    auto stage_bias = [&](int blk) {
        if (tid < 128) {
            const int j = blk * 128 + tid;
            s_d[(blk & 1) * 128 + tid] = j < Nk ? __fsub_rn(__ldg(bias_b + j), bmax) : 0.f;
        }
    };
    const uint32_t my_lane = (uint32_t)lane_base << 16;
    const uint32_t my_col = (uint32_t)(half * 256);     // this tile's two 128-column score buffers
    const uint32_t idesc = umma_idesc_bf16_f32(128, 128);
    uint32_t ph_k = 0u, ph_m = 0u, ph_q = 0u;           // bit s = phase of barrier s (registers, not a local array)

    int kmin[4], spread[4];
    bool wide = false;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        kmin[b] = b < nb ? (int)p.head_meta[head * 8 + b] - 200 : 0;
        const int kmax = b < nb ? 200 - (int)p.head_meta[head * 8 + 4 + b] : 0;
        spread[b] = kmax - kmin[b];
        wide |= spread[b] > K1_MAX_SPREAD;
    }
    const int NW = (Nk + 31) >> 5;
    // zero rows of Kp (score exactly 0) among THIS lane's key columns: only the last block has any
    const int last0 = (nblk - 1) * 128 + 64 * part;
    const int my_npad = max(0, min(64, last0 + 64 - Nk));
    // u16 counters, bin b of a thread at [b * KL_T + slot]: the 32 lanes of a warp sit in 32 different
    // 32-bit words (banks) - two warps interleave the half-words - so the per-key read-modify-writes of
    // a warp never conflict, whatever bins its lanes hit
    const int hslot = (warp >> 1) * 64 + 2 * lane + (warp & 1);
    unsigned short* my_hist = s_hist + hslot;           // bin b at my_hist[b * KL_T]
    const unsigned short* their_hist = s_hist + ((warp >> 1) * 64 + 2 * (lane ^ 16) + (warp & 1));

    for (int pt = blockIdx.x % p.splits; pt < n_pairs; pt += p.splits) {
        const int nh = 2 * pt + 1 < O.q_tiles ? 2 : 1;  // tiles of this pair
        const int tile = 2 * pt + half;
        const int i = tile * KL_TILE + rr;
        const bool valid = half < nh && i < Nq;
        const int64_t row = (int64_t)head * Nq + (valid ? i : 0);
        if (tid == 0) {
            *s_nlev = 0;
            *s_wide = 0;
            *s_l2 = 0;
            *s_gen = (p.adaptive && L.bins == KL_FBINS) ? 0 : 1;
            mbar_expect_tx(bar_q, (uint32_t)(nh * O.q_tile_bytes));
            tma_bulk_g2s(sQ, q_pp + (size_t)(2 * pt) * O.q_tile_bytes, (uint32_t)(nh * O.q_tile_bytes), bar_q);
        }
        // K block in sK[s] x the pair's query tiles -> score buffer s of each tile (thread 0 only)
        auto issue_mma = [&](int s) {
            tcgen05_fence_after_sync();
            const unsigned char* kb = sK + (size_t)s * O.k_blk_bytes;
            for (int h = 0; h < nh; ++h) {
                const unsigned char* qt = sQ + (size_t)h * O.q_tile_bytes;
                for (int ks = 0; ks < (O.hdp >> 4); ++ks) {
                    const uint64_t da = umma_smem_desc(smem_u32(qt + (size_t)(2 * ks) * KL_TILE * 16), KL_TILE * 16, 128);
                    const uint64_t db = umma_smem_desc(smem_u32(kb + (size_t)(2 * ks) * 128 * 16), 128 * 16, 128);
                    umma_bf16_ss(tmem + (uint32_t)(h * 256 + s * 128), da, db, idesc, ks > 0);
                }
            }
            umma_commit(&bar_mma[s]);
        };
        // ---- integer-key parameters of this thread's row (same window rules as the short kernels)
        int epq[4];
        {
            const int8_t* e4 = p.q_ep + ((size_t)head * q_rows_pad + (half < nh ? i : 0)) * 4;
#pragma unroll
            for (int b = 0; b < 4; ++b) epq[b] = b < nb ? (int)e4[b] : 0;
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
        if (M > KL_WIDE_M) fast = false;
        if (BIAS && fast) {
            const int mu = min(g, bunit);
            const float span = (float)((((int)M + 1) >> 1) + 1) * exp2i(g + 1);      // key 0's offset x 2^(g+1)
            const float lim = 23 + mu < -126 ? 0.f : exp2i(min(23 + mu, 127));
            if (dunit < g + 1 || (dunit != 0x7fffffff && g > bunit + 1) || !(fabsf(bmax) <= lim) || !(span <= lim))
                fast = false;
        }
        const bool narrow = M <= K1_MAX_M;                          // keys fit the 15-bit fp16 patterns of the short kernels
        if (valid && part == 0) p.flags[row] = fast ? 0 : 1;
        if (!fast) M = 0;
        const int moff = ((int)M + 1) & ~1;
        const float scl = fast ? exp2i(-g - 1) : 0.f;
        // BIAS: the score value of key 0 (scores clamp there); any value for other rows (scl = 0)
        const float xfloor = fast ? -(float)((moff >> 1) + 1) * exp2i(g + 1) : 0.f;
        // histogram passes rank on the plain key u = S/2 + moff/2 + 1 (fewest digits); the emit pass adds
        // the fp16 bias of the short kernel so that two keys per word compare with one HSET2
        const uint32_t key0 = (uint32_t)((moff >> 1) + 1);          // key of a score of exactly 0
        const float cadd = 8388608.0f + (float)key0;
        const float cadd_e = cadd + (float)K1_KEY_BIAS;
        const int wtot = 32 - __clz(moff + 1);                      // key width in bits
        const int my_lev = (wtot + 5) / 6;
        __syncthreads();                                            // *s_nlev = 0 visible
        {
            const int wl = __reduce_max_sync(FULL, fast ? my_lev : 0);
            const bool ww = __any_sync(FULL, fast && !narrow);
            if (lane == 0) {
                atomicMax(s_nlev, wl);
                if (ww) atomicOr(s_wide, 1);
            }
        }
        __syncthreads();
        const int nlev = *s_nlev;
        const bool wide_pair = *s_wide != 0;
        mbar_wait(bar_q, ph_q);
        ph_q ^= 1u;

        // ---- adaptive front end, step 1: the sample (key blocks 0 and 1 - block 0 alone for short rows - scored once
        // into the score buffers); worth it when sample (~2.5 block steps per sampled block) + fine + emit beat the
        // nlev + 1 passes of the radix select
        const int nsamp = nblk >= 16 ? 2 : 1;                      // measured: N = 1024 better with one block, 2048 with two
        bool adapt = nlev > 0 && *s_gen == 0 && 5 * nsamp + 4 * nblk < 2 * (nlev + 1) * nblk;
        int lo_key = 0, fs = 0;                                     // fine bin e <-> keys [lo_key + (e << fs), + 2^fs)
        if (adapt) {
            if (BIAS) {
                for (int b = 0; b < nsamp; ++b) stage_bias(b);
                __syncthreads();
            }
            if (tid == 0) {
                for (int b = 0; b < nsamp; ++b) {
                    mbar_expect_tx(&bar_k[b], (uint32_t)O.k_blk_bytes);
                    tma_bulk_g2s(sK + (size_t)b * O.k_blk_bytes, k_pp + (size_t)b * O.k_blk_bytes, (uint32_t)O.k_blk_bytes, &bar_k[b]);
                }
            }
            for (int b = 0; b < nsamp; ++b) {
                mbar_wait(&bar_k[b], (ph_k >> b) & 1u);
                ph_k ^= 1u << b;
                if (tid == 0) issue_mma(b);
            }
            for (int b = 0; b < nsamp; ++b) {
                mbar_wait(&bar_mma[b], (ph_m >> b) & 1u);
                ph_m ^= 1u << b;
            }
            tcgen05_fence_after_sync();
            const bool any_fast = __any_sync(FULL, fast);
            const uint32_t tbase = tmem + my_lane + my_col;
            float fmn = 3.0e38f, fmx = 0.f;
            if (any_fast) {
#pragma unroll 1
                for (int q4 = 0; q4 < 2 * nsamp; ++q4) {                    // buffer q4 >> 1, this lane's columns 32 (q4 & 1) + c
                    uint32_t r[32];
                    tmem_ld_16x32bx2_s64_x32(tbase + (q4 >> 1) * 128 + (q4 & 1) * 32, r);
                    tmem_ld_wait();
                    if (BIAS) kl_add_bias(r, s_d + (q4 >> 1) * 128 + 64 * part + 32 * (q4 & 1), xfloor);
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const float f = fmaf(__uint_as_float(r[c]), scl, cadd);
                        fmn = fminf(fmn, f);
                        fmx = fmaxf(fmx, f);
                    }
                }
            }
            fmn = fminf(fmn, __shfl_xor_sync(FULL, fmn, 16));
            fmx = fmaxf(fmx, __shfl_xor_sync(FULL, fmx, 16));
            const int umin = (int)(__float_as_uint(fmn) & 0x7fffffu), umax = (int)(__float_as_uint(fmx) & 0x7fffffu);
            const int range = fast ? umax - umin : 0;
            const int csh = 32 - __clz(range >> 7);                 // (range >> csh) < 128
            for (int b = 0; b < KL_FBINS; ++b) my_hist[b * KL_T] = 0;
            if (any_fast) {
#pragma unroll 1
                for (int q4 = 0; q4 < 2 * nsamp; ++q4) {
                    uint32_t r[32];
                    tmem_ld_16x32bx2_s64_x32(tbase + (q4 >> 1) * 128 + (q4 & 1) * 32, r);
                    tmem_ld_wait();
                    if (BIAS) kl_add_bias(r, s_d + (q4 >> 1) * 128 + 64 * part + 32 * (q4 & 1), xfloor);
                    if (fast) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            const int u = (int)(__float_as_uint(fmaf(__uint_as_float(r[c]), scl, cadd)) & 0x7fffffu);
                            my_hist[((u - umin) >> csh) * KL_T] += 1;
                        }
                    }
                }
            }
            __syncwarp();                                           // the partner lane's column is complete
            if (fast) {
                const int ks = max(1, (kk * 128 * nsamp + (Nk >> 1)) / Nk);    // the sample's share of top_k
                int cum = 0, bin = KL_FBINS - 1;
                for (; bin > 0; --bin) {
                    const int h = (int)my_hist[bin * KL_T] + (int)their_hist[bin * KL_T];
                    if (cum + h >= ks) break;
                    cum += h;
                }
                // bins of one key value while the sample spreads over <= KL_MAX_RANGE values; beyond that bins of 2^fs
                // values (window >= 0.18 of the sample range) and one more level for the digit inside the bin
                if (range > KL_MAX_RANGE) fs = 32 - __clz(range / (KL_MAX_RANGE / 2));
                const int c_est = umin + (bin << csh) + ((1 << csh) >> 1);
                lo_key = ((c_est >> fs) - KL_FBINS / 2) << fs;
                if (fs > 6) atomicOr(s_gen, 1);                     // too wide even so: radix levels
                else if (fs > 0) atomicOr(s_l2, 1);
            }
            tcgen05_fence_before_sync();
            __syncthreads();                                        // score buffers free again; *s_gen final
            adapt = *s_gen == 0;
        }
        const bool pair_l2 = adapt && *s_l2 != 0;
        const int lo_sh = (0x4B000000 + lo_key) >> fs;              // (bits of 2^23 + lo_key) >> fs; lo_key is a multiple of 2^fs

        uint32_t prefix = 0u;
        int krem = kk;
        // pass sequence of the pair (uniform): [fine window -> (one level for the digit inside a bin)] or
        // [nlev radix levels], then emit; no pass at all when no row of the pair is fast.  A level counts digit
        // (u >> lo_cur) & (2^dbits - 1) among the keys whose higher bits equal prefix (per-thread lo_cur / dbits).
        enum { P_FINE, P_LEVEL, P_EMIT, P_DONE };
        int kind = nlev == 0 ? P_DONE : (adapt ? P_FINE : P_LEVEL);
        int levels_left = nlev;
        bool first_level = true;                                    // first radix level: no prefix yet, every key counts
        int lo_cur = 6 * (my_lev - 1), dbits = 6;
        while (kind != P_DONE) {
            const bool fine = kind == P_FINE;
            const bool emit = kind == P_EMIT;
            const int lo = lo_cur;                                  // < 0: this row already has its full key
            const bool counting = fine ? fast : (!emit && fast && lo >= 0);
            const uint32_t dmask = (1u << dbits) - 1u;
            if (!emit) {
                const int nbins = fine ? KL_FBINS : KL_BINS;
                for (int b = 0; b < nbins; ++b) my_hist[b * KL_T] = 0;
            }
            int rem = krem, pos = 0;                                // emit state (identical in both lanes)
            // BIAS: a threshold on key 0 lies among the clamped keys: the row goes to the CUDA-core kernel
            if (BIAS && emit && valid && fast && part == 0 && prefix == 0u) p.flags[row] = 1;
            // emit compares fp16 patterns: the biased key against T + bias, or (wide pair) the key re-centred on T against 0x4000
            const uint32_t T = wide_pair ? 0x4000u : prefix + K1_KEY_BIAS;
            const int aw = 0x4000 - (0x4B000000 + (int)prefix);
            if (tid == 0) {
                const int pre = min(2, nblk);
                for (int b = 0; b < pre; ++b) {
                    mbar_expect_tx(&bar_k[b], (uint32_t)O.k_blk_bytes);
                    tma_bulk_g2s(sK + (size_t)b * O.k_blk_bytes, k_pp + (size_t)b * O.k_blk_bytes, (uint32_t)O.k_blk_bytes, &bar_k[b]);
                }
            }
            for (int it = 0; it <= nblk; ++it) {
                // BIAS: block it's buffer was last read in iteration it - 1, which ended with a barrier
                if (BIAS && it < nblk) stage_bias(it);
                if (it < nblk) {
                    const int s = it & 1;
                    mbar_wait(&bar_k[s], (ph_k >> s) & 1u);
                    ph_k ^= 1u << s;
                    if (tid == 0) issue_mma(s);
                }
                if (it > 0) {
                    const int j = it - 1, s = j & 1;
                    mbar_wait(&bar_mma[s], (ph_m >> s) & 1u);
                    ph_m ^= 1u << s;
                    tcgen05_fence_after_sync();
                    if (tid == 0 && j + 2 < nblk) {                 // MMA j has finished reading sK[s]
                        mbar_expect_tx(&bar_k[s], (uint32_t)O.k_blk_bytes);
                        tma_bulk_g2s(sK + (size_t)s * O.k_blk_bytes, k_pp + (size_t)(j + 2) * O.k_blk_bytes,
                                     (uint32_t)O.k_blk_bytes, &bar_k[s]);
                    }
                    const uint32_t tbase = tmem + my_lane + my_col + (uint32_t)(s * 128);
                    if (!emit) {
                        if (__any_sync(FULL, counting)) {
#pragma unroll 1
                            for (int q2 = 0; q2 < 2; ++q2) {        // this lane's keys 64 part + 32 q2 + c
                                uint32_t r[32];
                                tmem_ld_16x32bx2_s64_x32(tbase + q2 * 32, r);
                                tmem_ld_wait();
                                if (BIAS) kl_add_bias(r, s_d + s * 128 + 64 * part + 32 * q2, xfloor);
                                if (counting) {
                                    // fine window: bin = clamp((key - lo_key) >> fs, 0, 127), one VIADDMNMX.  The counter
                                    // updates go in PAIRS - both loads issued before either store, the second store adding
                                    // 2 when the bins coincide - so that two shared-memory round trips overlap (the loop is
                                    // bound by that latency, not by issue slots)
                                    if (fine && !pair_l2) {
#pragma unroll
                                        for (int c = 0; c < 32; c += 2) {
                                            const int e0 = __viaddmin_s32_relu(__float_as_int(fmaf(__uint_as_float(r[c]), scl, cadd)), -lo_sh, KL_FBINS - 1);
                                            const int e1 = __viaddmin_s32_relu(__float_as_int(fmaf(__uint_as_float(r[c + 1]), scl, cadd)), -lo_sh, KL_FBINS - 1);
                                            const unsigned short v0 = my_hist[e0 * KL_T], v1 = my_hist[e1 * KL_T];
                                            my_hist[e0 * KL_T] = (unsigned short)(v0 + 1);
                                            my_hist[e1 * KL_T] = (unsigned short)(v1 + (e0 == e1 ? 2 : 1));
                                        }
                                    } else if (fine) {              // bins of 2^fs keys (per row)
#pragma unroll
                                        for (int c = 0; c < 32; c += 2) {
                                            const int e0 = __viaddmin_s32_relu(__float_as_int(fmaf(__uint_as_float(r[c]), scl, cadd)) >> fs, -lo_sh, KL_FBINS - 1);
                                            const int e1 = __viaddmin_s32_relu(__float_as_int(fmaf(__uint_as_float(r[c + 1]), scl, cadd)) >> fs, -lo_sh, KL_FBINS - 1);
                                            const unsigned short v0 = my_hist[e0 * KL_T], v1 = my_hist[e1 * KL_T];
                                            my_hist[e0 * KL_T] = (unsigned short)(v0 + 1);
                                            my_hist[e1 * KL_T] = (unsigned short)(v1 + (e0 == e1 ? 2 : 1));
                                        }
                                    } else if (first_level) {       // no prefix yet: every key counts
#pragma unroll
                                        for (int c = 0; c < 32; ++c) {
                                            const uint32_t u = __float_as_uint(fmaf(__uint_as_float(r[c]), scl, cadd));
                                            my_hist[((u >> lo) & 63u) * KL_T] += 1;
                                        }
                                    } else {
#pragma unroll
                                        for (int c = 0; c < 32; ++c) {
                                            const uint32_t u = __float_as_uint(fmaf(__uint_as_float(r[c]), scl, cadd)) & 0x7fffffu;
                                            if ((u >> (lo + dbits)) == prefix) my_hist[((u >> lo) & dmask) * KL_T] += 1;
                                        }
                                    }
                                }
                            }
                        }
                    } else {
                        // two words of 32 keys per lane and block, keys (c, c + 16) packed per register and
                        // compared as fp16 bit patterns; ties are taken in ascending key index: the lower
                        // lane's 64 keys come first, so the lanes exchange their tie counts per block
                        const __half2 t2 = u32_as_h2(T * 0x00010001u);
                        uint32_t gtw[2], eqw[2];
#pragma unroll
                        for (int q2 = 0; q2 < 2; ++q2) {
                            uint32_t r[32];
                            tmem_ld_16x32bx2_s64_x32(tbase + q2 * 32, r);
                            tmem_ld_wait();
                            if (BIAS) kl_add_bias(r, s_d + s * 128 + 64 * part + 32 * q2, xfloor);
                            uint32_t gt, eq;
                            if (wide_pair) kl_compare_window<true>(r, scl, cadd, aw, t2, gt, eq);
                            else kl_compare_window<false>(r, scl, cadd_e, 0, t2, gt, eq);
                            const int nv = Nk - (j * 128 + 64 * part + 32 * q2);
                            const uint32_t vm = nv >= 32 ? 0xffffffffu : (nv <= 0 ? 0u : (1u << nv) - 1u);
                            gtw[q2] = gt & vm;
                            eqw[q2] = eq & vm;
                        }
                        const int ties_m = __popc(eqw[0]) + __popc(eqw[1]);
                        const int ties_o = __shfl_xor_sync(FULL, ties_m, 16);
                        int r_here = part == 0 ? rem : max(rem - ties_o, 0);        // ties still wanted at my first key
                        rem = max(rem - ties_m - ties_o, 0);
                        uint32_t word[2];
#pragma unroll
                        for (int q2 = 0; q2 < 2; ++q2) {
                            const int cnt = __popc(eqw[q2]);
                            uint32_t take = eqw[q2];
                            if (cnt > r_here) take = keep_lowest_bits_fast(eqw[q2], r_here);
                            r_here -= min(cnt, r_here);
                            word[q2] = gtw[q2] | take;
                        }
                        const int kept_m = __popc(word[0]) + __popc(word[1]);
                        const int kept_o = __shfl_xor_sync(FULL, kept_m, 16);
                        int pos_here = pos + (part == 0 ? 0 : kept_o);
                        pos += kept_m + kept_o;
                        if (valid && fast) {
#pragma unroll
                            for (int q2 = 0; q2 < 2; ++q2) {
                                const int j0 = j * 128 + 64 * part + 32 * q2;
                                if ((j0 >> 5) < NW) {
                                    p.mask[row * NW + (j0 >> 5)] = word[q2];
                                    if (p.idx) {
                                        uint32_t w2 = word[q2];
                                        while (w2) {
                                            const int bpos = __ffs(w2) - 1;
                                            w2 &= w2 - 1u;
                                            p.idx[row * kk + pos_here++] = j0 + bpos;
                                        }
                                    }
                                }
                            }
                        }
                    }
                }
                tcgen05_fence_before_sync();
                __syncthreads();                                    // TMEM buffer of block j is free again
            }
            if (fine) {
                // the zero rows of Kp all scored key0: discount them (each lane its own columns)
                if (counting && my_npad > 0)
                    my_hist[__viaddmin_s32_relu((0x4B000000 + (int)key0) >> fs, -lo_sh, KL_FBINS - 1) * KL_T] -= (unsigned short)my_npad;
                __syncwarp();                                       // the partner lane's column is complete
                int cum = 0, bin = KL_FBINS - 1;
                if (counting) {
                    for (; bin > 0; --bin) {
                        const int h = (int)my_hist[bin * KL_T] + (int)their_hist[bin * KL_T];
                        if (cum + h >= kk) break;
                        cum += h;
                    }
                    if (bin == 0 || bin == KL_FBINS - 1) atomicOr(s_gen, 1);    // threshold in a clamp bin
                }
                __syncthreads();                                    // (also: both lanes have scanned)
                if (*s_gen == 0) {                                  // every row of the pair has its threshold bin
                    prefix = (uint32_t)((lo_key >> fs) + bin);      // = key >> fs
                    krem = kk - cum;
                    first_level = false;
                    lo_cur = fs > 0 ? 0 : -1;                       // rows with wider bins: one level for the low fs bits
                    dbits = fs;
                    levels_left = 1;
                    kind = pair_l2 ? P_LEVEL : P_EMIT;
                } else {
                    kind = P_LEVEL;                                 // the radix levels, from the top
                }
            } else if (!emit) {
                // the zero rows of Kp all scored key0: discount them (each lane its own columns)
                if (counting && my_npad > 0 && (key0 >> (lo + dbits)) == prefix)
                    my_hist[((key0 >> lo) & dmask) * KL_T] -= (unsigned short)my_npad;
                __syncwarp();                                       // the partner lane's column is complete
                if (counting) {
                    int cum = 0, bin = (int)dmask;
                    for (; bin > 0; --bin) {
                        const int h = (int)my_hist[bin * KL_T] + (int)their_hist[bin * KL_T];
                        if (cum + h >= krem) break;
                        cum += h;
                    }
                    krem -= cum;
                    prefix = (prefix << dbits) | (uint32_t)bin;
                }
                __syncwarp();                                       // both lanes have scanned before the next zeroing
                first_level = false;
                lo_cur -= 6;
                if (--levels_left == 0) kind = P_EMIT;
            } else {
                kind = P_DONE;
            }
        }
    }
    tcgen05_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512u);
}

}  // namespace mxp
