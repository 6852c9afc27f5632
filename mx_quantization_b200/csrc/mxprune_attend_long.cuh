// K2-long-pair: exact MXINT8 attention over the kept keys for Nk > 256 (config C5, the sequence-length sweep) with TWO
// LANES PER QUERY ROW and a pipelined key-block stream.  The key blocks of 128 (OpsLayout) are streamed twice per query
// tile: pass 1 forms the row maximum and sum with an online softmax, pass 2 recomputes S on the tensor core to form P
// and accumulate O in its own TMEM columns.  256 threads per CTA, two CTAs per SM (256 TMEM columns each):
//   * a warp owns 16 query rows (TMEM lanes), lanes l and l + 16 share row l; of a block's four 32-key windows lane
//     half h takes windows 2h and 2h + 1 (tcgen05.ld.16x32bx2, column split 64).  Each lane keeps its own running
//     maximum / sum over its columns; the row's two halves are combined once, after the last block.
//   * pass 1 (row max and sum of exp over the kept keys): K blocks arrive by TMA two ahead (the V region is idle in
//     this pass and serves as the second K buffer), S = Q.K_blk^T is issued one block ahead into one of two TMEM
//     buffers (the O columns are idle in this pass), so the tensor core and the copies run under the epilogue.
//   * pass 2 (P = exp(t - max) / sum -> A1 -> MXINT8 per window -> bf16 operand, O += P_blk . V_blk): the Q tile
//     keeps its own region (no re-fetch per block), V blocks are double-buffered, K(blk + 1) is fetched as soon as
//     S(blk) is complete and S(blk + 1) is issued right behind the P.V MMAs of block blk.
// Reference semantics: workloads/DiT/models.py:168-225 at N > 256 (gather -> softmax over the kept keys -> scatter ->
// mx.matmul(attn, v)), as k_attend_pair for Nk <= 256.
#pragma once
#include "mxprune_attend.cuh"

namespace mxp {

struct KLPSmem {
    size_t off_v0, off_v1, off_p, off_q, total;
};
__host__ __device__ inline KLPSmem klp_smem_layout(const OpsLayout& O) {
    KLPSmem L;
    size_t o = O.k_blk_bytes;                   // K block (pass 1: buffer 0)
    L.off_v0 = o; o += O.v_blk_bytes;           // V buffer 0 (pass 1: K buffer 1 - the two block sizes are equal)
    L.off_v1 = o; o += O.v_blk_bytes;           // V buffer 1
    L.off_p = o;  o += K2_P_BYTES;              // P operand of a block (4 windows); O staging at the end
    L.off_q = o;  o += O.q_tile_bytes;          // the Q tile, resident for the whole tile
    L.total = o;
    return L;
}

// OT: output element type (DT_*).  BIAS: p.key_bias is set - t = fl32(fl32(s * scale) + bias_j) as in k_attend_pair.
// The bias is read through the read-only cache (a lane's 32 keys of a window are consecutive), not staged: shared
// memory for it would cost the second CTA per SM at head_dim 72 / 80
template <bool BF16, int OT = DT_F32, bool BIAS = false>
__global__ void __launch_bounds__(K2P_T, 2)
k_attend_long_pair(const AttnParams p) {
    extern __shared__ __align__(128) unsigned char smem_klp[];
    __shared__ uint64_t bar_k[2], bar_v[2], bar_s[2], bar_o, bar_q;
    __shared__ uint32_t tmem_base_s;
    constexpr bool bf16 = BF16;
    const int Nk = p.Nk, Nq = p.Nq, hd = p.hd;
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    const KLPSmem L = klp_smem_layout(O);
    const int hdp = O.hdp, NW = O.nw, nblk = O.nblk;
    unsigned char* const smem = smem_klp;
    // K buffers of pass 1: the K region and V buffer 0 (equal block sizes); V buffers of pass 2
    auto sKb = [&](int b) { return smem + (size_t)b * L.off_v0; };
    auto sVb = [&](int b) { return smem + L.off_v0 + (size_t)b * (L.off_v1 - L.off_v0); };
    unsigned char* const sP = smem + L.off_p;
    unsigned char* const sQ = smem + L.off_q;
    // linear grid, query tile fastest: the CTAs resident at one time belong to a handful of heads, whose K / V operands
    // (streamed twice / once per tile) then come from L2 - head-fastest order had every head's operands in flight at once
    // (ncu at N = 4096: 16 GB of DRAM reads for 0.7 GB of operands)
    const int head = blockIdx.x / O.q_tiles, bb = head / p.H, hh = head % p.H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int lane_base = 32 * (warp & 3) + 16 * (warp >> 2);
    const int rr = lane_base + (lane & 15);                         // row of the tile
    const int part = lane >> 4;                                     // windows 2 part, 2 part + 1 of every block
    const bool flush = p.flush != 0;
    const float scale = p.scale;
    const unsigned char* q_op = p.q_op + (size_t)head * O.q_head_bytes;
    const unsigned char* k_op = p.k_op + (size_t)head * O.k_head_bytes;
    const unsigned char* v_op = p.v_op + (size_t)head * O.v_head_bytes;
    float* out_head = out_elem(p.out, bb * p.o_sB + hh * p.o_sH, OT != DT_F32);
    const uint32_t kbytes = (uint32_t)O.k_blk_bytes, vbytes = (uint32_t)O.v_blk_bytes;
    const float* const bias_b = BIAS ? p.key_bias + bb * p.kb_sB : nullptr;
    // BIAS: bias of key j (keys past Nk read the last key's; they are never kept)
    auto bias_at = [&](int j) { return __ldg(bias_b + min(j, Nk - 1)); };

    if (tid == 0) {
        mbar_init(&bar_k[0], 1); mbar_init(&bar_k[1], 1);
        mbar_init(&bar_v[0], 1); mbar_init(&bar_v[1], 1);
        mbar_init(&bar_s[0], 1); mbar_init(&bar_s[1], 1);
        mbar_init(&bar_o, 1); mbar_init(&bar_q, 1);
    }
    if (warp == 0) tmem_alloc(&tmem_base_s, 256u);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    const uint32_t tmem = tmem_base_s;
    const uint32_t my_tmem = tmem + ((uint32_t)lane_base << 16);
    const uint32_t o_col = 128u;
    const uint32_t idesc_s = umma_idesc_bf16_f32(128, 128);
    const uint32_t idesc_o = umma_idesc_bf16_f32(128, hdp);
    uint32_t ph_k = 0u, ph_v = 0u, ph_s = 0u, ph_o = 0u, ph_q = 0u;      // ph_k / ph_v / ph_s: bit b = phase of barrier b

    auto issue_s = [&](const unsigned char* kb, uint32_t dcol, uint64_t* bar) {      // one thread: S = Q . K_blk^T
        tcgen05_fence_after_sync();
        for (int ks = 0; ks < (hdp >> 4); ++ks) {
            const uint64_t da = umma_smem_desc(smem_u32(sQ + (size_t)(2 * ks) * K2T * 16), K2T * 16, 128);
            const uint64_t db = umma_smem_desc(smem_u32(kb + (size_t)(2 * ks) * 128 * 16), 128 * 16, 128);
            umma_bf16_ss(tmem + dcol, da, db, idesc_s, ks > 0);
        }
        umma_commit(bar);
    };

    for (int tile = blockIdx.x % O.q_tiles; tile < O.q_tiles; tile += O.q_tiles) {      // one tile per CTA
        const int i = tile * K2T + rr;
        const bool valid = i < Nq;
        const uint32_t* mrow = p.mask + ((size_t)head * Nq + (valid ? i : 0)) * NW;

        // ================= pass 1: running max / sum of exp over this lane's kept keys
        if (tid == 0) {
            mbar_expect_tx(&bar_q, (uint32_t)O.q_tile_bytes);
            tma_bulk_g2s(sQ, q_op + (size_t)tile * O.q_tile_bytes, (uint32_t)O.q_tile_bytes, &bar_q);
            for (int b = 0; b < 2 && b < nblk; ++b) {
                mbar_expect_tx(&bar_k[b], kbytes);
                tma_bulk_g2s(sKb(b), k_op + (size_t)b * kbytes, kbytes, &bar_k[b]);
            }
            mbar_wait(&bar_q, ph_q);
            mbar_wait(&bar_k[0], (ph_k >> (0)) & 1u);
            issue_s(sKb(0), 0u, &bar_s[0]);
        }
        ph_q ^= 1u;
        ph_k ^= 1u << (0);
        float m = -INFINITY, l = 0.f;
        for (int blk = 0; blk < nblk; ++blk) {
            const int s = blk & 1;
            const int kb = blk * 128 + 64 * part;                   // key of this lane's column 0
            // S(blk + 1) into the other TMEM buffer (its last reader, the epilogue of blk - 1, ended with a barrier)
            if (blk + 1 < nblk) {
                if (tid == 0) {
                    mbar_wait(&bar_k[s ^ 1], (ph_k >> (s ^ 1)) & 1u);
                    issue_s(sKb(s ^ 1), (uint32_t)((s ^ 1) * 128), &bar_s[s ^ 1]);
                }
                ph_k ^= 1u << (s ^ 1);
            }
            uint32_t mw[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int w = 4 * blk + 2 * part + j;
                mw[j] = (valid && w < NW) ? __ldg(mrow + w) : 0u;
            }
            mbar_wait(&bar_s[s], (ph_s >> (s)) & 1u);                          // S(blk) complete: its K buffer is free
            ph_s ^= 1u << (s);
            tcgen05_fence_after_sync();
            if (tid == 0 && blk + 2 < nblk) {
                mbar_expect_tx(&bar_k[s], kbytes);
                tma_bulk_g2s(sKb(s), k_op + (size_t)(blk + 2) * kbytes, kbytes, &bar_k[s]);
            }
            const uint32_t sb = my_tmem + (uint32_t)(s * 128);
            // one TMEM read per window: t = bf16?(s) * scale (A7) stays in registers between the maximum over the kept keys
            // and the exponentials; the running maximum / sum are updated window by window (online softmax)
#pragma unroll 1
            for (int j = 0; j < 2; ++j) {
                uint32_t r[32];
                tmem_ld_16x32bx2_s64_x32(sb + 32 * j, r);
                tmem_ld_wait();
                const uint32_t mwj = j ? mw[1] : mw[0];
                float mb4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
                for (int c = 0; c < 32; ++c) {                      // dropped keys become -inf: no part in the maximum, exp = 0
                    float sv = __uint_as_float(r[c]);
                    if (bf16) sv = bf16_half_away(sv);
                    float ts = __fmul_rn(sv, scale);
                    if (BIAS) ts = __fadd_rn(ts, bias_at(kb + 32 * j + c));
                    const float tv = ((mwj >> c) & 1u) ? ts : -INFINITY;
                    r[c] = __float_as_uint(tv);
                    mb4[c & 3] = fmaxf(mb4[c & 3], tv);
                }
                const float mb = fmaxf(fmaxf(mb4[0], mb4[1]), fmaxf(mb4[2], mb4[3]));
                const float m_new = fmaxf(m, mb);
                const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
                if (m != -INFINITY && m_new != m) l *= exp_nonpos(m - m_use);
                // 2^((t - m) log2 e) straight from MUFU.EX2 (exp_fast_nonpos: <= 2 ulp per term, the argument error
                // grows with |t - m|, i.e. only where the term no longer matters), a third of exp_nonpos's instructions
                float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int c = 0; c < 32; ++c) {
                    sum4[c & 3] += exp_fast_nonpos(__fsub_rn(__uint_as_float(r[c]), m_use));
                }
                l += (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
                m = m_new;
            }
            tcgen05_fence_before_sync();
            __syncthreads();                                        // every lane has read S(blk): its TMEM buffer is free
        }
        // the row's two halves -> row maximum and row sum
        const float m_o = __shfl_xor_sync(FULL, m, 16), l_o = __shfl_xor_sync(FULL, l, 16);
        const float m_row = fmaxf(m, m_o);
        const float m_fin = (m_row == -INFINITY) ? 0.f : m_row;
        float l_row = 0.f;
        if (m != -INFINITY) l_row = l * exp_nonpos(m - m_fin);
        if (m_o != -INFINITY) l_row += l_o * exp_nonpos(m_o - m_fin);
        const float inv = l_row > 0.f ? 1.0f / l_row : 0.f;

        // ================= pass 2: P -> A1 -> MXINT8 per window -> bf16 operand; O += P_blk . V_blk
        if (tid == 0) {
            mbar_expect_tx(&bar_k[0], kbytes);
            tma_bulk_g2s(sKb(0), k_op, kbytes, &bar_k[0]);
            for (int b = 0; b < 2 && b < nblk; ++b) {
                mbar_expect_tx(&bar_v[b], vbytes);
                tma_bulk_g2s(sVb(b), v_op + (size_t)b * vbytes, vbytes, &bar_v[b]);
            }
            mbar_wait(&bar_k[0], (ph_k >> (0)) & 1u);
            issue_s(sKb(0), 0u, &bar_s[0]);
        }
        ph_k ^= 1u << (0);
        bool first_mma = true;
        for (int blk = 0; blk < nblk; ++blk) {
            const int vb = blk & 1;
            const int kb = blk * 128 + 64 * part;                   // key of this lane's column 0
            uint32_t mw[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int w = 4 * blk + 2 * part + j;
                mw[j] = (valid && w < NW) ? __ldg(mrow + w) : 0u;
            }
            mbar_wait(&bar_s[0], (ph_s >> (0)) & 1u);                          // S(blk) complete: sK is free
            ph_s ^= 1u << (0);
            tcgen05_fence_after_sync();
            if (tid == 0 && blk + 1 < nblk) {
                mbar_expect_tx(&bar_k[0], kbytes);
                tma_bulk_g2s(sKb(0), k_op + (size_t)(blk + 1) * kbytes, kbytes, &bar_k[0]);
            }
            if (blk > 0) {                                          // P.V(blk - 1) done: sP and V buffer (blk + 1) & 1 are free
                mbar_wait(&bar_o, ph_o);
                ph_o ^= 1u;
                if (tid == 0 && blk + 1 < nblk) {
                    mbar_expect_tx(&bar_v[vb ^ 1], vbytes);
                    tma_bulk_g2s(sVb(vb ^ 1), v_op + (size_t)(blk + 1) * vbytes, vbytes, &bar_v[vb ^ 1]);
                }
            }
#pragma unroll 1
            for (int j = 0; j < 2; ++j) {
                const int wl = 2 * part + j;                        // window slot within the block
                uint32_t r[32];
                tmem_ld_16x32bx2_s64_x32(my_tmem + 32 * j, r);
                tmem_ld_wait();
                const uint32_t mwj = j ? mw[1] : mw[0];
                uint32_t mx4[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int c = 0; c < 32; ++c) {
                    float sv = __uint_as_float(r[c]);
                    if (bf16) sv = bf16_half_away(sv);
                    float ts = __fmul_rn(sv, scale);
                    if (BIAS) ts = __fadd_rn(ts, bias_at(kb + 32 * j + c));
                    const float ex = exp_fast_nonpos(__fsub_rn(ts, m_fin));     // as in pass 1: sum(p) stays 1
                    const float ev = ((mwj >> c) & 1u) ? ex : 0.f;
                    uint32_t pb = __float_as_uint(ev * inv);
                    if (bf16) pb = bf16_half_away(pb);
                    r[c] = pb;
                    mx4[c & 3] = max(mx4[c & 3], pb);               // p >= 0: bit patterns order like the values
                }
                const uint32_t mx = max(max(mx4[0], mx4[1]), max(mx4[2], mx4[3]));
                const int e = mx_shared_exp(mx);
                const bool dead = (flush && e <= -127) || mx == 0u;
                unsigned char* pdst = sP + ((size_t)(wl * 4) * K2T + rr) * 16;
                if (dead || e >= -120) {
                    // code = min(127, floor(p * 2^(6-e) + 0.5)) without F2I / I2F (see K1); a dead window (no kept
                    // key / flushed) runs the same code with scale 0: code 0
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
            __syncthreads();                                        // P complete; every lane has read S(blk)
            if (tid == 0) {
                mbar_wait(&bar_v[vb], (ph_v >> (vb)) & 1u);
                tcgen05_fence_after_sync();
                for (int wl = 0; wl < 4; ++wl) {
                    if (4 * blk + wl >= NW) break;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint64_t da = umma_smem_desc(smem_u32(sP + (size_t)(wl * 4 + 2 * h) * K2T * 16), K2T * 16, 128);
                        const uint64_t db = umma_smem_desc(smem_u32(sVb(vb) + (size_t)(wl * 4 + 2 * h) * hdp * 16), hdp * 16, 128);
                        umma_bf16_ss(tmem + o_col, da, db, idesc_o, !first_mma);
                        first_mma = false;
                    }
                }
                umma_commit(&bar_o);
                if (blk + 1 < nblk) {                               // S(blk + 1) right behind the P.V MMAs
                    mbar_wait(&bar_k[0], (ph_k >> (0)) & 1u);
                    issue_s(sKb(0), 0u, &bar_s[0]);
                }
            }
            ph_v ^= 1u << (vb);
            if (blk + 1 < nblk) ph_k ^= 1u << (0);
            first_mma = false;
        }
        mbar_wait(&bar_o, ph_o);
        ph_o ^= 1u;
        tcgen05_fence_after_sync();

        // ---- O -> A1 -> global (coalesced through the P region, which the finished MMAs no longer read)
        store_o_tile<BF16, OT>(tmem + o_col, sP, warp, lane, tile, Nq, hd, hdp, out_head, p.o_sN, OT != DT_F32);
        fence_proxy_async_smem();
        tcgen05_fence_before_sync();
        __syncthreads();                                            // O read; smem / TMEM reusable by the next tile
        tcgen05_fence_after_sync();
    }
    if (warp == 0) tmem_dealloc(tmem, 256u);
}

// defined in mxprune_long.cu: launches k_attend_long_pair, returns the status (MXP_E_UNSUPPORTED when the layout does
// not fit the kernel's shared memory)
int launch_attend_long_pair(const AttnParams& p, cudaStream_t st);

}  // namespace mxp
