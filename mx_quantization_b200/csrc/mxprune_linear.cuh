// MX Linear (SURVEY.md 8 f2: "the step either side" of the attention core): the reference's
// mx.Linear forward (microxscaling/mx/linear.py:20-103) for MXINT8 activations and weights,
//     y = A1( A1( MXq(A1(x)) . MXq(A1(W))^T ) + A1(bias) )            A1 = bf16 half-away rounding or identity
// with both operands MX-quantized along in_features in blocks of 32.  Every MXINT8 value c * 2^(e-6)
// is exact in bf16, so the contraction is a bf16 x bf16 -> fp32 GEMM on the tcgen05 tensor cores with
// no product altered (only the fp32 summation order differs from the reference's BLAS).
//
//   k_quantize_gemm_operand  fp32 / bf16 / fp16 (rows, K) -> bf16 operand in the MMA-ready order the GEMM streams:
//                            [row tile][k step of 64][8 chunks][tile rows][16 B]  (K-major, no swizzle:
//                            one stage of one tile is ONE contiguous block -> one TMA bulk copy).
//                            One thread per 32-wide MX block, same F2I-free arithmetic as the predictor; a
//                            16-bit row is widened to its exact fp32 values as it loads.
//   k_mx_linear_umma         128 x 256 output tile per CTA, 192 threads, warp-specialised:
//                              warp 0   TMA producer   (cp.async.bulk, ring of stages, full/empty mbarriers)
//                              warp 1   MMA issuer     (4 tcgen05.mma of K = 16 per stage, commit -> empty)
//                              warps 2-5 epilogue      (TMEM lane = output row: A1, + bias, A1, then the store in
//                                                       the output type: 128-bit fp32 or 64-bit bf16 / fp16, RNE)
//                            Persistent, one CTA per SM walking the output tiles; the accumulator is
//                            double-buffered in TMEM (2 x 256 columns), so the epilogue of one tile overlaps
//                            the main loop of the next.
//                            EPI = EPI_GELU / EPI_GELU_TANH (the fused MLP's fc1): the epilogue applies the
//                            activation and writes the NEXT GEMM's A operand instead of the output; each 32-column
//                            pass over a TMEM row is one MX block of fc2's input, held by one thread.
//                            EPI = EPI_GATED_RESIDUAL (an adaLN block's proj / fc2): the coalesced store path stores
//                            residual + gate * y, with the residual read in the store's width and pattern.
//   With MOD, k_quantize_gemm_operand applies the adaLN modulation x * (1 + scale) + shift to the elements it loads.
#pragma once
#include "mxprune_predict_tc.cuh"

namespace mxp {

constexpr int GL_BM = 128;            // output rows (tokens) per CTA == TMEM lanes
constexpr int GL_BN = 256;            // output features per CTA == TMEM columns
constexpr int GL_BK = 64;             // K per pipeline stage (8 chunks of 8 bf16)
constexpr int GL_T = 192;

struct GemmOpLayout {
    int ksteps;                       // K / 64
    size_t a_stage, b_stage;          // bytes of one stage of one tile
};
__host__ __device__ inline GemmOpLayout gemm_op_layout(int K) {
    GemmOpLayout L;
    L.ksteps = K / GL_BK;
    L.a_stage = (size_t)8 * GL_BM * 16;
    L.b_stage = (size_t)8 * GL_BN * 16;
    return L;
}

// an fp32 value rounded to nearest even in DT and widened back (identity for fp32)
template <int DT>
__device__ __forceinline__ float round_to_dt(float x) {
    if constexpr (DT == DT_BF16) return __bfloat162float(__float2bfloat16_rn(x));
    else if constexpr (DT == DT_F16) return __half2float(__float2half_rn(x));
    else return x;
}

// four consecutive elements of type DT at element offset off as fp32 bit patterns: one 16-byte (fp32) or 8-byte load
template <int DT>
__device__ __forceinline__ uint4 load_elem4_bits(const float* p, int64_t off) {
    if constexpr (DT == DT_F32) {
        return *reinterpret_cast<const uint4*>(p + off);
    } else {
        const uint2 w = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(p) + off);
        return make_uint4(widen1<DT>((uint16_t)(w.x & 0xffffu)), widen1<DT>((uint16_t)(w.x >> 16)),
                          widen1<DT>((uint16_t)(w.y & 0xffffu)), widen1<DT>((uint16_t)(w.y >> 16)));
    }
}

// adaLN modulation of the activation operand (DiT / PixArt blocks: modulate(x, shift, scale)): row r of x belongs to
// batch entry r / tokens, whose shift and scale rows (K elements of x's type each, row strides ld_shift / ld_scale)
// turn x into x * (1 + scale) + shift, each operation rounded to x's type as eager torch evaluates it.
struct ModParams {
    const float *shift, *scale;
    int64_t ld_shift, ld_scale;
    int tokens;
};
// the 32 elements of one MX block (fp32 bit patterns of x's values, columns col..col+31 of batch entry bi), modulated
template <int DT>
__device__ __forceinline__ void modulate_block(uint32_t (&xv)[32], const ModParams& m, int bi, int col) {
    const float* sc = view_elem<DT>(m.scale, (int64_t)bi * m.ld_scale + col);
    const float* sh = view_elem<DT>(m.shift, (int64_t)bi * m.ld_shift + col);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
        const uint4 s4 = load_elem4_bits<DT>(sc, j4), h4 = load_elem4_bits<DT>(sh, j4);
        const uint32_t s[4] = {s4.x, s4.y, s4.z, s4.w}, h[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float t = round_to_dt<DT>(__fadd_rn(1.0f, __uint_as_float(s[j])));                 // 1 + scale
            const float u = round_to_dt<DT>(__fmul_rn(__uint_as_float(xv[j4 + j]), t));              // x * (1 + scale)
            xv[j4 + j] = __float_as_uint(round_to_dt<DT>(__fadd_rn(u, __uint_as_float(h[j]))));      // + shift
        }
    }
}

// rows_tile = 128 (activations) or 256 (weights); rows_pad = multiple of rows_tile (zero rows past `rows`).
// x holds elements of type DT (DT_*); ld in elements.  MOD: the operand is quantized from x modulated by `mod` (rows
// past `rows` stay zero rows and read no modulation).
template <int DT, bool MOD = false>
__global__ void __launch_bounds__(256)
k_quantize_gemm_operand(const float* __restrict__ x, int64_t ld, int rows, int rows_pad, int K, int rows_tile,
                        int bf16, int flush, unsigned char* __restrict__ op, const ModParams mod) {
    const int nb = K >> 5, ksteps = K / GL_BK;
    const int64_t ntask = (int64_t)rows_pad * nb;
    const size_t stage_bytes = (size_t)8 * rows_tile * 16;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < ntask; t += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(t / rows_pad), row = (int)(t - (int64_t)b * rows_pad);      // block-major: coalesced stores
        uint32_t xv[32];
        load_block_bits<DT>(view_elem<DT>(x, (int64_t)row * ld + 32 * b), 32, row < rows, xv);
        if constexpr (MOD) {
            if (row < rows) modulate_block<DT>(xv, mod, row / mod.tokens, 32 * b);
        }
        BlockQ r;
        quantize_block_thread<false, false>(xv, 32, bf16, flush, r);
        const int tile = row / rows_tile, rt = row - tile * rows_tile;
        const int kstep = b >> 1, kc0 = (b & 1) * 4;
        unsigned char* dst = op + ((size_t)tile * ksteps + kstep) * stage_bytes + ((size_t)kc0 * rows_tile + rt) * 16;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(dst + (size_t)ch * rows_tile * 16) = r.op[ch];
    }
}

// Epilogues of k_mx_linear_umma: store the output, apply an activation (MXP_ACT_* + 1) and write the next GEMM's
// A operand, or store residual + gate * output (the adaLN block's gated residual).
constexpr int EPI_STORE = 0, EPI_GELU = 1, EPI_GELU_TANH = 2, EPI_GATED_RESIDUAL = 3;

// torch.nn.functional.gelu on CUDA, bit for bit: ATen's GeluCUDAKernelImpl (ActivationGeluKernel.cu) in fp32 opmath,
//     approximate='none'  x * 0.5 * (1 + erf(x * M_SQRT1_2))
//     approximate='tanh'  0.5 * x * (1 + tanh(sqrt(2/pi) * (x + 0.044715 * x^3)))
// with the operation order and the one contraction (kappa * x^3 + x -> FFMA) of torch's sm_100 SASS, and the same
// CUDA libdevice erff / tanhf.  Explicit _rn intrinsics keep the compiler from contracting anything else.
__device__ __forceinline__ float gelu_erf(float x) {
    return __fmul_rn(__fmul_rn(x, 0.5f), __fadd_rn(1.0f, erff(__fmul_rn(x, 0.70710678118654752440f))));
}
__device__ __forceinline__ float gelu_tanh(float x) {
    const float inner = __fmul_rn(0.7978845608028654f, __fmaf_rn(0.044715f, __fmul_rn(__fmul_rn(x, x), x), x));
    return __fmul_rn(__fmul_rn(x, 0.5f), __fadd_rn(1.0f, tanhf(inner)));
}
template <int EPI>
__device__ __forceinline__ float activation(float x) {
    return EPI == EPI_GELU_TANH ? gelu_tanh(x) : gelu_erf(x);
}

// elementwise activation of n elements of type DT (the fused epilogue's function; parity aid)
template <int DT, int EPI>
__global__ void k_activation(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float y = activation<EPI>(__uint_as_float(load_elem_bits<DT>(x, i)));
        if constexpr (DT == DT_F32) out[i] = y;
        else if constexpr (DT == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(y);
        else reinterpret_cast<__half*>(out)[i] = __float2half_rn(y);
    }
}

struct LinearParams {
    const unsigned char *a_op, *w_op;
    const float* bias;                // already A1-rounded by the host wrapper kernel, or null
    float* out;                       // elements of the kernel's OUT_DT
    int64_t ldo;
    int M, N, K, bf16, stages;
    int flush;                        // EPI_GELU*: the next GEMM's quantizer setting
    unsigned char* h_op;              // EPI_GELU*: the next GEMM's A operand (K = N), written instead of out
    const float* residual;            // EPI_GATED_RESIDUAL: (M, N) of OUT_DT, row stride ldr
    const float* gate;                // EPI_GATED_RESIDUAL: (M / tokens, N) of OUT_DT, row stride ldg; row r uses r / tokens
    int64_t ldr, ldg;
    int tokens;
};

// the gated residual of four outputs y (columns col..col+3 of row `row`, fp32 values before the store's rounding):
// residual + gate * y, each operation rounded to DT as eager torch evaluates it on tensors of that type
template <int DT>
__device__ __forceinline__ float4 gated_residual4(float4 y, const LinearParams& p, int row, int col) {
    const uint4 r = load_elem4_bits<DT>(p.residual, (int64_t)row * p.ldr + col);
    const uint4 g = load_elem4_bits<DT>(p.gate, (int64_t)(row / p.tokens) * p.ldg + col);
    auto f = [](float yv, uint32_t gv, uint32_t rv) {
        const float gy = round_to_dt<DT>(__fmul_rn(__uint_as_float(gv), round_to_dt<DT>(yv)));
        return round_to_dt<DT>(__fadd_rn(__uint_as_float(rv), gy));
    };
    return make_float4(f(y.x, g.x, r.x), f(y.y, g.y, r.y), f(y.z, g.z, r.z), f(y.w, g.w, r.w));
}

// bias of element type DT -> A1(bias), N floats (tiny)
template <int DT>
__global__ void k_round_bias(const float* __restrict__ b, float* __restrict__ o, int N, int bf16) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        const float v = __uint_as_float(load_elem_bits<DT>(b, i));
        o[i] = bf16 ? bf16_half_away(v) : v;
    }
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void epilogue_barrier() {               // the 128 epilogue threads
    asm volatile("bar.sync 1, 128;" ::: "memory");
}

// Persistent: one CTA per SM walks the output tiles (feature tile fastest, so the CTAs that share an
// activation tile run together and the weight operand stays L2-resident).  The accumulator is
// double-buffered in TMEM (2 x 256 columns): the epilogue of tile i overlaps the main loop of tile i+1.
// OUT_DT (DT_*) is the element type of p.out; only the final store depends on it.  With EPI_GELU* it is the type the
// output and the activation are rounded to before fc2's quantizer reads them (what mx_linear stores and what torch's
// GELU returns on a tensor of that type); with EPI_GATED_RESIDUAL also the type of the residual and the gate.
template <int OUT_DT, int EPI = EPI_STORE>
__global__ void __launch_bounds__(GL_T, 1)
k_mx_linear_umma(const LinearParams p) {
    extern __shared__ __align__(1024) unsigned char smem_gl[];
    const GemmOpLayout L = gemm_op_layout(p.K);
    const int stages = p.stages;
    const size_t stage_bytes = L.a_stage + L.b_stage;
    float* s_bias = reinterpret_cast<float*>(smem_gl + stages * stage_bytes);                 // [2][256]
    float* s_tr = s_bias + 2 * GL_BN;                                                          // [4 warps][32][36]
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem_gl + stages * stage_bytes + 2048 + 4 * 32 * 36 * 4);   // [8]
    uint64_t* bar_empty = bar_full + 8;                                                        // [8]
    uint64_t* bar_acc_full = bar_empty + 8;                                                    // [2]
    uint64_t* bar_acc_empty = bar_acc_full + 2;                                                // [2]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_acc_empty + 2);

    constexpr bool ACT_EPI = EPI == EPI_GELU || EPI == EPI_GELU_TANH;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_n = (p.N + GL_BN - 1) / GL_BN, tiles_m = (p.M + GL_BM - 1) / GL_BM;
    const int ntiles = tiles_n * tiles_m;

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&bar_acc_full[b], 1); mbar_init(&bar_acc_empty[b], 1); }
    }
    if (warp == 1) tmem_alloc(s_tmem, 512u);
    tcgen05_fence_before_sync();
    __syncthreads();
    tcgen05_fence_after_sync();
    const uint32_t tmem = *s_tmem;

    if (warp == 0) {
        // ---------------- TMA producer
        if (lane == 0) {
            int it = 0;                                             // running stage counter across tiles
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
                const int tile_m = t / tiles_n, tile_n = t - tile_m * tiles_n;
                const unsigned char* a_src = p.a_op + (size_t)tile_m * L.ksteps * L.a_stage;
                const unsigned char* b_src = p.w_op + (size_t)tile_n * L.ksteps * L.b_stage;
                for (int ks = 0; ks < L.ksteps; ++ks, ++it) {
                    const int s = it % stages;
                    mbar_wait(&bar_empty[s], (uint32_t)(((it / stages) & 1) ^ 1));      // first lap passes at once
                    unsigned char* dst = smem_gl + (size_t)s * stage_bytes;
                    mbar_expect_tx(&bar_full[s], (uint32_t)stage_bytes);
                    tma_bulk_g2s(dst, a_src + (size_t)ks * L.a_stage, (uint32_t)L.a_stage, &bar_full[s]);
                    tma_bulk_g2s(dst + L.a_stage, b_src + (size_t)ks * L.b_stage, (uint32_t)L.b_stage, &bar_full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_bf16_f32(GL_BM, GL_BN);
            int it = 0, i = 0;
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
                const int buf = i & 1;
                mbar_wait(&bar_acc_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));         // epilogue has drained this buffer
                tcgen05_fence_after_sync();
                const uint32_t acc = tmem + (uint32_t)(buf * GL_BN);
                for (int ks = 0; ks < L.ksteps; ++ks, ++it) {
                    const int s = it % stages;
                    mbar_wait(&bar_full[s], (uint32_t)((it / stages) & 1));
                    tcgen05_fence_after_sync();
                    const unsigned char* sa = smem_gl + (size_t)s * stage_bytes;
                    const unsigned char* sb = sa + L.a_stage;
#pragma unroll
                    for (int k4 = 0; k4 < GL_BK / 16; ++k4) {
                        const uint64_t da = umma_smem_desc(smem_u32(sa + (size_t)(2 * k4) * GL_BM * 16), GL_BM * 16, 128);
                        const uint64_t db = umma_smem_desc(smem_u32(sb + (size_t)(2 * k4) * GL_BN * 16), GL_BN * 16, 128);
                        umma_bf16_ss(acc, da, db, idesc, ks > 0 || k4 > 0);
                    }
                    umma_commit(&bar_empty[s]);                     // stage free once these MMAs have read it
                }
                umma_commit(&bar_acc_full[buf]);                    // accumulator of this tile complete
            }
        }
    } else {
        // ---------------- epilogue: warps 2..5 -> TMEM lane quarter (warp & 3), thread = output row
        const int q = warp & 3;
        const int et = tid - 64;                                    // 0..127
        const bool bf16 = p.bf16 != 0;
        int i = 0;
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
            const int tile_m = t / tiles_n, tile_n = t - tile_m * tiles_n;
            const int n0 = tile_n * GL_BN, buf = i & 1;
            float* sb = s_bias + buf * GL_BN;
            const float no_bias = ACT_EPI ? -0.f : 0.f;                     // -0: the identity of the GELU epilogue's add
            for (int j = et; j < GL_BN; j += 128) sb[j] = (p.bias && n0 + j < p.N) ? __ldg(p.bias + n0 + j) : no_bias;
            epilogue_barrier();
            mbar_wait(&bar_acc_full[buf], (uint32_t)((i >> 1) & 1));
            tcgen05_fence_after_sync();
            const uint32_t t0 = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * GL_BN);
            if constexpr (ACT_EPI) {
                // thread = row; 32 TMEM columns = one MX block of fc2's input (n0 + c0 is a multiple of 32).  The
                // block is quantized in registers and its four 16-byte chunks go straight to fc2's A operand
                // [row tile][k step of 64][8 chunks][128 rows][16 B]: a warp writes 512 contiguous bytes per chunk.
                const int row = tile_m * GL_BM + q * 32 + lane;
                const int cend = p.N - n0 < GL_BN ? p.N - n0 : GL_BN;          // N is a multiple of 64
                const size_t stage_bytes = (size_t)8 * GL_BM * 16;
                unsigned char* h_tile = p.h_op + (size_t)tile_m * (p.N / GL_BK) * stage_bytes + (size_t)(q * 32 + lane) * 16;
#pragma unroll 1
                for (int c0 = 0; c0 < cend; c0 += 32) {
                    uint32_t xv[32];
                    tmem_ld_32x32b_x32(t0 + c0, xv);
                    tmem_ld_wait();
                    // branch-free, so that the 32 independent activations interleave: without a bias sb holds -0,
                    // and A1(A1(y) + -0) == A1(y) for every y (A1 is idempotent), which is the store epilogue's value
#pragma unroll
                    for (int j4 = 0; j4 < 32; j4 += 4) {
                        const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + j4);
                        const float bj[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            float y = __uint_as_float(xv[j4 + j]);
                            if (bf16) y = bf16_half_away(y);                    // A1, linear.py:85-87
                            y = __fadd_rn(y, bj[j]);
                            if (bf16) y = bf16_half_away(y);                    // :89-93
                            xv[j4 + j] = __float_as_uint(round_to_dt<OUT_DT>(y));
                        }
                    }
                    const uint32_t row_mask = row < p.M ? ~0u : 0u;             // padding rows: zero operand rows
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        xv[j] = __float_as_uint(round_to_dt<OUT_DT>(activation<EPI>(__uint_as_float(xv[j])))) & row_mask;
                    BlockQ r;
                    quantize_block_thread<false, false>(xv, 32, bf16, p.flush != 0, r);
                    const int b = (n0 + c0) >> 5;
                    unsigned char* dst = h_tile + (size_t)(b >> 1) * stage_bytes + (size_t)((b & 1) * 4) * GL_BM * 16;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(dst + (size_t)ch * GL_BM * 16) = r.op[ch];
                }
                tcgen05_fence_before_sync();
                epilogue_barrier();
                if (et == 0) mbar_arrive(&bar_acc_empty[buf]);
                continue;
            }
            // Coalesced stores: each warp transposes its 32 rows x 32 columns through shared memory
            // (row pitch 36 words: conflict-free 128-bit writes and reads), so that 8 lanes write 128
            // contiguous bytes of one fp32 output row (64 bytes of a 16-bit one) instead of 32 lanes
            // writing 16 bytes of 32 rows.
            float* tr = s_tr + (warp - 2) * (32 * 36);
            const int lr = lane >> 3, lc = (lane & 7) * 4;          // this lane's row (mod 4) and column group
            const int row_base = tile_m * GL_BM + q * 32;
#pragma unroll 1
            for (int c0 = 0; c0 < GL_BN; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32b_x32(t0 + c0, r);
                tmem_ld_wait();
#pragma unroll
                for (int v = 0; v < 8; ++v)
                    *reinterpret_cast<uint4*>(tr + lane * 36 + 4 * v) = make_uint4(r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]);
                __syncwarp();
                const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + lc);
                const bool col_ok = n0 + c0 + lc < p.N;             // N is a multiple of 4 (checked on the host)
#pragma unroll
                for (int i8 = 0; i8 < 8; ++i8) {
                    const int rl = lr + 4 * i8, row = row_base + rl;
                    float4 y = *reinterpret_cast<const float4*>(tr + rl * 36 + lc);
                    if (bf16) { y.x = bf16_half_away(y.x); y.y = bf16_half_away(y.y); y.z = bf16_half_away(y.z); y.w = bf16_half_away(y.w); }   // A1, linear.py:85-87
                    if (p.bias) {
                        y.x = __fadd_rn(y.x, b4.x); y.y = __fadd_rn(y.y, b4.y); y.z = __fadd_rn(y.z, b4.z); y.w = __fadd_rn(y.w, b4.w);
                        if (bf16) { y.x = bf16_half_away(y.x); y.y = bf16_half_away(y.y); y.z = bf16_half_away(y.z); y.w = bf16_half_away(y.w); }   // :89-93
                    }
                    if (row < p.M && col_ok) {                          // padding rows read no residual or gate
                        if constexpr (EPI == EPI_GATED_RESIDUAL) y = gated_residual4<OUT_DT>(y, p, row, n0 + c0 + lc);
                        store_out4<OUT_DT>(p.out, (int64_t)row * p.ldo + n0 + c0 + lc,
                                           make_uint4(__float_as_uint(y.x), __float_as_uint(y.y), __float_as_uint(y.z), __float_as_uint(y.w)));
                    }
                }
                __syncwarp();
            }
            tcgen05_fence_before_sync();
            epilogue_barrier();                                     // every epilogue thread has read its lanes
            if (et == 0) mbar_arrive(&bar_acc_empty[buf]);
        }
    }
    tcgen05_fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 512u);
}

}  // namespace mxp
