// gemm.cu -- fp16/bf16 GEMM on the 5th-gen tensor cores (kernel K5 of SURVEY.md 2.2):
//     C[M,N] = epilogue( A[M,K] . B[N,K]^T )        A, B K-major (row-major activations x nn.Linear
//                                                    weights as stored), fp32 accumulate in TMEM
//     epilogue: + bias[n], activation (none | GELU-erf | ReLU | tanh), + residual[m,n], cast to
//               fp16/bf16 or fp32.
// This is the op tritonserver's libtorch / ONNX-Runtime backends run through cuBLAS for the
// reference's DL endpoints (clearml_serving/engines/triton/triton_helper.py:378-385 picks the
// backend; examples/huggingface, examples/pytorch); here it is one hand-written sm_100a kernel:
//   * operands arrive by TMA (cp.async.bulk.tensor, 128-byte swizzle) into a multi-stage smem ring,
//   * one elected thread issues tcgen05.mma (UMMA 128 x BN x 16) straight from shared memory,
//   * accumulators live in TMEM, are read back with tcgen05.ld by four epilogue warps and the fused
//     epilogue writes C exactly once.
// Warp roles (192 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue.
// Roofline: tensor pipe (MEASURED_PEAKS.json bf16_tflops); algorithmic FLOPs = 2*M*N*K.
#include "common.cuh"
#include "sm100.cuh"

#include <cuda_fp16.h>
#include <cuda_bf16.h>

#include <stdlib.h>
#include <string.h>

#include <mutex>

namespace b2s {
static bool gemm_res_prefetch_enabled();
static bool gemm_2sm_enabled(int K, bool light_epilogue);
bool gemm_prefer_bn192(int M, int N, int K, int out_f32, int act);
bool gemm_pair_enabled();
static int prepare_tma_store(CUtensorMap *tc, GemmEpilogue &ep, int M, int N, int bn, const ConvGeom &cg);
int nchw_to_s2d(cudaStream_t st, const void *in, int in_dtype, int64_t n_img, int C, int H, int W, int Hz, int Wz, void *out);   // conv.cu

using namespace sm100;

enum GemmAct { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_TANH = 3, ACT_SWIGLU = 4 };

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;   // 64 x 16-bit = one 128-byte swizzle row
constexpr int GEMM_THREADS = 192;

template <int BN, int STAGES>
struct GemmSmem {
    static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
    static constexpr int B_BYTES = BN * GEMM_BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
    static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 1) * 8 + 16 + 1024;  // + alignment slack
};

// GELU (erf form, as torch.nn.functional.gelu): erf by Abramowitz-Stegun 7.1.26 (|abs err| < 1.5e-7, far
// below the fp16 rounding of the stored activation) -- one MUFU.RCP + one MUFU.EX2 instead of erff's
// ~25-instruction polynomial, which made the epilogue the bottleneck of the FFN-up GEMM.
// Both special functions are the raw MUFU forms: `__frcp_rn` / `exp2f` expand to MUFU + a fix-up sequence with a
// divergent slow-path branch per element (IEEE rounding, denormal scaling), which made this epilogue 2x the MMA
// time of a K = 768 tile.  The argument of the reciprocal is >= 1 and ex2 underflows to 0 exactly where erf is 1.
__device__ __forceinline__ float rcp_approx(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float gelu_erf(float x)
{
    const float z = fabsf(x) * 0.70710678118654752440f;
    const float t = rcp_approx(fmaf(0.3275911f, z, 1.0f));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    const float e = fmaf(-p * t, ex2_approx(z * z * -1.4426950408889634f), 1.0f);  // erf(|x|/sqrt2)
    const float hx = 0.5f * x;
    return fmaf(hx, copysignf(e, x), hx);
}

// tanh(x) = 1 - 2 / (exp(2x) + 1): branch-free (tanhf's range split costs a divergent branch per element);
// |err| ~ 1e-6, far below the 16-bit rounding of the stored activation; saturates correctly at +-inf
__device__ __forceinline__ float tanh_fast(float x)
{
    return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f);
}

// Warp-cooperative store of a 32-row x 64-byte slab: every lane holds the 64 bytes (16 words) of ITS row;
// written directly that is 32 rows x 16 B per store instruction, i.e. 32 half-filled 32-byte sectors.  Staged
// through a 2.5 KB per-warp shared-memory scratch (80-byte pitch: conflict-free 128-bit accesses) four adjacent
// lanes emit one row's 64 contiguous bytes, so each instruction writes 8 rows x 2 full sectors.
__device__ __forceinline__ void warp_store_rows64(uint32_t *scratch, const uint32_t (&w)[16], unsigned char *gbase,
                                                  size_t row_pitch_bytes, int rows_valid, int lane)
{
    uint4 *mine = reinterpret_cast<uint4 *>(scratch + lane * 20);
#pragma unroll
    for (int i = 0; i < 4; ++i) mine[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
    __syncwarp();
    const int seg = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = (lane >> 2) + 8 * i;
        const uint4 val = *reinterpret_cast<const uint4 *>(scratch + r * 20 + seg * 4);
        if (r < rows_valid) *reinterpret_cast<uint4 *>(gbase + (size_t)r * row_pitch_bytes + seg * 16) = val;
    }
    __syncwarp();
}

// Fused epilogue for 32 consecutive accumulator columns of one output row (fp32 bits in v[]):
// + bias, activation, + residual, cast, store.  `warp_row0` is the first output row of this warp's 32-row slab.
// `bv`: the 32 bias values of these columns already in registers (zero where there is no bias / past N), or
// nullptr to fetch them here (v1 kernel).  Fetching 32 predicated scalars per chunk through L1 was the
// bottleneck of the persistent kernels: the tile's own output stores keep evicting the bias lines from the
// ~30 KB of L1 left beside 197 KB of shared memory, so every chunk paid L2 latency 32 times
// (profiles/r01_ncu_gemm_tn_persistent.txt: long-scoreboard stalls on the FADDs behind LDG.E.CONSTANT).
//
// epilogue_math32: everything up to the final fp32 values f[] of this lane's row (bias, activation, residual).
__device__ __forceinline__ void epilogue_math32(const GemmEpilogue &ep, int row, bool row_ok, int col0, int ncols,
                                                const uint32_t (&v)[32], const float *bv, float (&f)[32],
                                                const uint4 *res16 = nullptr)
{
    const bool full = ncols == 32;
    const float *bias = static_cast<const float *>(ep.bias);
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
    if (bv) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] += bv[j];
    } else if (bias && row_ok) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (j < ncols) f[j] += __ldg(bias + col0 + j);
    }
    const int act_pre = ep.act_after ? ACT_NONE : ep.act;
    if (act_pre == ACT_GELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
    } else if (act_pre == ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
    } else if (act_pre == ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = tanh_fast(f[j]);
    }
    const size_t off = (size_t)row * ep.ldc + col0;
    if (res16) {   // this lane's 32 residual values (fp16), fetched by the caller ahead of the accumulator
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
            const __half2 *h = reinterpret_cast<const __half2 *>(&res16[j >> 3]);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const float2 r2 = __half22float2(h[t]);
                f[j + 2 * t] += r2.x;
                f[j + 2 * t + 1] += r2.y;
            }
        }
    } else if (ep.residual && row_ok) {
        if (ep.out_f32) {
            const float *R = static_cast<const float *>(ep.residual) + off;
            if (full && (ep.ldc & 3) == 0) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 r4 = *reinterpret_cast<const float4 *>(R + j);
                    f[j] += r4.x; f[j + 1] += r4.y; f[j + 2] += r4.z; f[j + 3] += r4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < ncols) f[j] += R[j];
            }
        } else if (ep.is_bf16) {
            const __nv_bfloat16 *R = static_cast<const __nv_bfloat16 *>(ep.residual) + off;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (j < ncols) f[j] += __bfloat162float(R[j]);
        } else {
            const __half *R = static_cast<const __half *>(ep.residual) + off;
            if (full && (ep.ldc & 7) == 0) {
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const uint4 u = *reinterpret_cast<const uint4 *>(R + j);
                    const __half2 *h = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const float2 r2 = __half22float2(h[t]);
                        f[j + 2 * t] += r2.x;
                        f[j + 2 * t + 1] += r2.y;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < ncols) f[j] += __half2float(R[j]);
            }
        }
    }
    if (ep.act_after && ep.act == ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
    }
}

// 32 fp32 values -> 16 words of packed fp16 / bf16 pairs
__device__ __forceinline__ void pack16(const GemmEpilogue &ep, const float (&f)[32], uint32_t (&w)[16])
{
    if (ep.is_bf16) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
            w[j] = *reinterpret_cast<uint32_t *>(&p);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            __half2 p = __floats2half2_rn(f[2 * j], f[2 * j + 1]);
            w[j] = *reinterpret_cast<uint32_t *>(&p);
        }
    }
}

// `scratch`: per-warp shared memory for the cooperative store, or nullptr for per-thread row stores.
__device__ __forceinline__ void epilogue_store32(const GemmEpilogue &ep, int warp_row0, int lane, int col0, int M, int N,
                                                 const uint32_t (&v)[32], const float *bv = nullptr,
                                                 uint32_t *scratch = nullptr)
{
    if (col0 >= N) return;   // warp-uniform
    const int row = warp_row0 + lane;
    const bool row_ok = row < M;
    const int ncols = min(32, N - col0);
    const bool full = ncols == 32;
    float f[32];
    epilogue_math32(ep, row, row_ok, col0, ncols, v, bv, f);
    const size_t off = (size_t)row * ep.ldc + col0;
    const int rows_valid = min(32, max(0, M - warp_row0));
    if (ep.out_f32) {
        const bool vec = full && (ep.ldc & 3) == 0;
        float *C = static_cast<float *>(ep.C);
        if (vec && scratch) {   // two 64-byte halves per row
            uint32_t w[16];
#pragma unroll
            for (int hlf = 0; hlf < 2; ++hlf) {
#pragma unroll
                for (int j = 0; j < 16; ++j) w[j] = __float_as_uint(f[hlf * 16 + j]);
                warp_store_rows64(scratch, w, reinterpret_cast<unsigned char *>(C + (size_t)warp_row0 * ep.ldc + col0 + hlf * 16),
                                  (size_t)ep.ldc * 4, rows_valid, lane);
            }
        } else if (row_ok) {
            if (vec) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4 *>(C + off + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < ncols) C[off + j] = f[j];
            }
        }
        return;
    }
    // 16-bit output (fp16 / bf16)
    const bool vec = full && (ep.ldc & 7) == 0;
    uint32_t w[16];
    pack16(ep, f, w);
    unsigned char *C = static_cast<unsigned char *>(ep.C);
    if (vec && scratch) {
        warp_store_rows64(scratch, w, C + ((size_t)warp_row0 * ep.ldc + col0) * 2, (size_t)ep.ldc * 2, rows_valid, lane);
    } else if (row_ok) {
        if (vec) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
                *reinterpret_cast<uint4 *>(C + off * 2 + j * 4) = make_uint4(w[j], w[j + 1], w[j + 2], w[j + 3]);
        } else {
            unsigned short *Cs = reinterpret_cast<unsigned short *>(C) + off;
#pragma unroll
            for (int j = 0; j < 32; ++j)   // static indices + predicates: a dynamic index would put w[] / f[] in local memory
                if (j < ncols) Cs[j] = (unsigned short)((j & 1) ? (w[j >> 1] >> 16) : (w[j >> 1] & 0xffffu));
        }
    }
}

// SwiGLU epilogue (LLM gate/up projection): the weight rows are interleaved in blocks of 32 -- fused columns
// [64j, 64j+32) are gate_{32j..32j+31}, [64j+32, 64j+64) the matching up columns -- so two consecutive 32-column
// accumulator chunks of a warp hold (gate, up) of the same 32 outputs: out = silu(gate) * up, written as one
// 64-byte row segment into C[M, N/2] (16-bit).  `col0_gate` is the fused column of the gate chunk.
__device__ __forceinline__ void epilogue_swiglu32(const GemmEpilogue &ep, int warp_row0, int lane, int col0_gate, int M, int N,
                                                  const uint32_t (&g)[32], const uint32_t (&u)[32], uint32_t *scratch)
{
    if (col0_gate + 32 >= N) return;   // warp-uniform; N is a multiple of 64 (checked on the host)
    const int rows_valid = min(32, max(0, M - warp_row0));
    uint32_t w[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float g0 = __uint_as_float(g[2 * j]), g1 = __uint_as_float(g[2 * j + 1]);
        // silu(g) * u with the raw MUFU reciprocal (an IEEE `/` costs a fix-up sequence + slow-path branch per element)
        const float a0 = g0 * rcp_approx(1.0f + __expf(-g0)) * __uint_as_float(u[2 * j]);
        const float a1 = g1 * rcp_approx(1.0f + __expf(-g1)) * __uint_as_float(u[2 * j + 1]);
        if (ep.is_bf16) {
            __nv_bfloat162 p = __floats2bfloat162_rn(a0, a1);
            w[j] = *reinterpret_cast<uint32_t *>(&p);
        } else {
            __half2 p = __floats2half2_rn(a0, a1);
            w[j] = *reinterpret_cast<uint32_t *>(&p);
        }
    }
    unsigned char *C = static_cast<unsigned char *>(ep.C);
    warp_store_rows64(scratch, w, C + ((size_t)warp_row0 * ep.ldc + (col0_gate >> 1)) * 2, (size_t)ep.ldc * 2, rows_valid, lane);
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               int M, int N, int K, GemmEpilogue ep)
{
    using S = GemmSmem<BN, STAGES>;
    extern __shared__ unsigned char smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + S::BAR_OFFSET);
    uint64_t *empty_bar = full_bar + STAGES;
    uint64_t *tmem_full_bar = empty_bar + STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_blk = blockIdx.y, n_blk = blockIdx.x;
    const int num_k = (K + GEMM_BK - 1) / GEMM_BK;

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_b);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) {  // TMEM: BN fp32 columns x 128 lanes
        tmem_alloc(tmem_slot, BN < 32 ? 32 : BN);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int kb = 0; kb < num_k; ++kb) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                unsigned char *sa = smem + stage * S::STAGE_BYTES;
                unsigned char *sb = sa + S::A_BYTES;
                mbar_arrive_expect_tx(&full_bar[stage], S::STAGE_BYTES);
                tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * GEMM_BK, m_blk * GEMM_BM);
                tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * GEMM_BK, n_blk * BN);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (single thread) =====
        if (lane == 0) {
            constexpr uint32_t idesc_f16 = make_idesc_f16(GEMM_BM, BN, 0);
            constexpr uint32_t idesc_bf16 = make_idesc_f16(GEMM_BM, BN, 1);
            const uint32_t idesc = ep.is_bf16 ? idesc_bf16 : idesc_f16;
            int stage = 0;
            uint32_t phase = 0;
            for (int kb = 0; kb < num_k; ++kb) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                unsigned char *sa = smem + stage * S::STAGE_BYTES;
                unsigned char *sb = sa + S::A_BYTES;
                const uint64_t adesc = make_sw128_kmajor_desc(sa);
                const uint64_t bdesc = make_sw128_kmajor_desc(sb);
#pragma unroll
                for (int k = 0; k < GEMM_BK / 16; ++k) {
                    umma_f16(tmem_base, desc_advance(adesc, k * 32), desc_advance(bdesc, k * 32), idesc,
                             (uint32_t)((kb | k) != 0));
                }
                umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            umma_commit(tmem_full_bar);          // accumulator complete
        }
    } else {
        // ===== epilogue: TMEM -> registers -> fused bias/act/residual -> global =====
        const int q = warp & 3;  // TMEM lane quadrant this warp may access
        mbar_wait(tmem_full_bar, 0);
        tc_fence_after();
        const int warp_row0 = m_blk * GEMM_BM + q * 32;
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
            tmem_ld_wait();
            epilogue_store32(ep, warp_row0, lane, n_blk * BN + c * 32, M, N, v);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, BN < 32 ? 32 : BN);
    }
}

// One coalesced 128-bit load per lane fetches the bias of the 128 columns a warp drains (lane l holds columns
// 4l..4l+3); broadcast32() then hands every lane the 32 values of chunk c by warp shuffles.
__device__ __forceinline__ float4 load_bias128(const float *bias, int col_base, int lane, int N)
{
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) {
        const int c = col_base + lane * 4;
        if (c + 3 < N) b = __ldg(reinterpret_cast<const float4 *>(bias + c));
        else {
            if (c < N) b.x = __ldg(bias + c);
            if (c + 1 < N) b.y = __ldg(bias + c + 1);
            if (c + 2 < N) b.z = __ldg(bias + c + 2);
        }
    }
    return b;
}
__device__ __forceinline__ void broadcast32(const float4 &b, int chunk, float (&bv)[32])
{
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        const int src = chunk * 8 + (j >> 2);
        bv[j] = __shfl_sync(0xffffffffu, b.x, src);
        bv[j + 1] = __shfl_sync(0xffffffffu, b.y, src);
        bv[j + 2] = __shfl_sync(0xffffffffu, b.z, src);
        bv[j + 3] = __shfl_sync(0xffffffffu, b.w, src);
    }
}

// One epilogue warp's share (32 rows x HALF columns) of a finished accumulator, leaving through TMA stores.
// The per-thread row stores this replaces (even staged into 64-byte row segments, warp_store_rows64) kept the warp busy
// with a shared-memory round trip, address arithmetic and predicates for every 32-column chunk: ncu on ResNet's
// K = 64 expansion GEMM showed ~1800 cycles per chunk with the issue slots 29 % busy, i.e. 3.8 us of epilogue per
// 128 x 256 tile against 0.4 us of MMA (profiles/r01_ncu_gemm_epilogue_k64.txt).  Here a lane writes its row's bytes
// once, into a 4 KB per-warp staging tile in the tensor map's swizzled layout (conflict-free 128-bit stores), and one
// lane hands the tile to the TMA engine: full-line writes, rows / columns outside the matrix clipped by the hardware.
//   16-bit output, HALF >= 64: 32 rows x 128 B (two chunks per store), SWIZZLE_128B
//   16-bit output, HALF == 32: 32 rows x  64 B, SWIZZLE_64B
//   fp32 output:               32 rows x 128 B (one chunk per store), SWIZZLE_128B
// `zmap`: the C map is 3-D {N, tile_rows, m_tiles} (space-to-depth stem: tiles hold fewer than 128 rows), coordinates
// (col, row_in_tile, m_blk); otherwise 2-D {N, M}, coordinates (col, row).
template <int HALF>
__device__ __forceinline__ void epilogue_tile_tma(const GemmEpilogue &ep, const CUtensorMap *cmap, unsigned char *stage,
                                                  uint32_t t_addr, uint64_t *tmem_empty, int lane, int warp_row0, int M_tile,
                                                  int N, int col_base, bool zmap, int z_row, int z_blk, const float4 &b4,
                                                  uint32_t tmem_empty_cluster = 0 /* 2-SM kernel: the LEADER's barrier */)
{
    constexpr int NCH = HALF / 32;
    const uint32_t st = smem_u32(stage);
    const int row = warp_row0 + lane;
    const bool row_ok = row < M_tile;
    // fp16 residual with whole 16-byte row segments: this lane's 64 bytes of a chunk are requested BEFORE the TMEM load,
    // so their latency (L2 / HBM) overlaps the accumulator read and the bias shuffles instead of stalling the adds
    const bool res_early = ep.residual && !ep.out_f32 && !ep.is_bf16 && (ep.ldc & 7) == 0;
    const __half *res_row = static_cast<const __half *>(ep.residual) + (size_t)row * ep.ldc;
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
        uint32_t v[32];
        float bv[32];
        const int col0 = col_base + c * 32;
        uint4 rr[4];
        const bool rr_ok = res_early && col0 + 32 <= N;   // warp-uniform
        if (rr_ok) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                rr[i] = row_ok ? __ldg(reinterpret_cast<const uint4 *>(res_row + col0) + i) : make_uint4(0u, 0u, 0u, 0u);
        }
        tmem_ld_32x32(t_addr + (uint32_t)(c * 32), v);
        broadcast32(b4, c, bv);
        tmem_ld_wait();
        if (c == NCH - 1) {   // last TMEM read of this warp: hand the accumulator back before the math
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (tmem_empty_cluster) mbar_arrive_cluster(tmem_empty_cluster);
                else mbar_arrive(tmem_empty);
            }
        }
        if (col0 >= N) continue;   // warp-uniform
        float f[32];
        epilogue_math32(ep, row, row_ok, col0, min(32, N - col0), v, bv, f, rr_ok ? rr : nullptr);
        int store_col = -1;
        if (ep.out_f32) {
            if (lane == 0) bulk_wait_group_read<0>();   // the previous store has read the staging tile
            __syncwarp();
            const uint32_t ra = st + (uint32_t)lane * 128u;
            const int x = lane & 7;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                sts_v4(ra + (uint32_t)((i ^ x) << 4), __float_as_uint(f[4 * i]), __float_as_uint(f[4 * i + 1]),
                       __float_as_uint(f[4 * i + 2]), __float_as_uint(f[4 * i + 3]));
            store_col = col0;
        } else {
            uint32_t w[16];
            pack16(ep, f, w);
            if constexpr (NCH >= 2) {
                const int sub = c & 1;
                if (sub == 0) {
                    if (lane == 0) bulk_wait_group_read<0>();
                    __syncwarp();
                }
                const uint32_t ra = st + (uint32_t)lane * 128u;
                const int x = lane & 7;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    sts_v4(ra + (uint32_t)(((sub * 4 + i) ^ x) << 4), w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
                if (sub == 1 || col0 + 32 >= N) store_col = col0 - sub * 32;
            } else {
                if (lane == 0) bulk_wait_group_read<0>();
                __syncwarp();
                const uint32_t ra = st + (uint32_t)lane * 64u;
                const int x = (lane >> 1) & 3;
#pragma unroll
                for (int i = 0; i < 4; ++i) sts_v4(ra + (uint32_t)((i ^ x) << 4), w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
                store_col = col0;
            }
        }
        if (store_col >= 0) {   // warp-uniform
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                if (zmap) tma_store_3d(cmap, stage, store_col, z_row, z_blk);
                else tma_store_2d(cmap, stage, store_col, warp_row0);
                bulk_commit_group();
            }
        }
    }
}

// Residual rows of one warp's slab (32 rows x `ncols` columns) requested into L2 ahead of use.  The residual add of a
// memory-bound GEMM (ResNet's 1x1 expansions with K = 64..512: the identity tensor is as large as the output and never
// L2-resident) was latency-bound: a lane's four 16-byte loads per chunk are all a warp has in flight, ~16 KB per SM
// against the ~100 KB that HBM latency x bandwidth needs.  Every epilogue warp therefore asks for the slab of its NEXT
// tile while it drains the current one; the loads proper then hit L2.
__device__ __forceinline__ void prefetch_residual_slab(const GemmEpilogue &ep, int row, int M, int col0, int ncols, int N)
{
    if (!ep.residual || row >= M || col0 >= N) return;
    const int es = ep.out_f32 ? 4 : 2;
    const unsigned char *p = static_cast<const unsigned char *>(ep.residual) + ((size_t)row * ep.ldc + col0) * es;
    const int bytes = min(ncols, N - col0) * es;
    for (int b = 0; b < bytes; b += 128) asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p + b));
}

// Tile order of the persistent kernels.  With m fastest over ALL m-tiles a sweep of one weight panel touches
// the whole activation matrix: for the LLM prefill (M = 16384, K = 4096: 134 MB of A) that does not fit in
// L2 and every panel re-read A from DRAM (ncu: 9.6 GB of DRAM reads for a 0.37 GB problem,
// profiles/r01_ncu_gemm_tn_pair.txt).  Tiles are therefore walked in groups of `gm` m-tiles (a ~32 MB slab of A,
// chosen on the host): inside a group m is fastest, so the CTAs running together share a few weight panels and
// the slab stays L2-resident while all weight panels stream past it once.
__device__ __forceinline__ void tile_coords(int t, int m_tiles, int n_tiles, int gm, int &m_blk, int &n_blk)
{
    const int per_group = gm * n_tiles;
    const int g = t / per_group;
    const int m0 = g * gm;
    const int gsz = min(gm, m_tiles - m0);
    const int r = t - g * per_group;
    n_blk = r / gsz;
    m_blk = m0 + (r - n_blk * gsz);
}

// A-operand fetch of the persistent kernels.  Plain GEMM: a [128 x 64] box of the activation matrix.  Implicit-GEMM
// convolution (cg.taps > 0): the same 16 KB tile -- 128 consecutive output pixels x 64 input channels of ONE filter
// tap -- is gathered by im2col-mode TMA straight from the NHWC activation tensor (zero fill outside the image is
// the padding), so no patch matrix is ever written to or read from HBM.
struct ConvTileOrigin { int w, h, n; };
__device__ __forceinline__ ConvTileOrigin conv_tile_origin(const ConvGeom &cg, int m_blk)
{
    ConvTileOrigin o{0, 0, 0};
    if (cg.s2d) {   // whole output rows: tile = rows_per_tile rows of image n starting at row p
        const int row = m_blk * cg.rows_per_tile;
        o.n = row / cg.OH;
        o.h = row - o.n * cg.OH;
    } else if (cg.taps) {
        const int m0 = m_blk * GEMM_BM, hw = cg.OH * cg.OW;
        o.n = m0 / hw;
        const int rem = m0 - o.n * hw, p = rem / cg.OW, q = rem - p * cg.OW;
        o.w = q * cg.stride - cg.pad;
        o.h = p * cg.stride - cg.pad;
    }
    return o;
}
__device__ __forceinline__ void load_a_tile(void *sa, const CUtensorMap *tmap_a, uint64_t *bar, const ConvGeom &cg,
                                            const ConvTileOrigin &o, int kb, int m_blk)
{
    if (cg.s2d) {
        tma_load_5d(sa, tmap_a, bar, 0, 0, o.h, o.n, kb);
    } else if (cg.taps) {
        const int tap = kb / cg.cblocks, cb = kb - tap * cg.cblocks;
        const int r = tap / cg.KS, s_ = tap - r * cg.KS;
        tma_load_im2col_4d(sa, tmap_a, bar, cb * GEMM_BK, o.w, o.h, o.n, (uint16_t)s_, (uint16_t)r);
    } else {
        tma_load_2d(sa, tmap_a, bar, kb * GEMM_BK, m_blk * GEMM_BM);
    }
}

// ---------------------------------------------------------------------------------------------
// Kernel v2: persistent, 128 x 256 tiles, double-buffered TMEM accumulators.
//   * grid = min(#tiles, #SMs); each CTA walks tiles t = blockIdx.x, +gridDim.x, ... with m fastest,
//     so the CTAs that run together share one 256-row weight panel (L2 reuse of B);
//   * UMMA 128 x 256 x 16: per k-step A 4 KB + B 8 KB of shared-memory reads for 128 cycles of tensor
//     work (the 128 x 128 shape of v1 is shared-memory-bandwidth bound at 128 B/clk);
//   * TMEM holds two 256-column accumulators: the 8 epilogue warps drain tile i (tcgen05.ld, fused
//     bias / GELU / residual, stores) while the MMA warp already accumulates tile i+1;
//   * 4-stage TMA ring of 48 KB (A 16 KB + B 32 KB) per stage.
// Warp roles (384 threads): 0 TMA producer, 1 MMA issuer, 2 TMEM owner, 3 idle, 4-11 epilogue
// (warp w drains TMEM lane quadrant w % 4, column half (w - 4) / 4).
// ---------------------------------------------------------------------------------------------
constexpr int G2_THREADS = 384;
template <int G2_BN, int G2_STAGES>
struct G2Smem {
    static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;   // 16 KB
    static constexpr int B_BYTES = G2_BN * GEMM_BK * 2;     // 32 KB (BN 256) / 16 KB (BN 128)
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int BAR_OFFSET = G2_STAGES * STAGE_BYTES;
    static constexpr int SCRATCH_OFFSET = BAR_OFFSET + 1024;                      // 8 epilogue warps x 4 KB staging (1024-aligned)
    static constexpr int TOTAL = SCRATCH_OFFSET + 8 * 4096 + 1024;                // + alignment slack
};

// BN = 256 (4 stages) for wide outputs; BN = 128 (6 stages) when 128 x 256 tiles would leave the last
// wave of the persistent grid mostly empty (e.g. M = 7400 tokens, N = 768: 174 tiles on 148 SMs).
template <int G2_BN, int G2_STAGES>
__global__ void __launch_bounds__(G2_THREADS, 1)
gemm_tn_persistent_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                          const __grid_constant__ CUtensorMap tmap_c, int M, int N, int K, GemmEpilogue ep, int group_m,
                          ConvGeom cg)
{
    using S = G2Smem<G2_BN, G2_STAGES>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + S::BAR_OFFSET);
    uint64_t *empty_bar = full_bar + G2_STAGES;
    uint64_t *tmem_full_bar = empty_bar + G2_STAGES;   // [2]
    uint64_t *tmem_empty_bar = tmem_full_bar + 2;      // [2]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty_bar + 2);
    // per epilogue warp: 4 KB staging tile of the TMA-store epilogue; the row-store forms use its first 2.5 KB as scratch
    unsigned char *epi_stage = smem + S::SCRATCH_OFFSET + (((threadIdx.x >> 5) - 4) & 7) * 4096;
    uint32_t *epi_scratch = reinterpret_cast<uint32_t *>(epi_stage);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = (K + GEMM_BK - 1) / GEMM_BK;
    const int tile_rows = cg.tile_rows;   // 128 except for the space-to-depth stem (whole output rows per tile)
    const int m_tiles = (M + tile_rows - 1) / tile_rows, n_tiles = (N + G2_BN - 1) / G2_BN;
    const int total_tiles = m_tiles * n_tiles;

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_b);
        if (ep.tma_store) prefetch_tensormap(&tmap_c);
        for (int s = 0; s < G2_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1);
            mbar_init(&tmem_empty_bar[a], 8);   // one arrive per epilogue warp
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_slot, 2 * G2_BN);   // two accumulators
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int m_blk, n_blk;
                tile_coords(tile, m_tiles, n_tiles, group_m, m_blk, n_blk);
                const ConvTileOrigin org = conv_tile_origin(cg, m_blk);
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    mbar_arrive_expect_tx(&full_bar[stage], tile_rows * (GEMM_BK * 2) + S::B_BYTES);
                    load_a_tile(sa, &tmap_a, &full_bar[stage], cg, org, kb, m_blk);
                    tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * GEMM_BK, n_blk * G2_BN);
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_f16 = make_idesc_f16(GEMM_BM, G2_BN, 0);
            constexpr uint32_t idesc_bf16 = make_idesc_f16(GEMM_BM, G2_BN, 1);
            const uint32_t idesc = ep.is_bf16 ? idesc_bf16 : idesc_f16;
            int stage = 0, as = 0;
            uint32_t phase = 0, aphase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                mbar_wait(&tmem_empty_bar[as], aphase ^ 1);   // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * G2_BN);
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    const uint64_t adesc = make_sw128_kmajor_desc(sa);
                    const uint64_t bdesc = make_sw128_kmajor_desc(sb);
#pragma unroll
                    for (int k = 0; k < GEMM_BK / 16; ++k)
                        umma_f16(d_tmem, desc_advance(adesc, k * 32), desc_advance(bdesc, k * 32), idesc,
                                 (uint32_t)((kb | k) != 0));
                    umma_commit(&empty_bar[stage]);
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full_bar[as]);
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        int as = 0, bias_n = -1;
        uint32_t aphase = 0;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);   // this warp's bias slice (128 columns), fetched when the weight panel changes
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int m_blk, n_blk;
            tile_coords(tile, m_tiles, n_tiles, group_m, m_blk, n_blk);
            constexpr int HALF = G2_BN / 2, NCH = HALF / 32;
            if (ep.res_prefetch) {   // residual slab of this warp's next tile (and of its first one) into L2
                if (tile == (int)blockIdx.x)
                    prefetch_residual_slab(ep, m_blk * tile_rows + q * 32 + lane, min(M, (m_blk + 1) * tile_rows),
                                           n_blk * G2_BN + half * HALF, HALF, N);
                const int nxt = tile + (int)gridDim.x;
                if (nxt < total_tiles) {
                    int m2, n2;
                    tile_coords(nxt, m_tiles, n_tiles, group_m, m2, n2);
                    prefetch_residual_slab(ep, m2 * tile_rows + q * 32 + lane, min(M, (m2 + 1) * tile_rows),
                                           n2 * G2_BN + half * HALF, HALF, N);
                }
            }
            mbar_wait(&tmem_full_bar[as], aphase);
            tc_fence_after();
            const int warp_row0 = m_blk * tile_rows + q * 32;
            const int M_tile = min(M, (m_blk + 1) * tile_rows);   // rows of this tile that exist (stem tiles: < 128)
            const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * G2_BN + half * HALF);
            if (n_blk != bias_n) {   // consecutive tiles of a CTA mostly share the weight panel: keep its bias slice
                b4 = load_bias128(static_cast<const float *>(ep.bias), n_blk * G2_BN + half * HALF, lane, N);
                bias_n = n_blk;
            }
            if (ep.act == ACT_SWIGLU) {   // (gate, up) chunk pairs, see epilogue_swiglu32
                if constexpr (NCH >= 2) {
#pragma unroll 1
                    for (int c = 0; c < NCH; c += 2) {
                        uint32_t g[32], u[32];
                        tmem_ld_32x32(t_addr + (uint32_t)(c * 32), g);
                        tmem_ld_32x32(t_addr + (uint32_t)(c * 32 + 32), u);
                        tmem_ld_wait();
                        if (c == NCH - 2) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&tmem_empty_bar[as]);
                        }
                        epilogue_swiglu32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M_tile, N, g, u, epi_scratch);
                    }
                }
            } else if (ep.tma_store) {
                epilogue_tile_tma<HALF>(ep, &tmap_c, epi_stage, t_addr, &tmem_empty_bar[as], lane, warp_row0, M_tile, N,
                                        n_blk * G2_BN + half * HALF, cg.s2d != 0, q * 32, m_blk, b4);
            } else {
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
                uint32_t v[32];
                float bv[32];
                tmem_ld_32x32(t_addr + (uint32_t)(c * 32), v);
                broadcast32(b4, c, bv);
                tmem_ld_wait();
                if (c == NCH - 1) {   // last TMEM read of this warp: hand the accumulator back before the math
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tmem_empty_bar[as]);
                }
                epilogue_store32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M_tile, N, v, bv, epi_scratch);
            }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
        if (ep.tma_store && lane == 0) bulk_wait_group<0>();   // the staging tiles live in this CTA's shared memory
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 2 * G2_BN);
    }
}

// ---------------------------------------------------------------------------------------------
// Kernel v3: v2 on CTA PAIRS sharing the weight tile.  BERT-class GEMMs (K = 768) are bound by the
// L2 -> SM operand traffic of 1-CTA tiles (profiles/r01_ncu_gemm_tn_persistent.txt: tensor pipe 24 %
// active, long-scoreboard stalls): a 128 x 256 tile moves A 16 KB + B 32 KB per 64-deep k-block.  Here
// the two CTAs of a cluster compute vertically adjacent tiles (same 256 weight rows, different 128
// activation rows); each loads its own A tile and HALF of the B tile, multicast into both CTAs' shared
// memory, so a CTA pulls 32 KB instead of 48 KB per k-block.  A stage is free again only when BOTH MMA
// warps are done with it (tcgen05.commit multicast onto both CTAs' empty barriers, count 2).
// ---------------------------------------------------------------------------------------------
template <int G2_STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
gemm_tn_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b_half,
                    const __grid_constant__ CUtensorMap tmap_c, int M, int N, int K, GemmEpilogue ep, int group_mp,
                    ConvGeom cg)
{
    constexpr int G2_BN = 256;
    using S = G2Smem<G2_BN, G2_STAGES>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + S::BAR_OFFSET);
    uint64_t *empty_bar = full_bar + G2_STAGES;
    uint64_t *tmem_full_bar = empty_bar + G2_STAGES;
    uint64_t *tmem_empty_bar = tmem_full_bar + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty_bar + 2);
    // per epilogue warp: 4 KB staging tile of the TMA-store epilogue; the row-store forms use its first 2.5 KB as scratch
    unsigned char *epi_stage = smem + S::SCRATCH_OFFSET + (((threadIdx.x >> 5) - 4) & 7) * 4096;
    uint32_t *epi_scratch = reinterpret_cast<uint32_t *>(epi_stage);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const int num_k = (K + GEMM_BK - 1) / GEMM_BK;
    const int m_tiles = (M + GEMM_BM - 1) / GEMM_BM, n_tiles = (N + G2_BN - 1) / G2_BN;
    const int m_pairs = (m_tiles + 1) / 2;
    const int total = m_pairs * n_tiles;            // pair-tiles
    const int pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_b_half);
        if (ep.tma_store) prefetch_tensormap(&tmap_c);
        for (int s = 0; s < G2_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 2);            // both CTAs of the pair release a stage
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1);
            mbar_init(&tmem_empty_bar[a], 8);
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_slot, 2 * G2_BN);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    cluster_arrive();   // peer barriers initialised / peer CTA resident before any multicast or remote arrive
    cluster_wait();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int pt = pair0; pt < total; pt += pair_stride) {
                int mp, n_blk;
                tile_coords(pt, m_pairs, n_tiles, group_mp, mp, n_blk);
                const int m_blk = 2 * mp + (int)rank;
                const ConvTileOrigin org = conv_tile_origin(cg, m_blk);
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    mbar_arrive_expect_tx(&full_bar[stage], S::STAGE_BYTES);   // own A + both halves of B
                    load_a_tile(sa, &tmap_a, &full_bar[stage], cg, org, kb, m_blk);
                    tma_load_2d_multicast(sb + rank * (S::B_BYTES / 2), &tmap_b_half, &full_bar[stage], kb * GEMM_BK,
                                          n_blk * G2_BN + (int)rank * (G2_BN / 2), (uint16_t)0x3);
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc_f16 = make_idesc_f16(GEMM_BM, G2_BN, 0);
            constexpr uint32_t idesc_bf16 = make_idesc_f16(GEMM_BM, G2_BN, 1);
            const uint32_t idesc = ep.is_bf16 ? idesc_bf16 : idesc_f16;
            int stage = 0, as = 0;
            uint32_t phase = 0, aphase = 0;
            for (int pt = pair0; pt < total; pt += pair_stride) {
                mbar_wait(&tmem_empty_bar[as], aphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * G2_BN);
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    const uint64_t adesc = make_sw128_kmajor_desc(sa);
                    const uint64_t bdesc = make_sw128_kmajor_desc(sb);
#pragma unroll
                    for (int k = 0; k < GEMM_BK / 16; ++k)
                        umma_f16(d_tmem, desc_advance(adesc, k * 32), desc_advance(bdesc, k * 32), idesc,
                                 (uint32_t)((kb | k) != 0));
                    umma_commit_multicast(&empty_bar[stage], (uint16_t)0x3);   // frees the stage in BOTH CTAs
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full_bar[as]);
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        int as = 0, bias_n = -1;
        uint32_t aphase = 0;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);   // this warp's bias slice (128 columns), fetched when the weight panel changes
        for (int pt = pair0; pt < total; pt += pair_stride) {
            int mp, n_blk;
            tile_coords(pt, m_pairs, n_tiles, group_mp, mp, n_blk);
            const int m_blk = 2 * mp + (int)rank;
            constexpr int HALF = G2_BN / 2, NCH = HALF / 32;
            if (ep.res_prefetch) {   // residual slab of this warp's next tile (and of its first one) into L2
                if (pt == pair0)
                    prefetch_residual_slab(ep, m_blk * GEMM_BM + q * 32 + lane, M, n_blk * G2_BN + half * HALF, HALF, N);
                if (pt + pair_stride < total) {
                    int mp2, n2;
                    tile_coords(pt + pair_stride, m_pairs, n_tiles, group_mp, mp2, n2);
                    prefetch_residual_slab(ep, (2 * mp2 + (int)rank) * GEMM_BM + q * 32 + lane, M, n2 * G2_BN + half * HALF, HALF, N);
                }
            }
            mbar_wait(&tmem_full_bar[as], aphase);
            tc_fence_after();
            const int warp_row0 = m_blk * GEMM_BM + q * 32;
            const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * G2_BN + half * HALF);
            if (n_blk != bias_n) {   // consecutive tiles of a CTA mostly share the weight panel: keep its bias slice
                b4 = load_bias128(static_cast<const float *>(ep.bias), n_blk * G2_BN + half * HALF, lane, N);
                bias_n = n_blk;
            }
            if (ep.act == ACT_SWIGLU) {   // (gate, up) chunk pairs, see epilogue_swiglu32
                if constexpr (NCH >= 2) {
#pragma unroll 1
                    for (int c = 0; c < NCH; c += 2) {
                        uint32_t g[32], u[32];
                        tmem_ld_32x32(t_addr + (uint32_t)(c * 32), g);
                        tmem_ld_32x32(t_addr + (uint32_t)(c * 32 + 32), u);
                        tmem_ld_wait();
                        if (c == NCH - 2) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&tmem_empty_bar[as]);
                        }
                        epilogue_swiglu32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M, N, g, u, epi_scratch);
                    }
                }
            } else if (ep.tma_store) {
                epilogue_tile_tma<HALF>(ep, &tmap_c, epi_stage, t_addr, &tmem_empty_bar[as], lane, warp_row0, M, N,
                                        n_blk * G2_BN + half * HALF, false, 0, 0, b4);
            } else {
#pragma unroll 1
            for (int c = 0; c < NCH; ++c) {
                uint32_t v[32];
                float bv[32];
                tmem_ld_32x32(t_addr + (uint32_t)(c * 32), v);
                broadcast32(b4, c, bv);
                tmem_ld_wait();
                if (c == NCH - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tmem_empty_bar[as]);
                }
                epilogue_store32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M, N, v, bv, epi_scratch);
            }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
        if (ep.tma_store && lane == 0) bulk_wait_group<0>();   // the staging tiles live in this CTA's shared memory
    }

    tc_fence_before();
    __syncthreads();
    cluster_arrive();   // the peer may still multicast into this CTA's shared memory / arrive on its barriers
    cluster_wait();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 2 * G2_BN);
    }
}

// ---------------------------------------------------------------------------------------------
// Kernel v4: the CTA pair as ONE tensor-core unit (tcgen05 cta_group::2).  In v3 each CTA of the pair still issues its
// own 128 x 256 MMAs and reads A (16 KB) + the WHOLE weight tile (32 KB) from its shared memory per k-block: 96 B/clk of
// operand reads next to 64 B/clk of TMA writes, on a 128 B/clk shared-memory port.  Here the leader CTA issues
// 256 x 256 x 16 MMAs spanning both CTAs: each CTA keeps its 128 rows of A and its HALF of the weight tile (nothing is
// multicast, 32 KB per stage, 6 stages), the hardware reads both halves in place and each CTA's tensor memory receives
// its 128 accumulator rows.  Both CTAs' TMA loads complete bytes on the leader's full barrier; tcgen05.commit multicasts
// "stage free" / "accumulator ready" to both CTAs; both CTAs' epilogue warps release the accumulator on the leader's barrier.
// ---------------------------------------------------------------------------------------------
template <int STAGES, int BN2 = 256>
struct G2smSmem {
    static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;   // 16 KB: this CTA's 128 rows of A
    static constexpr int B_BYTES = (BN2 / 2) * GEMM_BK * 2;   // 16 / 12 KB: this CTA's half of the 256- / 192-row weight tile
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
    static constexpr int SCRATCH_OFFSET = BAR_OFFSET + 1024;
    static constexpr int TOTAL = SCRATCH_OFFSET + 8 * 4096 + 1024;
};

// BN2 = 192: pair-tiles of 256 x 192 for outputs whose width is a multiple of 192 but fills the last wave of 256-wide tiles
// badly (BERT hidden size 768: 3 x 256 -> 87 pair-tiles on 74 pairs, 4 x 192 -> 116 tiles of 3/4 the length); fp32 outputs
// only (three 32-column chunks per epilogue warp: the 16-bit TMA-store path pairs chunks).
template <int STAGES, int BN2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
gemm_tn_2sm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b_half,
                   const __grid_constant__ CUtensorMap tmap_c, int M, int N, int K, GemmEpilogue ep, int group_mp)
{
    constexpr int G2_BN = BN2;
    constexpr int TMEM_COLS = 2 * BN2 <= 256 ? 256 : 512;   // power of two >= two accumulators
    using S = G2smSmem<STAGES, BN2>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + S::BAR_OFFSET);   // used in the leader
    uint64_t *empty_bar = full_bar + STAGES;                                   // both CTAs (commit multicast)
    uint64_t *tmem_full_bar = empty_bar + STAGES;                              // both CTAs (commit multicast)
    uint64_t *tmem_empty_bar = tmem_full_bar + 2;                              // leader: 16 epilogue warps of the pair
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty_bar + 2);
    unsigned char *epi_stage = smem + S::SCRATCH_OFFSET + (((threadIdx.x >> 5) - 4) & 7) * 4096;
    uint32_t *epi_scratch = reinterpret_cast<uint32_t *>(epi_stage);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const bool leader = rank == 0;
    const int num_k = (K + GEMM_BK - 1) / GEMM_BK;
    const int m_tiles = (M + GEMM_BM - 1) / GEMM_BM, n_tiles = (N + G2_BN - 1) / G2_BN;
    const int m_pairs = (m_tiles + 1) / 2;
    const int total = m_pairs * n_tiles;            // pair-tiles
    const int pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_b_half);
        if (ep.tma_store) prefetch_tensormap(&tmap_c);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);    // the leader's producer arrives (with the byte count of BOTH CTAs' loads)
            mbar_init(&empty_bar[s], 1);   // one multicast commit
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1);
            mbar_init(&tmem_empty_bar[a], 16);
        }
        fence_barrier_init();
    }
    __syncthreads();
    cluster_arrive();   // peer barriers initialised / peer CTA resident before any remote arrive or paired instruction
    cluster_wait();
    if (warp == 2) {    // the same warp of BOTH CTAs: two accumulators of 256 columns in each CTA's tensor memory
        tmem_alloc_2sm(tmem_slot, TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int pt = pair0; pt < total; pt += pair_stride) {
                int mp, n_blk;
                tile_coords(pt, m_pairs, n_tiles, group_mp, mp, n_blk);
                const int m_blk = 2 * mp + (int)rank;
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * S::STAGE_BYTES);
                    const uint32_t bar = mapa_rank(&full_bar[stage], 0);
                    tma_load_2d_2sm(sa, &tmap_a, bar, kb * GEMM_BK, m_blk * GEMM_BM);
                    tma_load_2d_2sm(sb, &tmap_b_half, bar, kb * GEMM_BK, n_blk * G2_BN + (int)rank * (G2_BN / 2));
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {
            constexpr uint32_t idesc_f16 = make_idesc_f16(2 * GEMM_BM, G2_BN, 0);
            constexpr uint32_t idesc_bf16 = make_idesc_f16(2 * GEMM_BM, G2_BN, 1);
            const uint32_t idesc = ep.is_bf16 ? idesc_bf16 : idesc_f16;
            int stage = 0, as = 0;
            uint32_t phase = 0, aphase = 0;
            for (int pt = pair0; pt < total; pt += pair_stride) {
                mbar_wait(&tmem_empty_bar[as], aphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * G2_BN);
                for (int kb = 0; kb < num_k; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    unsigned char *sa = smem + stage * S::STAGE_BYTES;
                    unsigned char *sb = sa + S::A_BYTES;
                    const uint64_t adesc = make_sw128_kmajor_desc(sa);
                    const uint64_t bdesc = make_sw128_kmajor_desc(sb);
#pragma unroll
                    for (int k = 0; k < GEMM_BK / 16; ++k)
                        umma_f16_2sm(d_tmem, desc_advance(adesc, k * 32), desc_advance(bdesc, k * 32), idesc,
                                     (uint32_t)((kb | k) != 0));
                    umma_commit_2sm(&empty_bar[stage], (uint16_t)0x3);   // frees the stage in BOTH CTAs
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_2sm(&tmem_full_bar[as], (uint16_t)0x3);      // accumulator ready, in BOTH CTAs
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        int as = 0, bias_n = -1;
        uint32_t aphase = 0;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);   // this warp's bias slice (128 columns), fetched when the weight panel changes
        for (int pt = pair0; pt < total; pt += pair_stride) {
            int mp, n_blk;
            tile_coords(pt, m_pairs, n_tiles, group_mp, mp, n_blk);
            const int m_blk = 2 * mp + (int)rank;
            constexpr int HALF = G2_BN / 2, NCH = HALF / 32;
            if (ep.res_prefetch) {   // residual slab of this warp's next tile (and of its first one) into L2
                if (pt == pair0)
                    prefetch_residual_slab(ep, m_blk * GEMM_BM + q * 32 + lane, M, n_blk * G2_BN + half * HALF, HALF, N);
                if (pt + pair_stride < total) {
                    int mp2, n2;
                    tile_coords(pt + pair_stride, m_pairs, n_tiles, group_mp, mp2, n2);
                    prefetch_residual_slab(ep, (2 * mp2 + (int)rank) * GEMM_BM + q * 32 + lane, M, n2 * G2_BN + half * HALF, HALF, N);
                }
            }
            mbar_wait(&tmem_full_bar[as], aphase);
            tc_fence_after();
            const int warp_row0 = m_blk * GEMM_BM + q * 32;
            const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * G2_BN + half * HALF);
            const uint32_t release = mapa_rank(&tmem_empty_bar[as], 0);   // the leader counts all 16 warps of the pair
            if (n_blk != bias_n) {   // consecutive tiles of a CTA mostly share the weight panel: keep its bias slice
                b4 = load_bias128(static_cast<const float *>(ep.bias), n_blk * G2_BN + half * HALF, lane, N);
                bias_n = n_blk;
            }
            if (NCH % 2 == 0 && ep.act == ACT_SWIGLU) {   // (gate, up) chunk pairs, see epilogue_swiglu32
#pragma unroll 1
                for (int c = 0; c + 1 < NCH; c += 2) {
                    uint32_t g[32], u[32];
                    tmem_ld_32x32(t_addr + (uint32_t)(c * 32), g);
                    tmem_ld_32x32(t_addr + (uint32_t)(c * 32 + 32), u);
                    tmem_ld_wait();
                    if (c + 2 >= NCH) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(release);
                    }
                    epilogue_swiglu32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M, N, g, u, epi_scratch);
                }
            } else if (ep.tma_store) {
                epilogue_tile_tma<HALF>(ep, &tmap_c, epi_stage, t_addr, &tmem_empty_bar[as], lane, warp_row0, M, N,
                                        n_blk * G2_BN + half * HALF, false, 0, 0, b4, release);
            } else {
#pragma unroll 1
                for (int c = 0; c < NCH; ++c) {
                    uint32_t v[32];
                    float bv[32];
                    tmem_ld_32x32(t_addr + (uint32_t)(c * 32), v);
                    broadcast32(b4, c, bv);
                    tmem_ld_wait();
                    if (c == NCH - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(release);
                    }
                    epilogue_store32(ep, warp_row0, lane, n_blk * G2_BN + half * HALF + c * 32, M, N, v, bv, epi_scratch);
                }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
        if (ep.tma_store && lane == 0) bulk_wait_group<0>();   // the staging tiles live in this CTA's shared memory
    }

    tc_fence_before();
    __syncthreads();
    cluster_arrive();   // the leader's MMAs read this CTA's shared memory; peers arrive on each other's barriers
    cluster_wait();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------
// Host side: tensor maps via the driver entry point (no link-time libcuda dependency)
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, []() {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    });
    return fn;
}

// Output tensor map of the TMA-store epilogue (epilogue_tile_tma): box = one warp's staging tile, 32 rows x 128 B
// (64 B for 16-bit outputs of 64-wide tiles).  Plain GEMM / convolution: 2-D {N, M}.  Space-to-depth stem (tiles of
// tile_rows < 128 rows): 3-D {N, tile_rows, M / tile_rows}, so the rows a tile does not own are clipped.
// Falls back to the row-store epilogue (ep.tma_store = 0) when C is not 16-byte aligned / pitched.
static int prepare_tma_store(CUtensorMap *tc, GemmEpilogue &ep, int M, int N, int bn, const ConvGeom &cg)
{
    static const bool on = []() { const char *e = getenv("B2S_TMA_STORE"); return !(e && e[0] == '0'); }();
    memset(tc, 0, sizeof(*tc));
    ep.tma_store = 0;
    const int es = ep.out_f32 ? 4 : 2;
    if (!on || ep.act == ACT_SWIGLU || (reinterpret_cast<uintptr_t>(ep.C) & 15) != 0 || ((size_t)ep.ldc * es) % 16 != 0) return 0;
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point not available");
    const int rowb = (ep.out_f32 || bn >= 128) ? 128 : 64;
    const CUtensorMapDataType dt = ep.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                              : (ep.is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    const CUtensorMapSwizzle sw = rowb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const cuuint64_t pitch = (cuuint64_t)ep.ldc * es;
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r;
    if (cg.s2d) {
        if (M % cg.tile_rows != 0) return fail(B2S_ERR_INVALID, "stem: M is not a whole number of tiles");
        cuuint64_t gdim[3] = {(cuuint64_t)N, (cuuint64_t)cg.tile_rows, (cuuint64_t)(M / cg.tile_rows)};
        cuuint64_t gstride[2] = {pitch, pitch * (cuuint64_t)cg.tile_rows};
        cuuint32_t box[3] = {(cuuint32_t)(rowb / es), 32, 1};
        r = enc(tc, dt, 3, ep.C, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)M};
        cuuint64_t gstride[1] = {pitch};
        cuuint32_t box[2] = {(cuuint32_t)(rowb / es), 32};
        r = enc(tc, dt, 2, ep.C, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled (output) failed with %d", (int)r);
    ep.tma_store = 1;
    return 0;
}

// 2-D K-major tensor map: global [rows, K] row-major 16-bit, box [box_rows, 64], 128-byte swizzle
int make_tmap_2d_kmajor(CUtensorMap *out, const void *base, int64_t rows, int64_t K, int64_t ld_elems,
                        int box_rows, int is_bf16)
{
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point not available");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld_elems * 2) % 16 != 0)
        return fail(B2S_ERR_INVALID, "gemm: operand base / leading dimension must be 16-byte aligned");
    cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                     const_cast<void *>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", (int)r);
    return 0;
}

template <int BN, int STAGES>
static int launch_gemm(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb, int M, int N, int K,
                       const GemmEpilogue &ep)
{
    using S = GemmSmem<BN, STAGES>;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(gemm_tn_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(gemm)");
    dim3 grid((N + BN - 1) / BN, (M + GEMM_BM - 1) / GEMM_BM);
    gemm_tn_kernel<BN, STAGES><<<grid, GEMM_THREADS, S::TOTAL, st>>>(ta, tb, M, N, K, ep);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return 0;
}

static int g_num_sms()
{
    static int n = []() {
        int dev = 0, v = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        return v;
    }();
    return n;
}

// m-tiles per group of the persistent tile walk: a slab of A of about 32 MB (all of A when it is smaller)
static int gemm_group_m(int M, int K)
{
    const int m_tiles = (M + GEMM_BM - 1) / GEMM_BM;
    static const int64_t slab = []() { const char *e = getenv("B2S_GEMM_SLAB_MB"); return (int64_t)(e ? atoi(e) : 32) << 20; }();
    int64_t gm = slab / ((int64_t)GEMM_BM * K * 2);
    if (gm < 2) gm = 2;
    gm &= ~(int64_t)1;   // even: the pair kernel walks pairs of m-tiles
    return gm >= m_tiles ? (m_tiles + 1) & ~1 : (int)gm;
}

template <int BN, int STAGES>
static int launch_gemm_persistent(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb, int M, int N, int K,
                                  const GemmEpilogue &ep, const ConvGeom &cg = ConvGeom())
{
    using S = G2Smem<BN, STAGES>;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(gemm_tn_persistent_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(gemm v2)");
    const int tiles = ((M + cg.tile_rows - 1) / cg.tile_rows) * ((N + BN - 1) / BN);
    const int grid = tiles < g_num_sms() ? tiles : g_num_sms();
    // the L2 slab of a convolution is the activation tensor itself (K / taps channels per pixel), not the patch matrix
    const int group_m = gemm_group_m(M, cg.taps ? K / cg.taps : K);
    GemmEpilogue epk = ep;
    epk.res_prefetch = ep.residual != nullptr && gemm_res_prefetch_enabled();
    CUtensorMap tc;
    B2S_TRY(prepare_tma_store(&tc, epk, M, N, BN, cg));
    gemm_tn_persistent_kernel<BN, STAGES><<<grid, G2_THREADS, S::TOTAL, st>>>(ta, tb, tc, M, N, K, epk, group_m, cg);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return 0;
}

static int launch_gemm_pair(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb_half, int M, int N, int K,
                            const GemmEpilogue &ep, const ConvGeom &cg = ConvGeom())
{
    using S = G2Smem<256, 4>;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(gemm_tn_pair_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(gemm pair)");
    const int m_pairs = (((M + GEMM_BM - 1) / GEMM_BM) + 1) / 2;
    const int total = m_pairs * ((N + 255) / 256);
    const int max_pairs = g_num_sms() / 2;
    const int pairs = total < max_pairs ? total : max_pairs;
    const int group_mp = gemm_group_m(M, cg.taps ? K / cg.taps : K) / 2;
    GemmEpilogue epk = ep;
    epk.res_prefetch = ep.residual != nullptr && gemm_res_prefetch_enabled();
    CUtensorMap tc;
    B2S_TRY(prepare_tma_store(&tc, epk, M, N, 256, cg));
    if (gemm_2sm_enabled(K, ep.act == ACT_NONE && !ep.residual && !ep.out_f32) && cg.taps == 0 && !cg.s2d) {   // plain GEMM: the pair as one 256-row tensor-core unit
        using S2 = G2smSmem<6, 256>;
        static std::once_flag once2;
        static cudaError_t attr_err2 = cudaSuccess;
        std::call_once(once2, []() {
            attr_err2 = cudaFuncSetAttribute(gemm_tn_2sm_kernel<6, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2::TOTAL);
        });
        if (attr_err2 != cudaSuccess) return fail_cuda(attr_err2, "cudaFuncSetAttribute(gemm 2sm)");
        gemm_tn_2sm_kernel<6, 256><<<2 * pairs, G2_THREADS, S2::TOTAL, st>>>(ta, tb_half, tc, M, N, K, epk, group_mp);
        count_launch();
        B2S_CUDA(cudaGetLastError());
        return 0;
    }
    gemm_tn_pair_kernel<4><<<2 * pairs, G2_THREADS, S::TOTAL, st>>>(ta, tb_half, tc, M, N, K, epk, group_mp, cg);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return 0;
}

// The 2-SM form wins where the mainloop dominates (Llama prefill, K = 4096 / 14336: 1268 -> 1367 TFLOP/s, 8192^3 1392 ->
// 1495) and loses where the epilogue does (K = 768 with GELU, ResNet's K = 64..512 expansions: the leader's MMA stream
// waits for the epilogue warps of BOTH CTAs, so the slower CTA paces the pair): by default it takes the deep-K GEMMs.
// B2S_GEMM_2SM=0: never, =1: every plain GEMM (tests run the whole suite this way).
static bool gemm_2sm_enabled(int K, bool light_epilogue = false)
{
    static const int mode = []() { const char *e = getenv("B2S_GEMM_2SM"); return e ? atoi(e) : -1; }();
    if (mode >= 0) return mode != 0;
    return K >= 2048 || (K >= 768 && light_epilogue);   // light: 16-bit output, no activation, no residual (BERT's QKV projection)
}

static bool gemm_res_prefetch_enabled()
{
    static const bool on = []() { const char *e = getenv("B2S_RES_PREFETCH"); return !(e && e[0] == '0'); }();
    return on;
}

bool gemm_pair_enabled()
{
    static const bool on = []() { const char *e = getenv("B2S_GEMM_PAIR"); return !(e && e[0] == '0'); }();
    return on;
}

// 128 x 256 tiles move 1.5x fewer operand bytes per flop than 128 x 128, but on a persistent grid the
// cost is waves x tile time: pick the shape with the smaller estimate.
bool gemm_prefer_bn256(int M, int N, int K)
{
    if (N < 256) return false;
    const int sms = g_num_sms(), mt = (M + GEMM_BM - 1) / GEMM_BM;
    const int t256 = mt * ((N + 255) / 256), t128 = mt * ((N + 127) / 128);
    // cost of a 128 x 128 tile relative to half a 128 x 256 one: 1.15 measured on the K = 768 shapes against the v3 pair
    // kernel; against the 2-SM kernel (deep K) a 128 x 128 x 3072 tile takes 17.7 us where a CTA's 128 x 256 share of a
    // pair-tile takes 19.9 us: 128-wide tiles are bound by shared-memory operand reads (8 KB per 64-cycle MMA)
    const double f128 = (K > 0 && gemm_pair_enabled() && gemm_2sm_enabled(K, false)) ? 1.78 : 1.15;
    const double e256 = (double)((t256 + sms - 1) / sms) * 2.0;
    const double e128 = (double)((t128 + sms - 1) / sms) * f128;
    return e256 <= e128;
}

// narrow tile width for an N-column weight (box height of its "small" tensor map)
int gemm_bn_for(int N) { return N <= 64 ? 64 : 128; }

// 256 x 192 pair-tiles on the 2-SM kernel: `tb_half96` is the weight map with box height 96.  fp32 outputs only.
int gemm_tn_maps_2sm192(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb_half96, int M, int N, int K,
                        const GemmEpilogue &ep)
{
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    if (!ep.out_f32 || ep.act == ACT_SWIGLU || N % 192 != 0) return fail(B2S_ERR_INVALID, "gemm: 192-wide tiles need an fp32 output whose width is a multiple of 192");
    using S2 = G2smSmem<6, 192>;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(gemm_tn_2sm_kernel<6, 192>, cudaFuncAttributeMaxDynamicSharedMemorySize, S2::TOTAL);
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(gemm 2sm 192)");
    const int m_pairs = (((M + GEMM_BM - 1) / GEMM_BM) + 1) / 2;
    const int total = m_pairs * (N / 192);
    const int max_pairs = g_num_sms() / 2;
    const int pairs = total < max_pairs ? total : max_pairs;
    const int group_mp = gemm_group_m(M, K) / 2;
    GemmEpilogue epk = ep;
    epk.res_prefetch = ep.residual != nullptr && gemm_res_prefetch_enabled();
    CUtensorMap tc;
    B2S_TRY(prepare_tma_store(&tc, epk, M, N, 192, ConvGeom()));
    gemm_tn_2sm_kernel<6, 192><<<2 * pairs, G2_THREADS, S2::TOTAL, st>>>(ta, tb_half96, tc, M, N, K, epk, group_mp);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return 0;
}

// 192-wide 2-SM tiles pay when the output is fp32, its width a multiple of 192, the GEMM deep enough for the 2-SM kernel,
// and 256-wide tiles would leave the last wave mostly idle (cost in units of half a 256-wide tile, as gemm_prefer_bn256)
bool gemm_prefer_bn192(int M, int N, int K, int out_f32, int act)
{
    static const bool on = []() { const char *e = getenv("B2S_GEMM_192"); return !(e && e[0] == '0'); }();
    if (!on || !out_f32 || act == ACT_SWIGLU || N < 192 || N % 192 != 0 || !gemm_pair_enabled() || !gemm_2sm_enabled(K, false)) return false;
    const int pairs = g_num_sms() / 2, mp = (((M + GEMM_BM - 1) / GEMM_BM) + 1) / 2;
    const int t192 = mp * (N / 192), t256 = mp * ((N + 255) / 256);
    const double e192 = (double)((t192 + pairs - 1) / pairs) * 1.5, e256 = (double)((t256 + pairs - 1) / pairs) * 2.0;
    return e192 < e256;
}

// GEMM with caller-provided tensor maps (graph executor: maps are cached per stream / per model).
// `tb` must have been built with box height `bn` (64, 128 or 256).
// 128 x 256 tiles on CTA pairs: `tb_half` is the weight map with box height 128
int gemm_tn_maps_pair(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb_half, int M, int N, int K,
                      const GemmEpilogue &ep)
{
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    return launch_gemm_pair(st, ta, tb_half, M, N, K, ep);
}

int gemm_tn_maps(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb, int bn, int M, int N, int K,
                 const GemmEpilogue &ep)
{
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    static const bool v1_only = []() { const char *e = getenv("B2S_GEMM_V1"); return e && e[0] == '1'; }();
    // narrow outputs (ResNet stem / layer 1: N = 64 with M in the millions of pixels): same persistent kernel,
    // 128 x 64 tiles, 8-stage ring; the non-persistent v1 form stays for tiny problems (classifier heads)
    if (bn == 64) {
        if (v1_only || (int64_t)M * N < (int64_t)1 << 16) return launch_gemm<64, 6>(st, ta, tb, M, N, K, ep);
        return launch_gemm_persistent<64, 8>(st, ta, tb, M, N, K, ep);
    }
    if (bn == 256) return launch_gemm_persistent<256, 4>(st, ta, tb, M, N, K, ep);
    if (v1_only && ep.act != ACT_SWIGLU) return launch_gemm<128, 6>(st, ta, tb, M, N, K, ep);
    return launch_gemm_persistent<128, 6>(st, ta, tb, M, N, K, ep);
}

// ---------------------------------------------------------------------------------------------
// Implicit-GEMM convolution (kernel K6 of SURVEY.md 2.2): im2col-mode tensor map over NHWC activations
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                     const cuuint64_t *, const int *, const int *, cuuint32_t, cuuint32_t,
                                     const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                     CUtensorMapFloatOOBfill);

static PFN_encodeIm2col get_encode_im2col()
{
    static PFN_encodeIm2col fn = nullptr;
    static std::once_flag once;
    std::call_once(once, []() {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeIm2col>(p);
    });
    return fn;
}

// Activations x[n_img, H, W, C] fp16 (C % 64 == 0), KS x KS filter, `stride`, `pad`: one load = 128 consecutive
// output pixels (NHW order) x 64 channels of one tap, 128-byte swizzle (the layout make_sw128_kmajor_desc expects).
// The bounding box of filter base positions is [-pad, dim + pad - (KS - 1)) per spatial dim, walked with `stride`.
int make_tmap_im2col_nhwc(CUtensorMap *out, const void *base, int64_t n_img, int H, int W, int C, int KS, int stride, int pad)
{
    PFN_encodeIm2col enc = get_encode_im2col();
    if (!enc) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeIm2col driver entry point not available");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || C % GEMM_BK != 0)
        return fail(B2S_ERR_INVALID, "conv: activations must be 16-byte aligned with channels a multiple of 64");
    if (KS < 1 || KS > 7 || stride < 1 || stride > 8 || pad < 0 || pad > 7)
        return fail(B2S_ERR_INVALID, "conv: unsupported filter geometry (KS %d stride %d pad %d)", KS, stride, pad);
    cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_img};
    cuuint64_t gstride[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
    int lower[2] = {-pad, -pad};
    int upper[2] = {pad - (KS - 1), pad - (KS - 1)};
    cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void *>(base), gdim, gstride, lower, upper,
                     (cuuint32_t)GEMM_BK, (cuuint32_t)GEMM_BM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeIm2col failed with %d", (int)r);
    // drivers up to CUDA 13.1 set a descriptor bit for tensors below 128 KiB that im2col loads must not carry
    int drv = 0;
    if (cudaDriverGetVersion(&drv) == cudaSuccess && drv <= 13010 && (int64_t)n_img * H * W * C * 2 < 131072)
        reinterpret_cast<uint64_t *>(out)[1] &= ~(1ull << 21);
    return 0;
}

// Space-to-depth stem operand: z[n_img, Hz, Wz, 16] fp16.  Row (n, p, q) of k-block a is the 128 contiguous bytes
// z[n, p + a, q .. q + 3, 0 .. 15]: a 5-D view {64 k, OW q (stride 1 pixel), OH p, n_img, 4 a} whose q / a strides
// overlap the inner extent; box = {64, OW, rows_per_tile} -> rows_per_tile * OW rows of 128 B, 128-byte swizzle.
int make_tmap_stem_s2d(CUtensorMap *out, const void *base, int64_t n_img, int Hz, int Wz, int OH, int OW, int rows_per_tile)
{
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point not available");
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || OW + 3 > Wz || OH + 3 > Hz || OW > 256 || rows_per_tile * OW > GEMM_BM)
        return fail(B2S_ERR_INVALID, "stem: bad space-to-depth geometry");
    const cuuint64_t px = 16 * 2;   // bytes per z pixel
    cuuint64_t gdim[5] = {64, (cuuint64_t)OW, (cuuint64_t)OH, (cuuint64_t)n_img, 4};
    cuuint64_t gstride[4] = {px, (cuuint64_t)Wz * px, (cuuint64_t)Hz * Wz * px, (cuuint64_t)Wz * px};
    cuuint32_t box[5] = {64, (cuuint32_t)OW, (cuuint32_t)rows_per_tile, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void *>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(B2S_ERR_CUDA, "cuTensorMapEncodeTiled (stem) failed with %d", (int)r);
    return 0;
}

ConvGeom make_stem_geom(int OH, int OW)
{
    ConvGeom cg;
    cg.s2d = 1;
    cg.OH = OH;
    cg.OW = OW;
    int r = GEMM_BM / OW;
    if (r < 1) r = 1;
    while (r > 1 && OH % r != 0) --r;   // tiles never straddle two images
    cg.rows_per_tile = r;
    cg.tile_rows = r * OW;
    return cg;
}

// y[n_img*OH*OW, Cout] = act(stem conv + bias): `ta` from make_tmap_stem_s2d, `tb` over w'[Cout, 256] (box height `bn`)
int conv_stem_maps(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb, int bn, int M, int N, const GemmEpilogue &ep,
                   const ConvGeom &cg)
{
    if (M <= 0 || N <= 0) return 0;
    if (!cg.s2d || cg.tile_rows > GEMM_BM || M % cg.tile_rows != 0) return fail(B2S_ERR_INVALID, "stem: bad tile geometry");
    if (bn == 64) return launch_gemm_persistent<64, 8>(st, ta, tb, M, N, 256, ep, cg);
    if (bn == 128) return launch_gemm_persistent<128, 6>(st, ta, tb, M, N, 256, ep, cg);
    return fail(B2S_ERR_INVALID, "stem: unsupported tile width %d", bn);
}

ConvGeom make_conv_geom(int H, int W, int C, int KS, int stride, int pad)
{
    ConvGeom cg;
    cg.taps = KS * KS;
    cg.KS = KS;
    cg.cblocks = C / GEMM_BK;
    cg.OH = (H + 2 * pad - KS) / stride + 1;
    cg.OW = (W + 2 * pad - KS) / stride + 1;
    cg.stride = stride;
    cg.pad = pad;
    return cg;
}

// Convolution as GEMM with caller-provided maps: `ta` from make_tmap_im2col_nhwc, `tb` over the weight
// [Cout, KS*KS*C] with box height `bn` (64 / 128 / 256; 128 = half tile of the CTA-pair kernel when `pair`).
int conv_implicit_maps(cudaStream_t st, const CUtensorMap &ta, const CUtensorMap &tb, int bn, bool pair, int M, int N, int K,
                       const GemmEpilogue &ep, const ConvGeom &cg)
{
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    if (cg.taps <= 0 || K != cg.taps * cg.cblocks * GEMM_BK) return fail(B2S_ERR_INVALID, "conv: K does not match the filter geometry");
    if (pair) return launch_gemm_pair(st, ta, tb, M, N, K, ep, cg);
    if (bn == 64) return launch_gemm_persistent<64, 8>(st, ta, tb, M, N, K, ep, cg);
    if (bn == 256) return launch_gemm_persistent<256, 4>(st, ta, tb, M, N, K, ep, cg);
    return launch_gemm_persistent<128, 6>(st, ta, tb, M, N, K, ep, cg);
}

// C = epilogue(A[M,K] . B[N,K]^T).  A: lda elements per row, B: ldb elements per row.
int gemm_tn(cudaStream_t st, const void *A, int64_t lda, const void *B, int64_t ldb, int M, int N, int K,
            const GemmEpilogue &ep)
{
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    if (ep.act == ACT_SWIGLU && (N % 64 != 0 || N < 128 || ep.out_f32 || ep.bias || ep.residual || (ep.ldc & 7)))
        return fail(B2S_ERR_INVALID, "gemm: SwiGLU epilogue needs N %% 64 == 0, N >= 128, 16-bit output, no bias / residual");
    CUtensorMap ta, tb;
    const int bn = N <= 64 ? 64 : (gemm_prefer_bn256(M, N, K) ? 256 : 128);
    B2S_TRY(make_tmap_2d_kmajor(&ta, A, M, K, lda, GEMM_BM, ep.is_bf16));
    if (gemm_prefer_bn192(M, N, K, ep.out_f32, ep.act)) {
        B2S_TRY(make_tmap_2d_kmajor(&tb, B, N, K, ldb, 96, ep.is_bf16));
        return gemm_tn_maps_2sm192(st, ta, tb, M, N, K, ep);
    }
    if (bn == 256 && gemm_pair_enabled()) {
        B2S_TRY(make_tmap_2d_kmajor(&tb, B, N, K, ldb, 128, ep.is_bf16));
        return gemm_tn_maps_pair(st, ta, tb, M, N, K, ep);
    }
    B2S_TRY(make_tmap_2d_kmajor(&tb, B, N, K, ldb, bn, ep.is_bf16));
    return gemm_tn_maps(st, ta, tb, bn, M, N, K, ep);
}

}  // namespace b2s

// ---------------------------------------------------------------------------------------------
// C ABI: operator-level entry point (device pointers), used by the parity tests and the graph executor
// ---------------------------------------------------------------------------------------------
extern "C" B2S_API int b2s_op_gemm(int device, void *cuda_stream, const void *A, const void *B, void *C,
                                    int M, int N, int K, const float *bias, const void *residual, int act,
                                    int is_bf16, int out_f32)
{
    using namespace b2s;
    B2S_CUDA(cudaSetDevice(device));
    GemmEpilogue ep;
    ep.bias = bias;
    ep.residual = residual;
    ep.C = C;
    ep.ldc = act == 4 ? N / 2 : N;   // ACT_SWIGLU: C is [M, N / 2]
    ep.act = act;
    ep.out_f32 = out_f32;
    ep.is_bf16 = is_bf16;
    ep.act_after = 0;
    return gemm_tn(static_cast<cudaStream_t>(cuda_stream), A, K, B, K, M, N, K, ep);
}

/* y[n_img, OH, OW, Cout] = act(conv(x[n_img, H, W, C], w[Cout, KS, KS, C]) + bias) (+ residual, activation after the
 * add when act_after): implicit GEMM, no patch matrix (see conv_implicit_maps). */
extern "C" B2S_API int b2s_op_conv(int device, void *cuda_stream, const void *x, int64_t n_img, int H, int W, int C,
                                    const void *w, int Cout, int KS, int stride, int pad, const float *bias,
                                    const void *residual, void *y, int act, int act_after)
{
    using namespace b2s;
    B2S_CUDA(cudaSetDevice(device));
    if (n_img <= 0) return 0;
    const ConvGeom cg = make_conv_geom(H, W, C, KS, stride, pad);
    const int64_t M64 = n_img * cg.OH * cg.OW;
    if (M64 > 0x7fffffff) return fail(B2S_ERR_INVALID, "conv: too many output pixels");
    const int M = (int)M64, K = KS * KS * C;
    GemmEpilogue ep;
    ep.bias = bias;
    ep.residual = residual;
    ep.C = y;
    ep.ldc = Cout;
    ep.act = act;
    ep.out_f32 = 0;
    ep.is_bf16 = 0;
    ep.act_after = act_after;
    CUtensorMap ta, tb;
    B2S_TRY(make_tmap_im2col_nhwc(&ta, x, n_img, H, W, C, KS, stride, pad));
    const bool bn256 = gemm_prefer_bn256(M, Cout, 0);
    const bool pair = bn256 && gemm_pair_enabled();
    const int bn = Cout <= 64 ? 64 : (bn256 && !pair ? 256 : 128);
    B2S_TRY(make_tmap_2d_kmajor(&tb, w, Cout, K, K, bn, 0));
    return conv_implicit_maps(static_cast<cudaStream_t>(cuda_stream), ta, tb, bn, pair, M, Cout, K, ep, cg);
}

/* Stem convolution (7x7, stride 2, pad 3, <= 4 input channels) straight from the request pixels: space-to-depth into
 * `z_scratch`, then the 4x4 stride-1 form on the tensor cores (see make_tmap_stem_s2d).  `w2` is the filter rearranged
 * by the packer to [Cout, 256] (k = a*64 + b*16 + (dy*2 + dx)*4 + c <- w[co, c, 2a + dy, 2b + dx], 0 where the tap or
 * channel does not exist). */
extern "C" B2S_API int b2s_op_conv_stem(int device, void *cuda_stream, const void *x_nchw, int in_dtype, int64_t n_img, int C,
                                         int H, int W, const void *w2, int Cout, const float *bias, void *z_scratch, void *y,
                                         int act)
{
    using namespace b2s;
    B2S_CUDA(cudaSetDevice(device));
    if (n_img <= 0) return 0;
    const int OH = (H + 6 - 7) / 2 + 1, OW = (W + 6 - 7) / 2 + 1, Hz = OH + 3, Wz = OW + 3;
    if (Cout > 128 || Cout % 8 != 0 || OW > 128) return fail(B2S_ERR_INVALID, "stem: Cout <= 128 (multiple of 8) and OW <= 128");
    const int64_t M64 = n_img * OH * OW;
    if (M64 > 0x7fffffff) return fail(B2S_ERR_INVALID, "stem: too many output pixels");
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    B2S_TRY(nchw_to_s2d(st, x_nchw, in_dtype, n_img, C, H, W, Hz, Wz, z_scratch));
    const ConvGeom cg = make_stem_geom(OH, OW);
    GemmEpilogue ep;
    ep.bias = bias;
    ep.residual = nullptr;
    ep.C = y;
    ep.ldc = Cout;
    ep.act = act;
    ep.out_f32 = 0;
    ep.is_bf16 = 0;
    ep.act_after = 0;
    CUtensorMap ta, tb;
    B2S_TRY(make_tmap_stem_s2d(&ta, z_scratch, n_img, Hz, Wz, OH, OW, cg.rows_per_tile));
    const int bn = Cout <= 64 ? 64 : 128;
    B2S_TRY(make_tmap_2d_kmajor(&tb, w2, Cout, 256, 256, bn, 0));
    return conv_stem_maps(st, ta, tb, bn, (int)M64, Cout, ep, cg);
}
