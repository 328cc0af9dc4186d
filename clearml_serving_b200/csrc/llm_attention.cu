// llm_attention.cu -- causal grouped-query attention over the KV cache for the decoder-only LLM endpoint
// (BASELINE.json configs[4]; the reference delegates it to vLLM's paged attention,
// clearml_serving/serving/preprocess_service.py:1097-1348).  head_dim = 128, bf16 in, fp32 softmax/accumulate.
//
// KV cache layout (one layer): PAGED.  K and V each [page][kv_head][64][128] bf16; a sequence (KV slot) owns the pages its
// row of the page table names: token `pos` of slot `s` lives in page page_table[s * pages_per_seq + pos / 64] at row
// pos % 64.  A page is exactly one 64-key block of these kernels, so a block of one (sequence, kv head) is still one
// contiguous [64, 128] matrix streamed with full 256-byte rows -- the indirection costs one 4-byte load per block.
//
//  * prefill: one CTA = (64-query tile, q head, sequence), 4 warps x 16 query rows; K/V blocks of 64 keys are
//    double-buffered through shared memory with cp.async; S = QK^T and O += PV on mma.sync m16n8k16 (bf16) with
//    the online softmax in registers; only key blocks at or below the diagonal are visited.
//    FLOPs: 4 * 128 * S^2 / 2 per (sequence, q head).  ~1 % of the prefill FLOPs of Llama-3-8B at S=512, so
//    it stays on the legacy tensor path; the tcgen05 budget is in the GEMMs.
//  * decode: one CTA = (sequence, kv head); the G query heads of the group are the rows of one 16-row MMA tile,
//    keys stream through a 3-stage cp.async ring, RoPE + KV append are fused into the prologue (see below).
//    A first CUDA-core version (one lane per 4 dims, shuffle reductions) was issue-bound at ~25 us per layer
//    for 32 x 8 x 576 cached keys; HBM-bound target: 512 bytes per cached token per kv head.
#include "common.cuh"
#include "sm100.cuh"

#include <cuda_bf16.h>

#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <vector>

namespace b2s {

constexpr int LA_D = 128;
constexpr int LA_BQ = 64;
constexpr int LA_BK = 64;
constexpr int LA_LD = LA_D + 8;   // padded smem row: 272 B stride, conflict-free ldmatrix

__device__ __forceinline__ void la_ldmatrix_x4(uint32_t (&r)[4], const void *smem_ptr)
{
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_ptr);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void la_ldmatrix_x4_trans(uint32_t (&r)[4], const void *smem_ptr)
{
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_ptr);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void la_mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t la_pack_bf16(float lo, float hi)
{
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&h);
}
// [64 rows x 128] bf16 tile -> padded smem, 16-byte cp.async, rows >= valid zero-filled
__device__ __forceinline__ void la_load_tile_async(__nv_bfloat16 *dst, const __nv_bfloat16 *src, int64_t ld_src,
                                                   int valid_rows, int tid)
{
    for (int i = tid; i < 64 * 16; i += 128) {
        const int r = i >> 4, c = (i & 15) * 8;
        const bool ok = r < valid_rows;
        const __nv_bfloat16 *g = src + (int64_t)(ok ? r : 0) * ld_src + c;
        const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + r * LA_LD + c);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(g), "r"(ok ? 16 : 0) : "memory");
    }
}
__device__ __forceinline__ void la_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void la_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

constexpr int LA_PREFILL_SMEM = (LA_BQ + 4 * LA_BK) * LA_LD * 2;   // Q + 2 x (K, V)

__global__ void __launch_bounds__(128)
llm_attn_prefill_kernel(const __nv_bfloat16 *__restrict__ qkv, int ld_qkv, const __nv_bfloat16 *__restrict__ kc,
                        const __nv_bfloat16 *__restrict__ vc, const int32_t *__restrict__ cu_seqlens,
                        const int32_t *__restrict__ slots, const int32_t *__restrict__ page_table, int pages_per_seq,
                        __nv_bfloat16 *__restrict__ out, int ld_out, int group, int kvh_r, float scale_log2e)
{
    extern __shared__ __align__(16) unsigned char la_smem[];
    __nv_bfloat16 *Qs = reinterpret_cast<__nv_bfloat16 *>(la_smem);
    __nv_bfloat16 *Ks2 = Qs + LA_BQ * LA_LD;            // [2][64 * LD]
    __nv_bfloat16 *Vs2 = Ks2 + 2 * LA_BK * LA_LD;

    const int b = blockIdx.z, h = blockIdx.y;
    const int qt = gridDim.x - 1 - blockIdx.x;          // longest (diagonal-most) tiles first
    const int s0 = __ldg(cu_seqlens + b);
    const int S = __ldg(cu_seqlens + b + 1) - s0;
    const int q0 = qt * LA_BQ;
    if (q0 >= S) return;
    const int slot = __ldg(slots + b), kvh = h / group;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int32_t *pages = page_table + (int64_t)slot * pages_per_seq;
    const int k_end = min(S, q0 + LA_BQ);                // keys [0, k_end) can be visible to this tile

    la_load_tile_async(Qs, qkv + (int64_t)(s0 + q0) * ld_qkv + h * LA_D, ld_qkv, min(LA_BQ, S - q0), tid);
    auto issue_block = [&](int k0, int buf) {
        const int kv_valid = min(LA_BK, k_end - k0);
        const int64_t blk = ((int64_t)__ldg(pages + (k0 >> 6)) * kvh_r + kvh) * (LA_BK * LA_D);   // one page = one key block
        la_load_tile_async(Ks2 + buf * LA_BK * LA_LD, kc + blk, LA_D, kv_valid, tid);
        la_load_tile_async(Vs2 + buf * LA_BK * LA_LD, vc + blk, LA_D, kv_valid, tid);
        la_commit();
    };
    issue_block(0, 0);   // group 0 = Q + first K/V block

    uint32_t qa[8][4];
    float o[16][4];
#pragma unroll
    for (int n = 0; n < 16; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
    const int r_lo = q0 + warp * 16 + g, r_hi = r_lo + 8;   // query positions of this thread's two rows

    int buf = 0;
    for (int k0 = 0; k0 < k_end; k0 += LA_BK, buf ^= 1) {
        const bool more = k0 + LA_BK < k_end;
        if (more) issue_block(k0 + LA_BK, buf ^ 1);
        if (more) la_wait<1>(); else la_wait<0>();
        __syncthreads();
        if (k0 == 0) {
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
                la_ldmatrix_x4(qa[kk], Qs + (warp * 16 + (lane & 15)) * LA_LD + kk * 16 + (lane >> 4) * 8);
        }
        const __nv_bfloat16 *Ks = Ks2 + buf * LA_BK * LA_LD, *Vs = Vs2 + buf * LA_BK * LA_LD;

        float s[8][4];
#pragma unroll
        for (int n = 0; n < 8; ++n) s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                uint32_t kb[4];
                la_ldmatrix_x4(kb, Ks + (np * 16 + (lane & 7) + (lane >> 4) * 8) * LA_LD + kk * 16 + ((lane >> 3) & 1) * 8);
                la_mma_bf16(s[2 * np], qa[kk], kb[0], kb[1]);
                la_mma_bf16(s[2 * np + 1], qa[kk], kb[2], kb[3]);
            }
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            const int key = k0 + n * 8 + 2 * t;
            s[n][0] = key <= r_lo ? s[n][0] * scale_log2e : -INFINITY;
            s[n][1] = key + 1 <= r_lo ? s[n][1] * scale_log2e : -INFINITY;
            s[n][2] = key <= r_hi ? s[n][2] * scale_log2e : -INFINITY;
            s[n][3] = key + 1 <= r_hi ? s[n][3] * scale_log2e : -INFINITY;
            mx[0] = fmaxf(mx[0], fmaxf(s[n][0], s[n][1]));
            mx[1] = fmaxf(mx[1], fmaxf(s[n][2], s[n][3]));
        }
        float corr[2], rs[2] = {0.f, 0.f};
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
            const float m_new = fmaxf(m_run[r], mx[r]);
            corr[r] = (m_new == -INFINITY) ? 1.f : exp2f(m_run[r] - m_new);
            m_run[r] = m_new;
        }
        const float m0 = (m_run[0] == -INFINITY) ? 0.f : m_run[0];
        const float m1 = (m_run[1] == -INFINITY) ? 0.f : m_run[1];
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            s[n][0] = exp2f(s[n][0] - m0);
            s[n][1] = exp2f(s[n][1] - m0);
            s[n][2] = exp2f(s[n][2] - m1);
            s[n][3] = exp2f(s[n][3] - m1);
            rs[0] += s[n][0] + s[n][1];
            rs[1] += s[n][2] + s[n][3];
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 1);
            rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 2);
            l_run[r] = l_run[r] * corr[r] + rs[r];
        }
#pragma unroll
        for (int n = 0; n < 16; ++n) {
            o[n][0] *= corr[0]; o[n][1] *= corr[0];
            o[n][2] *= corr[1]; o[n][3] *= corr[1];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // 16 keys per k-step
            uint32_t pa[4];
            pa[0] = la_pack_bf16(s[2 * j][0], s[2 * j][1]);
            pa[1] = la_pack_bf16(s[2 * j][2], s[2 * j][3]);
            pa[2] = la_pack_bf16(s[2 * j + 1][0], s[2 * j + 1][1]);
            pa[3] = la_pack_bf16(s[2 * j + 1][2], s[2 * j + 1][3]);
#pragma unroll
            for (int np = 0; np < 8; ++np) {   // pairs of 8-wide d tiles
                uint32_t vb[4];
                la_ldmatrix_x4_trans(vb, Vs + (j * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LA_LD + np * 16 + (lane >> 4) * 8);
                la_mma_bf16(o[2 * np], pa, vb[0], vb[1]);
                la_mma_bf16(o[2 * np + 1], pa, vb[2], vb[3]);
            }
        }
        __syncthreads();
    }

    const float inv0 = l_run[0] > 0.f ? 1.f / l_run[0] : 0.f;
    const float inv1 = l_run[1] > 0.f ? 1.f / l_run[1] : 0.f;
#pragma unroll
    for (int n = 0; n < 16; ++n) {
        const int col = h * LA_D + n * 8 + 2 * t;
        if (r_lo < S) *reinterpret_cast<uint32_t *>(out + (int64_t)(s0 + r_lo) * ld_out + col) = la_pack_bf16(o[n][0] * inv0, o[n][1] * inv0);
        if (r_hi < S) *reinterpret_cast<uint32_t *>(out + (int64_t)(s0 + r_hi) * ld_out + col) = la_pack_bf16(o[n][2] * inv1, o[n][3] * inv1);
    }
}

int llm_attn_prefill(cudaStream_t st, const void *qkv, int ld_qkv, const void *kc, const void *vc, const int32_t *cu_seqlens,
                     const int32_t *slots, const int32_t *page_table, int pages_per_seq, void *out, int ld_out, int n_seq,
                     int max_seqlen, int hq_r, int kvh_r, float scale)
{
    if (n_seq <= 0 || max_seqlen <= 0) return 0;
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(llm_attn_prefill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LA_PREFILL_SMEM);
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(llm prefill attention)");
    dim3 grid((max_seqlen + LA_BQ - 1) / LA_BQ, hq_r, n_seq);
    llm_attn_prefill_kernel<<<grid, 128, LA_PREFILL_SMEM, st>>>(
        static_cast<const __nv_bfloat16 *>(qkv), ld_qkv, static_cast<const __nv_bfloat16 *>(kc),
        static_cast<const __nv_bfloat16 *>(vc), cu_seqlens, slots, page_table, pages_per_seq, static_cast<__nv_bfloat16 *>(out),
        ld_out, hq_r / kvh_r, kvh_r, scale * 1.4426950408889634f);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ decode
// One CTA = (sequence, kv head), 4 warps.  Fused prologue: the q heads of the group and the new token's k / v
// are taken straight from the fp32 accumulator of the QKV projection (cleared here), RoPE is applied, k / v are
// appended to the cache.  The G query heads form the rows of ONE 16-row MMA tile (rows >= G are zero); cached
// keys stream through a 3-stage cp.async ring in blocks of 64, warp w owning keys 16w..16w+15 of every block
// (S = QK^T: 16 mma.sync, O += PV: 16 mma.sync per warp and block), and the four per-warp online-softmax
// states are merged through shared memory at the end.
constexpr int LDM_STAGES = 3;
constexpr int LDM_TILE = LA_BK * LA_LD;                                      // elements of one K or V tile
constexpr int LDM_SMEM = (16 * LA_LD + LDM_STAGES * 2 * LDM_TILE) * 2;       // Q + ring of (K, V)

__global__ void __launch_bounds__(128)
llm_attn_decode_kernel(float *__restrict__ ws_qkv, __nv_bfloat16 *__restrict__ kc, __nv_bfloat16 *__restrict__ vc,
                       const int32_t *__restrict__ ctx_len, const int32_t *__restrict__ slots,
                       const int32_t *__restrict__ page_table, int pages_per_seq,
                       const float *__restrict__ rope_cos, const float *__restrict__ rope_sin,
                       __nv_bfloat16 *__restrict__ out, int ld_out, int hq_r, int kvh_r, int max_ctx, float scale_log2e)
{
    extern __shared__ __align__(16) unsigned char la_smem[];
    __nv_bfloat16 *Qs = reinterpret_cast<__nv_bfloat16 *>(la_smem);
    __nv_bfloat16 *ring = Qs + 16 * LA_LD;

    asm volatile("griddepcontrol.wait;\n" ::: "memory");                 // QKV projection complete
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");    // the O projection may prefetch its weights
    const int b = blockIdx.x, kvh = blockIdx.y;
    const int G = hq_r / kvh_r;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int QKV = (hq_r + 2 * kvh_r) * LA_D;
    int pos = __ldg(ctx_len + b);
    pos = pos < max_ctx ? pos : max_ctx - 1;
    const int n_ctx = pos + 1;
    const int slot = __ldg(slots + b);
    const int32_t *pages = page_table + (int64_t)slot * pages_per_seq;
    // the row appended by this step: page of `pos`, row pos % 64
    const int64_t app = (((int64_t)__ldg(pages + (pos >> 6)) * kvh_r + kvh) * LA_BK + (pos & 63)) * LA_D;
    __nv_bfloat16 *Kapp = kc + app, *Vapp = vc + app;

    const int n_blocks = (n_ctx + LA_BK - 1) / LA_BK;
    auto issue_block = [&](int blk) {
        if (blk < n_blocks) {
            const int k0 = blk * LA_BK;
            __nv_bfloat16 *dst = ring + (blk % LDM_STAGES) * 2 * LDM_TILE;
            const int64_t off = ((int64_t)__ldg(pages + blk) * kvh_r + kvh) * (LA_BK * LA_D);   // one page = one key block
            la_load_tile_async(dst, kc + off, LA_D, min(LA_BK, n_ctx - k0), tid);
            la_load_tile_async(dst + LDM_TILE, vc + off, LA_D, min(LA_BK, n_ctx - k0), tid);
        }
        la_commit();   // (possibly empty) group: keeps the wait_group arithmetic uniform
    };
    // Blocks 0 and 1 hold only OLD cache rows unless the row appended below falls into them: request them before
    // the RoPE prologue so its three dependent round trips overlap the first HBM fetches.
    const bool early = pos >= 2 * LA_BK;
    if (early) { issue_block(0); issue_block(1); }

    // ---- prologue: RoPE on q (-> Qs) and k (-> cache), v -> cache, accumulator cleared
    float *row = ws_qkv + (int64_t)b * QKV;
    for (int idx = tid; idx < 16 * 64; idx += 128) {
        const int r = idx >> 6, i = idx & 63;
        __nv_bfloat16 o1 = __float2bfloat16_rn(0.f), o2 = o1;
        if (r < G) {
            float *src = row + (kvh * G + r) * LA_D;
            const float x1 = src[i], x2 = src[i + 64];
            src[i] = 0.f;
            src[i + 64] = 0.f;
            const float c = __ldg(rope_cos + (int64_t)pos * 64 + i), sv = __ldg(rope_sin + (int64_t)pos * 64 + i);
            o1 = __float2bfloat16_rn(x1 * c - x2 * sv);
            o2 = __float2bfloat16_rn(x2 * c + x1 * sv);
        }
        Qs[r * LA_LD + i] = o1;
        Qs[r * LA_LD + i + 64] = o2;
    }
    if (tid < 64) {
        float *src = row + (hq_r + kvh) * LA_D;
        const float x1 = src[tid], x2 = src[tid + 64];
        src[tid] = 0.f;
        src[tid + 64] = 0.f;
        const float c = __ldg(rope_cos + (int64_t)pos * 64 + tid), sv = __ldg(rope_sin + (int64_t)pos * 64 + tid);
        Kapp[tid] = __float2bfloat16_rn(x1 * c - x2 * sv);
        Kapp[tid + 64] = __float2bfloat16_rn(x2 * c + x1 * sv);
    } else {
        const int i = tid - 64;
        float *src = row + (hq_r + kvh_r + kvh) * LA_D;
        const float x1 = src[i], x2 = src[i + 64];
        src[i] = 0.f;
        src[i + 64] = 0.f;
        Vapp[i] = __float2bfloat16_rn(x1);
        Vapp[i + 64] = __float2bfloat16_rn(x2);
    }
    __syncthreads();   // Qs complete; the appended K/V row is ordered before this CTA's tile loads

    if (!early) { issue_block(0); issue_block(1); }

    uint32_t qa[8][4];
#pragma unroll
    for (int kk = 0; kk < 8; ++kk)
        la_ldmatrix_x4(qa[kk], Qs + (lane & 15) * LA_LD + kk * 16 + (lane >> 4) * 8);
    float o[16][4];
#pragma unroll
    for (int n = 0; n < 16; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};

    for (int blk = 0; blk < n_blocks; ++blk) {
        issue_block(blk + 2);
        la_wait<2>();
        __syncthreads();
        const __nv_bfloat16 *Ks = ring + (blk % LDM_STAGES) * 2 * LDM_TILE, *Vs = Ks + LDM_TILE;
        const int key0 = blk * LA_BK + warp * 16;   // this warp's 16 keys
        if (key0 < n_ctx) {
            float s[2][4];
            s[0][0] = s[0][1] = s[0][2] = s[0][3] = s[1][0] = s[1][1] = s[1][2] = s[1][3] = 0.f;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
                uint32_t kb[4];
                la_ldmatrix_x4(kb, Ks + (warp * 16 + (lane & 7) + (lane >> 4) * 8) * LA_LD + kk * 16 + ((lane >> 3) & 1) * 8);
                la_mma_bf16(s[0], qa[kk], kb[0], kb[1]);
                la_mma_bf16(s[1], qa[kk], kb[2], kb[3]);
            }
            float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
            for (int n = 0; n < 2; ++n) {
                const int key = key0 + n * 8 + 2 * t;
                s[n][0] = key < n_ctx ? s[n][0] * scale_log2e : -INFINITY;
                s[n][1] = key + 1 < n_ctx ? s[n][1] * scale_log2e : -INFINITY;
                s[n][2] = key < n_ctx ? s[n][2] * scale_log2e : -INFINITY;
                s[n][3] = key + 1 < n_ctx ? s[n][3] * scale_log2e : -INFINITY;
                mx[0] = fmaxf(mx[0], fmaxf(s[n][0], s[n][1]));
                mx[1] = fmaxf(mx[1], fmaxf(s[n][2], s[n][3]));
            }
            float corr[2], rs[2] = {0.f, 0.f};
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
                mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
                const float m_new = fmaxf(m_run[r], mx[r]);   // finite: key0 < n_ctx
                corr[r] = exp2f(m_run[r] - m_new);
                m_run[r] = m_new;
            }
#pragma unroll
            for (int n = 0; n < 2; ++n) {
                s[n][0] = exp2f(s[n][0] - m_run[0]);
                s[n][1] = exp2f(s[n][1] - m_run[0]);
                s[n][2] = exp2f(s[n][2] - m_run[1]);
                s[n][3] = exp2f(s[n][3] - m_run[1]);
                rs[0] += s[n][0] + s[n][1];
                rs[1] += s[n][2] + s[n][3];
            }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 1);
                rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 2);
                l_run[r] = l_run[r] * corr[r] + rs[r];
            }
#pragma unroll
            for (int n = 0; n < 16; ++n) {
                o[n][0] *= corr[0]; o[n][1] *= corr[0];
                o[n][2] *= corr[1]; o[n][3] *= corr[1];
            }
            uint32_t pa[4];
            pa[0] = la_pack_bf16(s[0][0], s[0][1]);
            pa[1] = la_pack_bf16(s[0][2], s[0][3]);
            pa[2] = la_pack_bf16(s[1][0], s[1][1]);
            pa[3] = la_pack_bf16(s[1][2], s[1][3]);
#pragma unroll
            for (int np = 0; np < 8; ++np) {
                uint32_t vb[4];
                la_ldmatrix_x4_trans(vb, Vs + (warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LA_LD + np * 16 + (lane >> 4) * 8);
                la_mma_bf16(o[2 * np], pa, vb[0], vb[1]);
                la_mma_bf16(o[2 * np + 1], pa, vb[2], vb[3]);
            }
        }
        __syncthreads();   // all warps done with this stage before it is refilled
    }

    // ---- merge the four per-warp states (only rows g < G are real)
    float *sm_m = reinterpret_cast<float *>(ring);        // [4][8]
    float *sm_l = sm_m + 32;                              // [4][8]
    float *sm_o = sm_l + 32;                              // [4][8][128]
    if (t == 0) { sm_m[warp * 8 + g] = m_run[0]; sm_l[warp * 8 + g] = l_run[0]; }
#pragma unroll
    for (int n = 0; n < 16; ++n)
        *reinterpret_cast<float2 *>(sm_o + ((warp * 8 + g) * LA_D + n * 8 + 2 * t)) = make_float2(o[n][0], o[n][1]);
    __syncthreads();
    for (int idx = tid; idx < G * LA_D; idx += 128) {
        const int r = idx >> 7, d = idx & 127;
        float M = -INFINITY;
#pragma unroll
        for (int w = 0; w < 4; ++w) M = fmaxf(M, sm_m[w * 8 + r]);
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const float mw = sm_m[w * 8 + r];
            const float wgt = (mw == -INFINITY) ? 0.f : exp2f(mw - M);
            num = fmaf(wgt, sm_o[(w * 8 + r) * LA_D + d], num);
            den = fmaf(wgt, sm_l[w * 8 + r], den);
        }
        out[(int64_t)b * ld_out + (kvh * G + r) * LA_D + d] = __float2bfloat16_rn(den > 0.f ? num / den : 0.f);
    }
}


// ------------------------------------------------------------------------------------------------ decode, stream form
// The (sequence, kv head) form above is one wave of 256 CTAs that each walk their ~9 key blocks serially behind a
// 2-deep cp.async ring: 24 us per layer where the 75 MB of cached K/V of BASELINE.json configs[4] take 11.5 us at the
// measured HBM rate (profiles/r02_llm_decode_trace_tp1.txt).  This form deals the KEY BLOCKS, not the sequences:
//   * the (sequence, kv head, 64-key block) list of the whole batch is flattened in that order and cut into one
//     CONTIGUOUS range per SM (one persistent CTA each), so every SM streams the same number of bytes whatever the
//     context lengths are; a CTA's range covers a few (sequence, kv head) SEGMENTS;
//   * warp 0 is a TMA producer that keeps a 5-stage ring of (K, V) blocks (32 KB each, 128B-swizzled halves of the
//     [64, 128] page) full across segment boundaries -- 160 KB in flight per SM; consumer warps 1-4 / 5-8 take
//     alternate blocks (warp w of a group owns keys 16w..16w+15, as above) with the online softmax in registers;
//   * a segment that holds all blocks of its (sequence, kv head) writes the output directly; otherwise the CTA leaves
//     its (m, l, o) partial in a workspace slot and bumps a counter, and the LAST CTA to arrive for that
//     (sequence, kv head) merges the parts in part order (deterministic);
//   * RoPE + KV append stay fused: the CTA whose segment ends with the sequence's last block computes the new K / V
//     row, appends it to the cache and patches it into the staged block in shared memory (the TMA load of that page
//     may or may not have seen the row); the fp32 QKV accumulator is cleared by whoever finishes the
//     (sequence, kv head): its only reader, or the merging CTA.
// Shapes: GROUPS consumer groups of 4 warps (+ 1 producer warp) per CTA and a ring of ST stages.
//   <3, 1>: 160 threads, 111 KB -- TWO CTAs per SM (G <= 4).  A CTA's fixed latencies (partition, the q round trip and
//           the merge of every segment, the arrival at the end) overlap the other CTA's blocks; one 8-warp CTA per SM
//           measured 33 k cycles per range of 16 blocks of which 12 k were blocks (profiles/r02_llm_attn_decode_stream.txt).
//   <4, 2>: 288 threads, one CTA per SM (G > 4: the merge area of 8 x G states does not fit twice).
// With two groups, block i goes to group i & 1 and stage i % ST: ST must then be EVEN so that a stage is always consumed
// by the same group -- a group waits for the phases of a stage's barrier strictly in order.  With an odd depth the groups
// alternate on a stage, a group can start waiting for use u while use u - 1 (the other group's block) is still in
// flight, and the parity test of mbarrier.try_wait cannot tell phase u from phase u - 2: seen as a pipeline deadlock.
constexpr int LDS_STAGE_BYTES = 4 * 8192;                 // K lo / K hi / V lo / V hi halves, [64 rows][128 B] swizzled
constexpr int LDS_PART_LD = 132;                          // floats per partial row: o[128], m, l, pad
constexpr int LDS_MERGE_LD = 132;                         // floats per row of the in-CTA merge area (bank spread)
template <int ST, int GROUPS>
struct LdsSmem {
    static constexpr int OFF_Q = ST * LDS_STAGE_BYTES;            // [8][136] bf16
    static constexpr int OFF_NEW = OFF_Q + 8 * LA_LD * 2;         // k_new[128], v_new[128] bf16
    static constexpr int OFF_MISC = OFF_NEW + 512;                // prefix[34], flags[2], pos[32], slot[32] ints, barriers
    static constexpr int OFF_MERGE = OFF_MISC + 100 * 4 + 2 * ST * 8 + 16;   // m[4 GROUPS][8], l[4 GROUPS][8], o[4 GROUPS][G][132] fp32
    static constexpr int total(int G) { return OFF_MERGE + (2 * 32 * GROUPS + 4 * GROUPS * G * LDS_MERGE_LD) * 4 + 1024; }   // + alignment slack
};

struct LdsWalk {
    int b, h, j, nb;
};

__device__ __forceinline__ void lds_seek(LdsWalk &w, const int *prefix, int n_seq, int kvh_r, int f)
{
    // largest b < n_seq with prefix[b] * kvh_r <= f (prefix is increasing: every sequence has at least one block)
    int lo = 0, hi = n_seq - 1;
#pragma unroll 1
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (prefix[mid] * kvh_r <= f) lo = mid;
        else hi = mid - 1;
    }
    w.b = lo;
    w.nb = prefix[lo + 1] - prefix[lo];
    const int rem = f - prefix[lo] * kvh_r;
    w.h = rem / w.nb;
    w.j = rem - w.h * w.nb;
}
__device__ __forceinline__ void lds_next(LdsWalk &w, const int *prefix, int kvh_r)
{
    if (++w.j == w.nb) {
        w.j = 0;
        if (++w.h == kvh_r) {
            w.h = 0;
            ++w.b;
            w.nb = prefix[w.b + 1] - prefix[w.b];
        }
    }
}
// CTA whose range [T c / n, T (c + 1) / n) holds flattened block f:  T c < (f + 1) n <= T (c + 1)
__device__ __forceinline__ int lds_owner(int f, int T, int n)
{
    return (int)(((uint32_t)(f + 1) * (uint32_t)n - 1u) / (uint32_t)T);
}
template <int NC>
__device__ __forceinline__ void lds_bar_consumers() { asm volatile("bar.sync 1, %0;\n" ::"n"(NC) : "memory"); }
__device__ __forceinline__ void lds_bar_group(int grp) { asm volatile("bar.sync %0, 128;\n" ::"r"(2 + grp) : "memory"); }

template <int LDS_STAGES, int GROUPS>
__global__ void __launch_bounds__(32 + 128 * GROUPS, GROUPS == 1 ? 2 : 1)
llm_attn_decode_stream_kernel(const __grid_constant__ CUtensorMap tmap_k, const __grid_constant__ CUtensorMap tmap_v,
                              float *__restrict__ ws_qkv, __nv_bfloat16 *__restrict__ kc, __nv_bfloat16 *__restrict__ vc,
                              const int32_t *__restrict__ ctx_len, const int32_t *__restrict__ slots,
                              const int32_t *__restrict__ page_table, int pages_per_seq,
                              const float *__restrict__ rope_cos, const float *__restrict__ rope_sin,
                              __nv_bfloat16 *__restrict__ out, int ld_out, int n_seq, int hq_r, int kvh_r, int max_ctx,
                              float scale_log2e, float *__restrict__ part_ws, int *__restrict__ part_cnt, long long *__restrict__ dbg)
{
    using namespace sm100;
    extern __shared__ unsigned char lds_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(lds_raw) + 1023) & ~(uintptr_t)1023);
    using SM = LdsSmem<LDS_STAGES, GROUPS>;
    static_assert(GROUPS == 1 || (GROUPS == 2 && LDS_STAGES % 2 == 0), "a stage must always be consumed by the same warp group");
    constexpr int NC = 128 * GROUPS;        // consumer threads
    constexpr int NW = 4 * GROUPS;          // consumer warps = per-segment softmax states
    __nv_bfloat16 *Qs = reinterpret_cast<__nv_bfloat16 *>(smem + SM::OFF_Q);
    __nv_bfloat16 *s_new = reinterpret_cast<__nv_bfloat16 *>(smem + SM::OFF_NEW);
    float *sm_m = reinterpret_cast<float *>(smem + SM::OFF_MERGE), *sm_l = sm_m + 8 * NW, *sm_o = sm_l + 8 * NW;
    int *prefix = reinterpret_cast<int *>(smem + SM::OFF_MISC);
    int *s_flag = prefix + 34;      // [2]
    int *s_fast = prefix + 33;      // prefix[] uses 0 .. 32
    int *s_pos = prefix + 36, *s_slot = s_pos + 32;
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + SM::OFF_MISC + 100 * 4);
    uint64_t *empty_bar = full_bar + LDS_STAGES;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#define LDS_STAMP(i) do { if (dbg && lane == 0) dbg[blockIdx.x * 16 + (i)] = clock64(); } while (0)
    if (warp == 1) LDS_STAMP(0);
    griddep_launch_dependents();    // the O projection may move in and prefetch its weights as SMs free up
    if (tid == 0) {
        prefetch_tensormap(&tmap_k);
        prefetch_tensormap(&tmap_v);
        for (int s = 0; s < LDS_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 4);    // the four warps of the group that consumed the stage
        }
        fence_barrier_init();
    }
    // Context lengths, slots and the page table are constant for the whole decode step (the step's first kernel is NOT a
    // programmatic dependent, llm.cu), and cached K / V rows of earlier steps are immutable: the partition and the K / V
    // stream start right away, only q and the appended row (consumers) wait for the QKV projection.
    for (int i = tid; i < (8 - hq_r / kvh_r) * LA_LD; i += 32 + NC) Qs[(hq_r / kvh_r) * LA_LD + i] = __float2bfloat16_rn(0.f);   // heads >= G: zero columns of Q^T
    if (warp == 0) {
        int pos = 0, slot = 0, nblk = 0;
        if (lane < n_seq) {
            pos = __ldg(ctx_len + lane);
            pos = pos < max_ctx ? pos : max_ctx - 1;
            slot = __ldg(slots + lane);
            nblk = (pos + LA_BK) / LA_BK;
        }
        int incl = nblk;            // inclusive scan over the 32 lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        s_pos[lane] = pos;
        s_slot[lane] = slot;
        prefix[lane + 1] = incl;    // prefix[b] = key blocks of sequences < b (one kv head); lanes >= n_seq repeat the total
        if (lane == 0) prefix[0] = 0;
    }
    __syncthreads();
    const int T = prefix[n_seq] * kvh_r;     // <= 32 * kv heads * pages_per_seq: T * n_cta fits 32 bits
    // every CTA of the partition owns at least one block (so the parts of a sequence sit in CONSECUTIVE CTAs)
    const int n_cta = (int)gridDim.x < T ? (int)gridDim.x : T, cta = blockIdx.x;
    if (cta >= n_cta) return;
    const int f0 = (int)(((uint32_t)T * (uint32_t)cta) / (uint32_t)n_cta), f1 = (int)(((uint32_t)T * (uint32_t)(cta + 1)) / (uint32_t)n_cta);
    const int G = hq_r / kvh_r;
    const int QKV = (hq_r + 2 * kvh_r) * LA_D;
    if (warp == 1) LDS_STAMP(2);

    if (warp == 0) {
        // producer: the page ids of the next 32 blocks are fetched by the 32 lanes at once (one L2 round trip per 32
        // blocks instead of one per block in front of every TMA issue), lane 0 issues
        int stage = 0;
        uint32_t phase = 0;
        for (int fc = f0; fc < f1; fc += 32) {
            int row0 = 0;
            if (fc + lane < f1) {
                LdsWalk w;
                lds_seek(w, prefix, n_seq, kvh_r, fc + lane);
                const int page = __ldg(page_table + (int64_t)s_slot[w.b] * pages_per_seq + w.j);
                row0 = (page * kvh_r + w.h) * LA_BK;
            }
            const int cnt = (f1 - fc) < 32 ? (f1 - fc) : 32;
            for (int i = 0; i < cnt; ++i) {
                const int r0 = __shfl_sync(0xffffffffu, row0, i);
                if (lane == 0) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (fc == f0 && i == 0) LDS_STAMP(9);
                    unsigned char *st = smem + stage * LDS_STAGE_BYTES;
                    mbar_arrive_expect_tx(&full_bar[stage], LDS_STAGE_BYTES);
                    tma_load_2d(st, &tmap_k, &full_bar[stage], 0, r0);
                    tma_load_2d(st + 8192, &tmap_k, &full_bar[stage], 64, r0);
                    tma_load_2d(st + 16384, &tmap_v, &full_bar[stage], 0, r0);
                    tma_load_2d(st + 24576, &tmap_v, &full_bar[stage], 64, r0);
                }
                if (++stage == LDS_STAGES) { stage = 0; phase ^= 1; }
            }
        }
        LDS_STAMP(10);
        return;
    }

    // ------------------------------------------------------------------ consumers (NC threads)
    const int ct = tid - 32, cw = warp - 1, grp = cw >> 2, wq = cw & 3;
    const int g = lane >> 2, t = lane & 3;
    const int sw = lane & 7;        // row & 7 of every ldmatrix row this lane addresses
    LdsWalk w;
    lds_seek(w, prefix, n_seq, kvh_r, f0);
    int f = f0;
    int blk_idx = 0;                // blocks of this CTA consumed so far (both groups count all of them)
    long long wait_cycles = 0;
    int n_seg = 0;
    int n_pend = 0, pend_b[2] = {0, 0}, pend_h[2] = {0, 0}, pend_parts[2] = {0, 0}, pend_first[2] = {0, 0};   // split segments of this range (head and / or tail)
    // merge the parts of a split (b, h) from the workspace, in part order, and clear its slice of the QKV accumulator
    auto merge_from_ws = [&](int b, int h, int parts, int c_first) {
        for (int idx = ct; idx < G * 64; idx += NC) {
            const int r = idx >> 6, d = (idx & 63) * 2;
            float M = -INFINITY, num0 = 0.f, num1 = 0.f, den = 0.f;
            // in part order (the result does not depend on which CTA merges).  The first four parts -- all of them unless a
            // sequence is spread over more than four CTAs -- are loaded before the first use: one L2 round trip, not one per part
            float2 ml4[4], ov4[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                ml4[p] = make_float2(-INFINITY, 0.f);
                ov4[p] = make_float2(0.f, 0.f);
                if (p < parts) {
                    const float *pp = part_ws + ((int64_t)(c_first + p) * 2 + (p == 0 ? 1 : 0)) * 8 * LDS_PART_LD + r * LDS_PART_LD;
                    ml4[p] = __ldcg(reinterpret_cast<const float2 *>(pp + 128));
                    ov4[p] = __ldcg(reinterpret_cast<const float2 *>(pp + d));
                }
            }
            for (int p = 0; p < parts; ++p) {
                float2 ml, ov;
                if (p < 4) {
                    ml = p == 0 ? ml4[0] : p == 1 ? ml4[1] : p == 2 ? ml4[2] : ml4[3];
                    ov = p == 0 ? ov4[0] : p == 1 ? ov4[1] : p == 2 ? ov4[2] : ov4[3];
                } else {
                    const float *pp = part_ws + ((int64_t)(c_first + p) * 2) * 8 * LDS_PART_LD + r * LDS_PART_LD;
                    ml = __ldcg(reinterpret_cast<const float2 *>(pp + 128));
                    ov = __ldcg(reinterpret_cast<const float2 *>(pp + d));
                }
                const float Mn = fmaxf(M, ml.x);
                const float ca = (M == -INFINITY) ? 0.f : exp2f(M - Mn), cb = (ml.x == -INFINITY) ? 0.f : exp2f(ml.x - Mn);
                num0 = num0 * ca + ov.x * cb;
                num1 = num1 * ca + ov.y * cb;
                den = den * ca + ml.y * cb;
                M = Mn;
            }
            const float inv = den > 0.f ? 1.0f / den : 0.f;
            *reinterpret_cast<__nv_bfloat162 *>(out + (int64_t)b * ld_out + (h * G + r) * LA_D + d) = __floats2bfloat162_rn(num0 * inv, num1 * inv);
        }
        float *row = ws_qkv + (int64_t)b * QKV;
        for (int idx = ct; idx < G * LA_D; idx += NC) row[h * G * LA_D + idx] = 0.f;
        for (int idx = ct; idx < 2 * LA_D; idx += NC) row[(idx < LA_D ? hq_r + h : hq_r + kvh_r + h) * LA_D + (idx & (LA_D - 1))] = 0.f;
    };
    while (f < f1) {
        const int b = w.b, h = w.h, j0 = w.j, nb = w.nb;
        const int seg0 = f - j0;                                       // flattened index of block 0 of (b, h)
        const int j1 = (f1 - seg0) < nb ? (f1 - seg0) : nb;            // blocks [j0, j1) are ours
        const bool whole = (j0 == 0 && j1 == nb);
        int parts = 1, part = 0, c_first = cta;                        // the CTAs that share (b, h): consecutive, in block order
        if (!whole) {
            c_first = lds_owner(seg0, T, n_cta);
            parts = lds_owner(seg0 + nb - 1, T, n_cta) - c_first + 1;
            part = cta - c_first;
        }
        const int pkey = b * kvh_r + h;
        // Part 0 is the TAIL of its CTA's range (processed last), every other part the HEAD of its CTA's range (processed first):
        // the heads arrive on the pair's counter as soon as they are done, so when part 0 starts it normally finds all of them
        // in, fetches their partials WHILE it works on its own blocks and finishes the row without an arrival of its own --
        // no atomic and no dependent L2 round trip after the kernel's last block.  Anything else takes the arrival path below.
        const bool try_fast = (parts >= 2 && parts <= 4 && part == 0);
        if (n_seg == 0) {
            // QKV projection complete (q and the new k / v row are in ws_qkv) -- and with it every earlier kernel of the stream,
            // among them the previous launch of this kernel: its arrivals on part_cnt must not be read as this launch's
            griddep_wait();
            if (warp == 1) LDS_STAMP(1);
        }
        if (try_fast && ct == 0) {
            int seen;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(seen) : "l"(part_cnt + pkey) : "memory");
            *s_fast = (seen == parts - 1);
        }
        const int pos = s_pos[b];
        const int n_ctx = pos + 1;
        const bool has_last = (j1 == nb);
        const int slot = s_slot[b];
        float *row = ws_qkv + (int64_t)b * QKV;
        // ---- prologue: RoPE on the group's q heads -> Qs; the new k / v row if this segment ends the sequence.
        // Every global load is issued before the first use: one L2 round trip per segment.
        {
            const int i6 = ct & 63;
            constexpr int QIT = 512 / NC;       // G * 64 <= 512 (head, dim pair) items over NC threads
            float qx1[QIT], qx2[QIT], nx1 = 0.f, nx2 = 0.f;
            int64_t page = 0;
#pragma unroll
            for (int it = 0; it < QIT; ++it) {
                const int idx = ct + it * NC;
                qx1[it] = qx2[it] = 0.f;
                if (idx < G * 64) {
                    const float *src = row + (h * G + (idx >> 6)) * LA_D;
                    qx1[it] = __ldcg(src + i6);
                    qx2[it] = __ldcg(src + i6 + 64);
                }
            }
            const float c = __ldg(rope_cos + (int64_t)pos * 64 + i6), sv = __ldg(rope_sin + (int64_t)pos * 64 + i6);
            if (has_last && ct < 128) {
                const float *src = row + (ct < 64 ? hq_r + h : hq_r + kvh_r + h) * LA_D;
                nx1 = __ldcg(src + i6);
                nx2 = __ldcg(src + i6 + 64);
                page = __ldg(page_table + (int64_t)slot * pages_per_seq + (pos >> 6));
            }
#pragma unroll
            for (int it = 0; it < QIT; ++it) {
                const int idx = ct + it * NC;
                if (idx < G * 64) {
                    const int r = idx >> 6;
                    Qs[r * LA_LD + i6] = __float2bfloat16_rn(qx1[it] * c - qx2[it] * sv);
                    Qs[r * LA_LD + i6 + 64] = __float2bfloat16_rn(qx2[it] * c + qx1[it] * sv);
                }
            }
            if (has_last && ct < 128) {
                const int64_t app = ((page * kvh_r + h) * LA_BK + (pos & 63)) * LA_D;
                const bool is_k = ct < 64;
                const __nv_bfloat16 n1 = __float2bfloat16_rn(is_k ? nx1 * c - nx2 * sv : nx1);
                const __nv_bfloat16 n2 = __float2bfloat16_rn(is_k ? nx2 * c + nx1 * sv : nx2);
                __nv_bfloat16 *dst = is_k ? kc : vc;
                dst[app + i6] = n1;
                dst[app + i6 + 64] = n2;
                s_new[(is_k ? 0 : 128) + i6] = n1;
                s_new[(is_k ? 0 : 128) + i6 + 64] = n2;
            }
        }
        lds_bar_consumers<NC>();
        if (warp == 1 && n_seg == 0) LDS_STAMP(3);
        bool fast = try_fast && (*s_fast != 0);
        float2 pf_ml[2][3], pf_ov[2][3];        // the other parts' (m, l) and o pair for this thread's (row, dim pair) items
        auto fetch_parts = [&]() {
#pragma unroll
            for (int it = 0; it < 2; ++it) {
                const int idx = ct + it * NC;
#pragma unroll
                for (int p = 1; p < 4; ++p) {
                    pf_ml[it][p - 1] = make_float2(-INFINITY, 0.f);
                    pf_ov[it][p - 1] = make_float2(0.f, 0.f);
                    if (p < parts && idx < G * 64) {
                        const float *pp = part_ws + ((int64_t)(c_first + p) * 2) * 8 * LDS_PART_LD + (idx >> 6) * LDS_PART_LD;
                        pf_ml[it][p - 1] = __ldcg(reinterpret_cast<const float2 *>(pp + 128));
                        pf_ov[it][p - 1] = __ldcg(reinterpret_cast<const float2 *>(pp + (idx & 63) * 2));
                    }
                }
            }
        };
        if (fast) fetch_parts();
        // TRANSPOSED products (the 8 columns of an m16n8k16 tile are the q heads of the group, no padded rows):
        //   S^T[16 keys, 8 heads] = K[16 keys, 128] . Q^T        8 MMAs per warp and block (the [16 q rows] form needs 16)
        //   O^T[128 dims, 8 heads] += V^T[128, 16 keys] . P^T    8 MMAs (16)
        // the legacy tensor pipe is the busiest unit of this kernel (~29 cycles per m16n8k16 per SM sub-partition,
        // profiles/r02_llm_attn_decode_stream.txt); P^T goes from the accumulator layout of S^T to the B-operand layout
        // through two movmatrix transposes.
        uint32_t qb[16];            // B fragments of Q^T: qb[2 kk], qb[2 kk + 1] cover dims [16 kk, 16 kk + 16)
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) {
            uint32_t r4[4];
            la_ldmatrix_x4(r4, Qs + (lane & 7) * LA_LD + k2 * 32 + (lane >> 3) * 8);
            qb[k2 * 4] = r4[0]; qb[k2 * 4 + 1] = r4[1]; qb[k2 * 4 + 2] = r4[2]; qb[k2 * 4 + 3] = r4[3];
        }
        float o[8][4];              // O^T tiles: [16 dims] x [heads 2t, 2t+1]: {dim g: h0, h1, dim g + 8: h0, h1}
#pragma unroll
        for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
        float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};     // heads 2t, 2t + 1

        for (int j = j0; j < j1; ++j, ++blk_idx) {
            if (GROUPS == 2 && (blk_idx & 1) != grp) continue;
            const int stage = blk_idx % LDS_STAGES;
            const uint32_t phase = (uint32_t)(blk_idx / LDS_STAGES) & 1u;
            const long long tw0 = dbg ? clock64() : 0;
            mbar_wait(&full_bar[stage], phase);
            if (dbg) wait_cycles += clock64() - tw0;
            if (warp == 1 && blk_idx == 0) LDS_STAMP(4);
            unsigned char *st = smem + stage * LDS_STAGE_BYTES;
            if (j == nb - 1) {
                // the row appended by this step: patch it into the staged page (the TMA load may predate the append)
                const int gt = ct & 127, pr = pos & 63;
                if (gt < 32) {
                    const int c16 = gt & 15;
                    unsigned char *dst = st + (gt < 16 ? 0 : 16384) + (c16 >> 3) * 8192 + pr * 128 + (((c16 & 7) ^ (pr & 7)) << 4);
                    *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(s_new + (gt < 16 ? 0 : 128) + c16 * 8);
                }
                lds_bar_group(grp);
            }
            const int key0 = j * LA_BK + wq * 16;
            if (key0 < n_ctx) {
                const uint32_t kbase = smem_u32(st), vbase = kbase + 16384;
                float sa[4] = {0.f, 0.f, 0.f, 0.f}, sb[4] = {0.f, 0.f, 0.f, 0.f};   // two chains of four dependent MMAs
                const int krow = wq * 16 + (lane & 15);
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    uint32_t ka[4];
                    const int c16 = kk * 2 + (lane >> 4);
                    const uint32_t a = kbase + (c16 >> 3) * 8192 + krow * 128 + (((c16 & 7) ^ sw) << 4);
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                                 : "=r"(ka[0]), "=r"(ka[1]), "=r"(ka[2]), "=r"(ka[3]) : "r"(a));
                    if (kk & 1) la_mma_bf16(sb, ka, qb[2 * kk], qb[2 * kk + 1]);
                    else la_mma_bf16(sa, ka, qb[2 * kk], qb[2 * kk + 1]);
                }
                // sa[0..1]: key g, heads 2t / 2t+1;  sa[2..3]: key g + 8
                const bool va = key0 + g < n_ctx, vb8 = key0 + g + 8 < n_ctx;
                float s0 = va ? (sa[0] + sb[0]) * scale_log2e : -INFINITY, s1 = va ? (sa[1] + sb[1]) * scale_log2e : -INFINITY;
                float s2 = vb8 ? (sa[2] + sb[2]) * scale_log2e : -INFINITY, s3 = vb8 ? (sa[3] + sb[3]) * scale_log2e : -INFINITY;
                float mx[2] = {fmaxf(s0, s2), fmaxf(s1, s3)};
                float corr[2], rs[2];
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], 4));
                    mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], 8));
                    mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], 16));
                    const float m_new = fmaxf(m_run[hh], mx[hh]);   // finite: key0 < n_ctx
                    corr[hh] = exp2f(m_run[hh] - m_new);
                    m_run[hh] = m_new;
                }
                s0 = exp2f(s0 - m_run[0]); s1 = exp2f(s1 - m_run[1]);
                s2 = exp2f(s2 - m_run[0]); s3 = exp2f(s3 - m_run[1]);
                rs[0] = s0 + s2;
                rs[1] = s1 + s3;
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    rs[hh] += __shfl_xor_sync(0xffffffffu, rs[hh], 4);
                    rs[hh] += __shfl_xor_sync(0xffffffffu, rs[hh], 8);
                    rs[hh] += __shfl_xor_sync(0xffffffffu, rs[hh], 16);
                    l_run[hh] = l_run[hh] * corr[hh] + rs[hh];
                }
#pragma unroll
                for (int n = 0; n < 8; ++n) {
                    o[n][0] *= corr[0]; o[n][1] *= corr[1];
                    o[n][2] *= corr[0]; o[n][3] *= corr[1];
                }
                // P^T (keys x heads) from the accumulator layout to the B-operand layout: 8x8 transposes
                uint32_t pb0, pb1;
                {
                    const uint32_t plo = la_pack_bf16(s0, s1), phi = la_pack_bf16(s2, s3);
                    asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;\n" : "=r"(pb0) : "r"(plo));
                    asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;\n" : "=r"(pb1) : "r"(phi));
                }
                const int vrow = wq * 16 + (lane >> 4) * 8 + (lane & 7);
#pragma unroll
                for (int nd = 0; nd < 8; ++nd) {
                    uint32_t vt[4];
                    const int c16 = nd * 2 + ((lane >> 3) & 1);
                    const uint32_t a = vbase + (c16 >> 3) * 8192 + vrow * 128 + (((c16 & 7) ^ sw) << 4);
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                                 : "=r"(vt[0]), "=r"(vt[1]), "=r"(vt[2]), "=r"(vt[3]) : "r"(a));
                    la_mma_bf16(o[nd], vt, pb0, pb1);
                }
            }
            if (j == nb - 1) fence_proxy_async();   // the patched row (generic write) precedes the stage's next TMA fill
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[stage]);
        }

        if (warp == 1 && n_seg == 0) LDS_STAMP(5);
        // ---- merge the eight per-warp states of this segment (rows g < G are real)
        if (g == 0) {
            sm_m[cw * 8 + 2 * t] = m_run[0]; sm_l[cw * 8 + 2 * t] = l_run[0];
            sm_m[cw * 8 + 2 * t + 1] = m_run[1]; sm_l[cw * 8 + 2 * t + 1] = l_run[1];
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int head = 2 * t + hh;
            if (head < G) {
                float *dst = sm_o + (cw * G + head) * LDS_MERGE_LD + g;
#pragma unroll
                for (int n = 0; n < 8; ++n) {
                    dst[n * 16] = o[n][hh];
                    dst[n * 16 + 8] = o[n][2 + hh];
                }
            }
        }
        // second chance for a tail part that started before its heads were in (a range that is ONE tail segment starts with the
        // kernel): if they have arrived by now, fetch their partials here -- one L2 round trip, still no arrival of its own
        if (try_fast && !fast && ct == 0) {
            int seen;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(seen) : "l"(part_cnt + pkey) : "memory");
            *s_fast = (seen == parts - 1);
        }
        lds_bar_consumers<NC>();
        if (try_fast && !fast && *s_fast != 0) {
            fast = true;
            fetch_parts();
        }
        float *my_part = part_ws + ((int64_t)cta * 2 + (part == 0 ? 1 : 0)) * 8 * LDS_PART_LD;
#pragma unroll
        for (int it = 0; it < 2; ++it) {                    // (row, dim pair) items: G * 64 <= 2 NC
            const int idx = ct + it * NC;
            if (idx >= G * 64) break;
            const int r = idx >> 6, d = (idx & 63) * 2;
            float M = -INFINITY;
#pragma unroll
            for (int x = 0; x < NW; ++x) M = fmaxf(M, sm_m[x * 8 + r]);
            float num0 = 0.f, num1 = 0.f, den = 0.f;
#pragma unroll
            for (int x = 0; x < NW; ++x) {
                const float mw = sm_m[x * 8 + r];
                const float wgt = (mw == -INFINITY) ? 0.f : exp2f(mw - M);
                const float2 ov = *reinterpret_cast<const float2 *>(sm_o + (x * G + r) * LDS_MERGE_LD + d);
                num0 = fmaf(wgt, ov.x, num0);
                num1 = fmaf(wgt, ov.y, num1);
                den = fmaf(wgt, sm_l[x * 8 + r], den);
            }
            if (fast) {
                // this CTA holds part 0 in registers and the other parts prefetched: merge in part order (same arithmetic, same
                // order as merge_from_ws below: the row's bits do not depend on which path finished it)
                float Mr = M, n0 = num0, n1 = num1, dn = den;
#pragma unroll
                for (int p = 1; p < 4; ++p) {
                    if (p < parts) {
                        const float2 ml = pf_ml[it][p - 1], ov = pf_ov[it][p - 1];
                        const float Mn = fmaxf(Mr, ml.x);
                        const float ca = (Mr == -INFINITY) ? 0.f : exp2f(Mr - Mn), cb = (ml.x == -INFINITY) ? 0.f : exp2f(ml.x - Mn);
                        n0 = n0 * ca + ov.x * cb;
                        n1 = n1 * ca + ov.y * cb;
                        dn = dn * ca + ml.y * cb;
                        Mr = Mn;
                    }
                }
                M = Mr; num0 = n0; num1 = n1; den = dn;
            }
            if (parts == 1 || fast) {
                const float inv = den > 0.f ? 1.0f / den : 0.f;
                *reinterpret_cast<__nv_bfloat162 *>(out + (int64_t)b * ld_out + (h * G + r) * LA_D + d) = __floats2bfloat162_rn(num0 * inv, num1 * inv);
            } else {
                __stcg(reinterpret_cast<float2 *>(my_part + r * LDS_PART_LD + d), make_float2(num0, num1));
                if (d == 0) __stcg(reinterpret_cast<float2 *>(my_part + r * LDS_PART_LD + 128), make_float2(M, den));
            }
        }
        if (parts == 1 || fast) {
            // this CTA finished (b, h): clear its slice of the accumulator for the next layer's projection
            for (int idx = ct; idx < G * LA_D; idx += NC) row[h * G * LA_D + idx] = 0.f;
            for (int idx = ct; idx < 2 * LA_D; idx += NC) row[(idx < LA_D ? hq_r + h : hq_r + kvh_r + h) * LA_D + (idx & (LA_D - 1))] = 0.f;
            if (fast && ct == 0) part_cnt[pkey] = 0;        // every part has arrived: nobody touches the counter again in this launch
        } else if (part > 0) {
            // a HEAD part: arrive now (release / acquire at GPU scope by one thread between CTA barriers), the tail finds it in
            lds_bar_consumers<NC>();
            if (ct == 0) {
                int old;
                asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;\n" : "=r"(old) : "l"(part_cnt + pkey) : "memory");
                const int last = (old == parts - 1);
                if (last) part_cnt[pkey] = 0;
                s_flag[0] = last;
            }
            lds_bar_consumers<NC>();
            if (s_flag[0]) merge_from_ws(b, h, parts, c_first);   // the tail had already arrived (it took the arrival path)
        } else {
            // the TAIL part without the fast path: arrival after the range (one fence + one atomic round trip per CTA)
            if (n_pend == 0) { pend_b[0] = b; pend_h[0] = h; pend_parts[0] = parts; pend_first[0] = c_first; }
            else { pend_b[1] = b; pend_h[1] = h; pend_parts[1] = parts; pend_first[1] = c_first; }
            ++n_pend;
        }
        lds_bar_consumers<NC>();        // merge area, Qs and s_new are free for the next segment
        if (warp == 1 && n_seg == 0) LDS_STAMP(6);
        ++n_seg;
        // advance the walk to the next segment
        f += j1 - j0;
        if (f < f1) {
            w.j = j1 - 1;
            lds_next(w, prefix, kvh_r);
        }
    }

    if (warp == 1) {
        LDS_STAMP(7);
        if (dbg && lane == 0) { dbg[blockIdx.x * 16 + 11] = wait_cycles; dbg[blockIdx.x * 16 + 12] = n_seg; dbg[blockIdx.x * 16 + 13] = blk_idx; }
    }
    // ---- arrivals of the split segments; the last CTA to arrive for a (b, h) merges its parts in part order
    if (n_pend == 0) return;
    // release / acquire at GPU scope by one thread per split segment, CTA barriers on both sides: every partial this CTA
    // stored happens-before the arrival, and the merging CTA's reads happen-after the last arrival it observed
    lds_bar_consumers<NC>();
    if (ct < n_pend) {
        const int key = (ct == 0 ? pend_b[0] : pend_b[1]) * kvh_r + (ct == 0 ? pend_h[0] : pend_h[1]);
        int old;
        asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;\n" : "=r"(old) : "l"(part_cnt + key) : "memory");
        const int last = (old == (ct == 0 ? pend_parts[0] : pend_parts[1]) - 1);
        if (last) part_cnt[key] = 0;        // the next layer's launch is ordered after this kernel
        s_flag[ct] = last;
    }
    lds_bar_consumers<NC>();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        if (i >= n_pend || !s_flag[i]) continue;
        merge_from_ws(pend_b[i], pend_h[i], pend_parts[i], pend_first[i]);
    }
    if (warp == 1) LDS_STAMP(8);
#undef LDS_STAMP
}

// decode attention fused with RoPE + KV append: reads (and clears) the fp32 QKV accumulator [32, (hq+2hkv)*128]
int llm_attn_decode(cudaStream_t st, float *ws_qkv, void *kc, void *vc, const int32_t *ctx_len, const int32_t *slots,
                    const int32_t *page_table, int pages_per_seq, const float *rope_cos, const float *rope_sin, void *out,
                    int ld_out, int n_seq, int hq_r, int kvh_r, int max_ctx, float scale, const CUtensorMap *tmap_k,
                    const CUtensorMap *tmap_v, float *part_ws, int *part_cnt, int n_cta, int stream_form)
{
    if (n_seq <= 0) return 0;
    const int G = hq_r / kvh_r;
    if (G < 1 || G > 8 || G * kvh_r != hq_r) return fail(B2S_ERR_INVALID, "llm attention: query group size %d not supported (1..8)", G);
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, []() {
        attr_err = cudaFuncSetAttribute(llm_attn_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LDM_SMEM);
        if (attr_err == cudaSuccess)
            attr_err = cudaFuncSetAttribute(llm_attn_decode_stream_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdsSmem<3, 1>::total(4));
        if (attr_err == cudaSuccess)
            attr_err = cudaFuncSetAttribute(llm_attn_decode_stream_kernel<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, LdsSmem<4, 2>::total(8));
    });
    if (attr_err != cudaSuccess) return fail_cuda(attr_err, "cudaFuncSetAttribute(llm decode attention)");
    cudaLaunchConfig_t cfg = {};
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (stream_form && tmap_k && tmap_v && part_ws && part_cnt && n_cta > 0) {
        // developer aid (B2S_LLM_ATTN_TIMING=<launch number>): SM-clock stamps of every CTA of that launch, summarised on stderr
        static const long timing_at = []() { const char *e = getenv("B2S_LLM_ATTN_TIMING"); return e ? atol(e) : 0L; }();
        static long n_launch = 0;
        static long long *dbg = nullptr;
        long long *dbg_arg = nullptr;
        if (timing_at > 0 && ++n_launch == timing_at) {
            if (!dbg) cudaMalloc(&dbg, (size_t)n_cta * 2 * 16 * 8);
            cudaMemsetAsync(dbg, 0, (size_t)n_cta * 2 * 16 * 8, st);
            dbg_arg = dbg;
        }
        const bool two_per_sm = G <= 4;         // n_cta = SM count; the workspace holds 2 slots for each of 2 * n_cta CTAs
        // B2S_LLM_ATTN_CTAS_PER_SM=1: launch the 2-per-SM shape with one CTA per SM (fewer, longer ranges: fewer split sequences)
        static const int per_sm = []() { const char *e = getenv("B2S_LLM_ATTN_CTAS_PER_SM"); return (e && e[0] == '1') ? 1 : 2; }();
        const int grid = two_per_sm ? per_sm * n_cta : n_cta;
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(two_per_sm ? 160 : 288);
        cfg.dynamicSmemBytes = two_per_sm ? LdsSmem<3, 1>::total(G) : LdsSmem<4, 2>::total(G);
        B2S_CUDA(cudaLaunchKernelEx(&cfg, two_per_sm ? llm_attn_decode_stream_kernel<3, 1> : llm_attn_decode_stream_kernel<4, 2>, *tmap_k, *tmap_v, ws_qkv, static_cast<__nv_bfloat16 *>(kc),
                                    static_cast<__nv_bfloat16 *>(vc), ctx_len, slots, page_table, pages_per_seq, rope_cos, rope_sin,
                                    static_cast<__nv_bfloat16 *>(out), ld_out, n_seq, hq_r, kvh_r, max_ctx,
                                    scale * 1.4426950408889634f, part_ws, part_cnt, dbg_arg));
        count_launch();
        if (dbg_arg) {
            const int n_cta = grid;   // shadows the SM count: the stamps are per launched CTA
            std::vector<long long> h((size_t)n_cta * 16);
            cudaStreamSynchronize(st);
            cudaMemcpy(h.data(), dbg, h.size() * 8, cudaMemcpyDeviceToHost);
            static const char *const names[] = {"entry", "dep_wait", "partition", "q_ready(seg0)", "first_block_landed", "seg0_blocks_done",
                                                "seg0_merged", "range_done", "kernel_end", "producer_first_issue", "producer_last_issue"};
            fprintf(stderr, "llm decode attention (stream form) stamps, SM cycles since CTA entry, over %d CTAs: median [min .. max]\n", n_cta);
            for (int i = 1; i <= 10; ++i) {
                std::vector<long long> v;
                for (int c = 0; c < n_cta; ++c)
                    if (h[(size_t)c * 16 + i]) v.push_back(h[(size_t)c * 16 + i] - h[(size_t)c * 16]);
                if (v.empty()) continue;
                std::sort(v.begin(), v.end());
                fprintf(stderr, "  %-22s %8lld [%8lld .. %8lld]  (%zu CTAs)\n", names[i], v[v.size() / 2], v.front(), v.back(), v.size());
            }
            for (int i = 11; i <= 13; ++i) {
                std::vector<long long> v;
                for (int c = 0; c < n_cta; ++c) v.push_back(h[(size_t)c * 16 + i]);
                std::sort(v.begin(), v.end());
                fprintf(stderr, "  %-22s %8lld [%8lld .. %8lld]\n", i == 11 ? "warp1 full-wait cycles" : i == 12 ? "segments" : "blocks", v[v.size() / 2],
                        v.front(), v.back());
            }
        }
        return 0;
    }
    cfg.gridDim = dim3((unsigned)n_seq, (unsigned)kvh_r);
    cfg.blockDim = dim3(128);
    cfg.dynamicSmemBytes = LDM_SMEM;
    B2S_CUDA(cudaLaunchKernelEx(&cfg, llm_attn_decode_kernel, ws_qkv, static_cast<__nv_bfloat16 *>(kc), static_cast<__nv_bfloat16 *>(vc),
                                ctx_len, slots, page_table, pages_per_seq, rope_cos, rope_sin, static_cast<__nv_bfloat16 *>(out), ld_out,
                                hq_r, kvh_r, max_ctx, scale * 1.4426950408889634f));
    count_launch();
    return 0;
}

}  // namespace b2s
