// llm.cu -- decoder-only transformer executor (Llama family) for the tensor-parallel LLM endpoint of
// BASELINE.json configs[4].  In the reference this endpoint is `VllmPreprocessRequest`
// (clearml_serving/serving/preprocess_service.py:1097-1348), a thin wrapper that hands prompts to vLLM; here the
// model runs on the library's own kernels:
//   prefill : RMSNorm -> QKV GEMM (tcgen05, gemm.cu) -> RoPE + KV-cache write -> causal GQA attention
//             (llm_attention.cu) -> O GEMM -> [TP all-reduce] + residual + RMSNorm -> gate/up GEMM -> SwiGLU ->
//             down GEMM -> [TP all-reduce] + residual + RMSNorm ... -> lm_head -> greedy argmax
//   decode  : the same chain for <= 32 running sequences, every projection on the weight-streaming stream-K
//             kernel of skinny.cu; one decode step is captured in a CUDA graph (context lengths, positions and
//             the step counter live in device memory, so the same graph replays for every step).
// Tensor parallelism (Megatron split: QKV / gate / up by output rows, O / down by input columns, lm_head by
// vocabulary) runs as ONE PROCESS PER GPU.  The row-parallel partial sums are exchanged through peer memory
// (cudaIpc handles swapped by the host side over torch.distributed): the kernel that consumes a partial sum --
// residual add + RMSNorm -- reads the peer's half directly over NVLink and adds it on the fly, so the
// all-reduce is fused into its consumer and no NCCL call sits on the data path.  With two ranks each direction
// of the link carries exactly the bytes a reduce-scatter + all-gather would.
// Synchronisation: a monotonically increasing step counter `gen` in device memory and one flag word per
// exchange point; a rank publishes flag[k] = gen + 1 in the PEER's memory once its partial for point k is
// complete and spins (bounded) on its own flag[k].  Partial buffers alternate between two copies so a buffer
// is only rewritten after the peer has signalled the NEXT exchange point, i.e. finished reading it.
//
// Layouts: weights bf16 [out, in] as nn.Linear stores them; residual stream fp32 [T, H]; KV cache per layer
// K, V = PAGED: [page][kv_head][64][128] bf16 + a page table [slot][pages_per_seq] (llm_attention.cu); decode accumulators fp32 [32, N].
#include "common.cuh"
#include "sm100.cuh"

#include <cuda.h>
#include <cuda_bf16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

namespace b2s {

int gemm_tn(cudaStream_t st, const void *A, int64_t lda, const void *B, int64_t ldb, int M, int N, int K,
            const GemmEpilogue &ep);
int skinny_make_maps(CUtensorMap *tw, CUtensorMap *tx, const void *W, int64_t n_out, int64_t K, const void *X, int64_t x_rows);
int skinny_gemm_maps(cudaStream_t st, const CUtensorMap &tw, const CUtensorMap &tx, float *y, int n_out, int K, int m_rows,
                     const uint32_t *idle_flag = nullptr, const uint32_t *gen = nullptr, int idle_want = 0, float *y_peer = nullptr,
                     uint32_t *peer_done = nullptr, int *grid_out = nullptr);
int llm_attn_prefill(cudaStream_t st, const void *qkv, int ld_qkv, const void *kc, const void *vc, const int32_t *cu_seqlens,
                     const int32_t *slots, const int32_t *page_table, int pages_per_seq, void *out, int ld_out, int n_seq,
                     int max_seqlen, int hq_r, int kvh_r, float scale);
int llm_attn_decode(cudaStream_t st, float *ws_qkv, void *kc, void *vc, const int32_t *ctx_len, const int32_t *slots,
                    const int32_t *page_table, int pages_per_seq, const float *rope_cos, const float *rope_sin, void *out,
                    int ld_out, int n_seq, int hq_r, int kvh_r, int max_ctx, float scale, const CUtensorMap *tmap_k,
                    const CUtensorMap *tmap_v, float *part_ws, int *part_cnt, int n_cta, int stream_form);
int make_tmap_2d_kmajor(CUtensorMap *out, const void *base, int64_t rows, int64_t K, int64_t ld_elems, int box_rows, int is_bf16);

constexpr int LLM_MAXB = 32;          // decode batch (rows of the skinny GEMM)
constexpr int LLM_HD = 128;           // head dim
constexpr int LLM_FLAGS = 512;

// ------------------------------------------------------------------------------------------------
// deterministic on-device initialisation: value(tensor, row, col) is a pure integer function of the GLOBAL
// coordinates, so every tensor-parallel layout of the same model holds the same numbers (and numpy can
// reproduce them bit for bit: tests/test_llm_host.py)
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline uint64_t llm_mix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// Irwin-Hall(4) of 16-bit uniforms: mean 0, std 1 after scaling; exact in fp32
__host__ __device__ inline float llm_init_value(uint64_t seed, uint32_t tensor_id, uint32_t row, uint32_t col, float std)
{
    const uint64_t r = llm_mix64(seed ^ ((uint64_t)tensor_id << 48) ^ ((uint64_t)row << 24) ^ (uint64_t)col);
    const int32_t s = (int32_t)(r & 0xFFFF) + (int32_t)((r >> 16) & 0xFFFF) + (int32_t)((r >> 32) & 0xFFFF) +
                      (int32_t)((r >> 48) & 0xFFFF) - 2 * 65535;
    return (float)s * (std * (1.7320508f / 65536.0f));   // Var[sum of 4 U(0,65536)] = 65536^2 / 3
}

__global__ void __launch_bounds__(256)
llm_fill_kernel(__nv_bfloat16 *__restrict__ w, int64_t rows, int64_t cols, uint64_t seed, uint32_t tensor_id,
                uint32_t row0, uint32_t col0, float std)
{
    const int64_t n = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        w[i] = __float2bfloat16_rn(llm_init_value(seed, tensor_id, row0 + (uint32_t)r, col0 + (uint32_t)c, std));
    }
}
// fused gate/up weight [2 * I_r, H]: fused row 64j + w is gate row 32j + w (w < 32) or up row 32j + w - 32
__global__ void __launch_bounds__(256)
llm_fill_gate_up_kernel(__nv_bfloat16 *__restrict__ w, int64_t I_r, int64_t cols, uint64_t seed, uint32_t id_gate, uint32_t id_up,
                        uint32_t row0, float std)
{
    const int64_t n = 2 * I_r * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        const int64_t blk = r >> 6, within = r & 63;
        const bool up = within >= 32;
        const uint32_t src_row = row0 + (uint32_t)(blk * 32 + (within & 31));
        w[i] = __float2bfloat16_rn(llm_init_value(seed, up ? id_up : id_gate, src_row, (uint32_t)c, std));
    }
}
__global__ void __launch_bounds__(256) llm_fill_const_kernel(float *__restrict__ w, int64_t n, float v)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) w[i] = v;
}

// ------------------------------------------------------------------------------------------------
// peer-memory primitives
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// peer data must never be served from this SM's L1 (the same addresses are rewritten every step)
__device__ __forceinline__ uint4 ld_peer_v4(const void *p)
{
    uint4 v;
    asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint2 ld_peer_v2(const void *p)
{
    uint2 v;
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0,%1}, [%2];\n" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}

// Exchange point k of the current step: tell the peer our partial is complete, wait until its is.  All threads
// of the CTA call this; returns after a __syncthreads().  `gen` is read from device memory (stable during a step).
__device__ __forceinline__ void tp_exchange_point(uint32_t *my_flags, uint32_t *peer_flags, const uint32_t *gen, int k)
{
    if (peer_flags == nullptr) return;
    if (threadIdx.x == 0) {
        const uint32_t want = *reinterpret_cast<const volatile uint32_t *>(gen) + 1u;
        if (blockIdx.x == 0) st_release_sys(peer_flags + k, want);   // release at system scope: the partial (previous kernel, in L2) is ordered before the flag
        const long long t0 = clock64();
        while ((int32_t)(ld_acquire_sys(my_flags + k) - want) < 0) {
            if (clock64() - t0 > 20000000000ll) __trap();   // ~10 s: a lost peer must not hang the GPU
            __nanosleep(64);
        }
    }
    __syncthreads();
}

__device__ __forceinline__ float block_sum_256(float v, float *red /*[8]*/)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    return t;
}

// ------------------------------------------------------------------------------------------------
// embedding gather + first RMSNorm.  One CTA (256 threads) per token; H <= 8192, H % 4 == 0.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
llm_embed_rms_kernel(const int32_t *__restrict__ tokens, const __nv_bfloat16 *__restrict__ embed, const float *__restrict__ w,
                     float *__restrict__ h, __nv_bfloat16 *__restrict__ xn, int H, int vocab, float eps)
{
    __shared__ float red[8];
    sm100::griddep_launch_dependents();   // the projection that follows may start prefetching its weights
    sm100::griddep_wait();                // no-op unless launched as a programmatic dependent
    const int t = blockIdx.x;
    int tok = __ldg(tokens + t);
    tok = tok < 0 ? 0 : (tok >= vocab ? vocab - 1 : tok);
    const __nv_bfloat16 *e = embed + (int64_t)tok * H;
    float4 v[8];
    float ss = 0.f;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        if (i < H) {
            const uint2 u = *reinterpret_cast<const uint2 *>(e + i);
            const __nv_bfloat162 *p = reinterpret_cast<const __nv_bfloat162 *>(&u);
            const float2 a = __bfloat1622float2(p[0]), c = __bfloat1622float2(p[1]);
            v[it] = make_float4(a.x, a.y, c.x, c.y);
            *reinterpret_cast<float4 *>(h + (int64_t)t * H + i) = v[it];
            ss += a.x * a.x + a.y * a.y + c.x * c.x + c.y * c.y;
        }
    }
    const float inv = rsqrtf(block_sum_256(ss, red) / (float)H + eps);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        if (i < H) {
            const float4 g = __ldg(reinterpret_cast<const float4 *>(w + i));
            __nv_bfloat162 o0 = __floats2bfloat162_rn(v[it].x * inv * g.x, v[it].y * inv * g.y);
            __nv_bfloat162 o1 = __floats2bfloat162_rn(v[it].z * inv * g.z, v[it].w * inv * g.w);
            uint2 u;
            u.x = *reinterpret_cast<uint32_t *>(&o0);
            u.y = *reinterpret_cast<uint32_t *>(&o1);
            *reinterpret_cast<uint2 *>(xn + (int64_t)t * H + i) = u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// [TP all-reduce of a row-parallel partial] + residual add + RMSNorm, fused.  One CTA per token.
//   F32 = false (prefill): partial is bf16 [T, H];   F32 = true (decode): partial is fp32 [32, H] accumulated by
//   the skinny GEMM; the OLDER decode partial buffer (`zero_buf`) is cleared for the GEMM after next.
// h += mine + peer;  xn = bf16( h * rsqrt(mean(h^2) + eps) * w )
// ------------------------------------------------------------------------------------------------
template <bool F32>
__global__ void __launch_bounds__(256)
llm_reduce_rms_kernel(const void *__restrict__ mine, const void *peer, float *zero_buf, uint32_t *my_flags, uint32_t *peer_flags,
                      const uint32_t *gen, int k, const float *__restrict__ w, float *__restrict__ h,
                      __nv_bfloat16 *__restrict__ xn, int H, float eps, uint32_t *idle_flag, const uint32_t *pushed_cnt = nullptr,
                      const uint32_t *dstep = nullptr, int pushes_per_step = 0, int data_pushed = 0, float *mail_out = nullptr,
                      float *mail_in = nullptr)
{
    __shared__ float red[8];
    sm100::griddep_launch_dependents();
    // the norm weights are constants: fetched before the dependency resolves instead of after the row reduction (one L2 round trip
    // less on the step's critical path, twice per layer)
    float4 gam[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        gam[it] = i < H ? __ldg(reinterpret_cast<const float4 *>(w + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    sm100::griddep_wait();
    // the projection before this kernel has completed: tell the NEXT projection (already resident, ring full, spinning before its
    // own dependency wait) that HBM is idle for the next few microseconds (skinny.cu)
    if (idle_flag && blockIdx.x == 0 && threadIdx.x == 0)
        *reinterpret_cast<volatile uint32_t *>(idle_flag) = *reinterpret_cast<const volatile uint32_t *>(gen) * 1024u + (uint32_t)(k + 1);
    // Decode exchange, COUNT form (B2S_LLM_TP_PUSH=0): every CTA of the peer's projection counts itself on pushed_cnt[k] when its partial
    // sums are out (red.release.sys after its epilogue); once (step + 1) x grid counts are in, the peer's partial is complete and
    // is read over NVLink -- without waiting for the peer's NEXT kernel (this one, on its side) to start and send a flag.
    // PUSH form (data_pushed, B2S_LLM_TP_PUSH=1, slower): the peer has also ADDED its partial into `mine`: no peer read.
    // FLAG form (default, and the prefill): tp_exchange_point, then the peer's partial is read.  Measured 2.57 / 2.78 / 3.21 ms per
    // TP2 decode step for flag / count / push: system-scope traffic inside the projection costs more than it saves.
    // MAIL form (default for the decode, B2S_LLM_TP_PUSH=2): no flag at all.  Each rank stores its partial row into the PEER's
    // mailbox (plain 16-byte stores over NVLink) and polls its OWN mailbox, whose slots hold a sentinel until the peer's values
    // land: the value is its own arrival flag (the forest kernel's row exchange, across two GPUs).  One NVLink flight instead of
    // flag flight + poll + read round trip.
    const bool mailed = F32 && mail_in != nullptr;
    const bool pushed = F32 && !mailed && pushed_cnt != nullptr;
    if (mailed) {
        peer = nullptr;
    } else if (pushed) {
        if (threadIdx.x == 0) {
            const uint32_t want = (*reinterpret_cast<const volatile uint32_t *>(dstep) + 1u) * (uint32_t)pushes_per_step;
            const long long t0 = clock64();
            while ((int32_t)(ld_acquire_sys(pushed_cnt + k) - want) < 0) {
                if (clock64() - t0 > 20000000000ll) __trap();   // ~10 s: a lost peer must not hang the GPU
                __nanosleep(32);
            }
        }
        __syncthreads();
        if (data_pushed) peer = nullptr;        // else: COUNT form -- the count replaces the flag, the partial is still pulled
    } else {
        tp_exchange_point(my_flags, peer_flags, gen, k);
    }
    const int t = blockIdx.x;
    // Every load of the row is issued before the first use: the peer's partial comes over NVLink (~2.5 us per round trip), and
    // a load -> add -> store loop pays that once per 1024 columns (4 round trips at H = 4096: 10 of the 15 us this kernel took in
    // the TP 2 step, profiles/r02_llm_decode_trace_tp2.txt); the volatile peer loads also pinned the local loads behind them.
    float4 v[8], pa[8], pr[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        pr[it] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < H && peer) {
            if (F32) {
                const uint4 u = ld_peer_v4(static_cast<const float *>(peer) + (int64_t)t * H + i);
                pr[it] = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
            } else {
                const uint2 q = ld_peer_v2(static_cast<const __nv_bfloat16 *>(peer) + (int64_t)t * H + i);
                const __nv_bfloat162 *pq = reinterpret_cast<const __nv_bfloat162 *>(&q);
                const float2 q0 = __bfloat1622float2(pq[0]), q1 = __bfloat1622float2(pq[1]);
                pr[it] = make_float4(q0.x, q0.y, q1.x, q1.y);
            }
        }
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        pa[it] = v[it] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < H) {
            if (F32) {
                pa[it] = __ldcg(reinterpret_cast<const float4 *>(static_cast<const float *>(mine) + (int64_t)t * H + i));
            } else {
                const uint2 u = *reinterpret_cast<const uint2 *>(static_cast<const __nv_bfloat16 *>(mine) + (int64_t)t * H + i);
                const __nv_bfloat162 *p = reinterpret_cast<const __nv_bfloat162 *>(&u);
                const float2 m0 = __bfloat1622float2(p[0]), m1 = __bfloat1622float2(p[1]);
                pa[it] = make_float4(m0.x, m0.y, m1.x, m1.y);
            }
            v[it] = *reinterpret_cast<const float4 *>(h + (int64_t)t * H + i);
        }
    }
    if (mailed) {
        constexpr uint32_t EMPTY = 0xffffffffu;     // a NaN no computation produces; an (impossible) equal value is sent as 0x7fffffff
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int i = (it * 256 + threadIdx.x) * 4;
            if (i < H) {
                uint32_t a0 = __float_as_uint(pa[it].x), a1 = __float_as_uint(pa[it].y), a2 = __float_as_uint(pa[it].z), a3 = __float_as_uint(pa[it].w);
                a0 = a0 == EMPTY ? 0x7fffffffu : a0; a1 = a1 == EMPTY ? 0x7fffffffu : a1;
                a2 = a2 == EMPTY ? 0x7fffffffu : a2; a3 = a3 == EMPTY ? 0x7fffffffu : a3;
                asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%2,%3,%4};\n" ::"l"(mail_out + (int64_t)t * H + i), "r"(a0), "r"(a1), "r"(a2), "r"(a3) : "memory");
            }
        }
        const long long t0 = clock64();
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int i = (it * 256 + threadIdx.x) * 4;
            if (i < H) {
                float *slot = mail_in + (int64_t)t * H + i;
                uint4 u;
                for (;;) {
                    u = ld_peer_v4(slot);       // relaxed, system scope: never served from L1
                    if (u.x != EMPTY && u.y != EMPTY && u.z != EMPTY && u.w != EMPTY) break;
                    if (clock64() - t0 > 20000000000ll) __trap();   // ~10 s: a lost peer must not hang the GPU
                }
                pr[it] = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
                // empty the slot for exchange k + 2 (the peer writes it again only after it has seen this rank's push for k + 1)
                asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%1,%1,%1};\n" ::"l"(slot), "r"(EMPTY) : "memory");
            }
        }
    }
    float ss = 0.f;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        if (i < H) {
            float4 r = v[it];
            r.x += pa[it].x + pr[it].x; r.y += pa[it].y + pr[it].y; r.z += pa[it].z + pr[it].z; r.w += pa[it].w + pr[it].w;
            if (F32 && zero_buf) *reinterpret_cast<float4 *>(zero_buf + (int64_t)t * H + i) = make_float4(0.f, 0.f, 0.f, 0.f);   // pull: the OLDER buffer; push: `mine` itself
            *reinterpret_cast<float4 *>(h + (int64_t)t * H + i) = r;
            v[it] = r;
            ss += r.x * r.x + r.y * r.y + r.z * r.z + r.w * r.w;
        }
    }
    const float inv = rsqrtf(block_sum_256(ss, red) / (float)H + eps);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int i = (it * 256 + threadIdx.x) * 4;
        if (i < H) {
            const float4 g = gam[it];
            __nv_bfloat162 o0 = __floats2bfloat162_rn(v[it].x * inv * g.x, v[it].y * inv * g.y);
            __nv_bfloat162 o1 = __floats2bfloat162_rn(v[it].z * inv * g.z, v[it].w * inv * g.w);
            uint2 u;
            u.x = *reinterpret_cast<uint32_t *>(&o0);
            u.y = *reinterpret_cast<uint32_t *>(&o1);
            *reinterpret_cast<uint2 *>(xn + (int64_t)t * H + i) = u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// RoPE (rotate-half convention: pairs (i, i + 64)) on q and k, K/V append to the cache.  One CTA per token.
//   prefill: qkv bf16 [T, QKV] -- q rotated in place, position = tok_pos[t], slot = slots[tok_seq[t]]
//   decode : fused into the attention kernel's prologue (llm_attention.cu)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
llm_rope_cache_prefill_kernel(__nv_bfloat16 *__restrict__ qkv, __nv_bfloat16 *__restrict__ kc, __nv_bfloat16 *__restrict__ vc,
                              const int32_t *__restrict__ tok_seq, const int32_t *__restrict__ tok_pos,
                              const int32_t *__restrict__ slots, const int32_t *__restrict__ page_table, int pages_per_seq,
                              const float *__restrict__ rope_cos, const float *__restrict__ rope_sin, int hq_r, int kvh_r, int max_ctx)
{
    const int t = blockIdx.x;
    const int QKV = (hq_r + 2 * kvh_r) * LLM_HD;
    const int seq = __ldg(tok_seq + t);
    int pos = __ldg(tok_pos + t);
    pos = pos < max_ctx ? pos : max_ctx - 1;
    const int slot = __ldg(slots + seq);
    // paged cache: token `pos` of this slot lives in page page_table[slot][pos / 64], row pos % 64
    const int64_t page = __ldg(page_table + (int64_t)slot * pages_per_seq + (pos >> 6));
    const int prow = pos & 63;
    const float *cs = rope_cos + (int64_t)pos * 64, *sn = rope_sin + (int64_t)pos * 64;
    __nv_bfloat16 *srcb = qkv + (int64_t)t * QKV;
    const int n_rot = (hq_r + kvh_r) * 64;   // q heads first, then k heads: contiguous in the QKV row
    for (int idx = threadIdx.x; idx < n_rot; idx += 256) {
        const int head = idx >> 6, i = idx & 63;
        const int c0 = head * LLM_HD + i;
        const float x1 = __bfloat162float(srcb[c0]), x2 = __bfloat162float(srcb[c0 + 64]);
        const float c = cs[i], sv = sn[i];
        const __nv_bfloat16 o1 = __float2bfloat16_rn(x1 * c - x2 * sv), o2 = __float2bfloat16_rn(x2 * c + x1 * sv);
        if (head < hq_r) {
            srcb[c0] = o1;
            srcb[c0 + 64] = o2;
        } else {
            __nv_bfloat16 *dst = kc + ((page * kvh_r + (head - hq_r)) * 64 + prow) * LLM_HD;
            dst[i] = o1;
            dst[i + 64] = o2;
        }
    }
    const int v0 = (hq_r + kvh_r) * LLM_HD;
    for (int idx = threadIdx.x; idx < kvh_r * LLM_HD; idx += 256) {
        const int kh = idx >> 7, d = idx & 127;
        vc[((page * kvh_r + kh) * 64 + prow) * LLM_HD + d] = srcb[v0 + idx];
    }
}

// ------------------------------------------------------------------------------------------------
// SwiGLU: act = silu(gate) * up.  The fused gate/up weight interleaves its rows in blocks of 32 (fused columns
// [64j, 64j+32) = gate_{32j..}, [64j+32, 64j+64) = up_{32j..}) so that the prefill GEMM can apply SwiGLU in its
// epilogue (gemm.cu, epilogue_swiglu32).  This kernel is the decode form: it reads (and clears) the fp32
// accumulator [32, 2I] of the skinny GEMM.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float silu_mul(float g, float u) { return g / (1.0f + __expf(-g)) * u; }

__global__ void __launch_bounds__(256)
llm_swiglu_decode_kernel(float *__restrict__ gu, __nv_bfloat16 *__restrict__ act, int64_t rows, int I, uint32_t *idle_flag,
                         const uint32_t *gen, int idle_id)
{
    sm100::griddep_launch_dependents();
    sm100::griddep_wait();
    if (idle_flag && blockIdx.x == 0 && threadIdx.x == 0)     // see llm_reduce_rms_kernel
        *reinterpret_cast<volatile uint32_t *>(idle_flag) = *reinterpret_cast<const volatile uint32_t *>(gen) * 1024u + (uint32_t)idle_id;
    const int64_t n4 = rows * (I / 4);
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n4; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / (I / 4);
        const int c = (int)(idx - r * (I / 4)) * 4;                 // output column (multiple of 4)
        float *gp = gu + r * 2 * I + (c >> 5) * 64 + (c & 31);     // gate; up is 32 columns further
        const float4 g = *reinterpret_cast<float4 *>(gp), u = *reinterpret_cast<float4 *>(gp + 32);
        *reinterpret_cast<float4 *>(gp) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4 *>(gp + 32) = make_float4(0.f, 0.f, 0.f, 0.f);
        __nv_bfloat162 o0 = __floats2bfloat162_rn(silu_mul(g.x, u.x), silu_mul(g.y, u.y));
        __nv_bfloat162 o1 = __floats2bfloat162_rn(silu_mul(g.z, u.z), silu_mul(g.w, u.w));
        uint2 o;
        o.x = *reinterpret_cast<uint32_t *>(&o0);
        o.y = *reinterpret_cast<uint32_t *>(&o1);
        *reinterpret_cast<uint2 *>(act + r * I + c) = o;
    }
}

// last token of every sequence -> the 32-row activation block the lm_head GEMM reads
__global__ void __launch_bounds__(256)
llm_gather_last_kernel(const __nv_bfloat16 *__restrict__ xn, const int32_t *__restrict__ cu_seqlens, __nv_bfloat16 *__restrict__ xlast, int H)
{
    const int b = blockIdx.x;
    const int64_t t = __ldg(cu_seqlens + b + 1) - 1;
    for (int i = threadIdx.x * 8; i < H; i += 256 * 8)
        *reinterpret_cast<uint4 *>(xlast + (int64_t)b * H + i) = *reinterpret_cast<const uint4 *>(xn + t * H + i);
}

// ------------------------------------------------------------------------------------------------
// greedy sampling over the vocabulary shard + cross-rank exchange.  B2S_LLM_AMAX_SPLIT (32) CTAs per sequence (grid = n_seq x SPLIT): with
// one CTA per sequence the 16 MB read-and-clear of the logits ran on 32 SMs (33 us per step; 30 -> 7 us of the step with 32 x 32 CTAs); the per-CTA maxima meet in a packed
// 64-bit atomicMax (ordered value bits high, ~index low: the smallest index wins a tie, as before) and the last CTA of a
// sequence finishes the row.
// logits fp32 [32, V_r] (skinny GEMM accumulator, cleared here; optionally copied to `keep` first).
// ------------------------------------------------------------------------------------------------
struct AmaxSlot { float val; int32_t idx; };
static int llm_amax_split()
{
    static const int v = []() { const char *e = getenv("B2S_LLM_AMAX_SPLIT"); const int x = e ? atoi(e) : 32; return x < 1 ? 1 : (x > 64 ? 64 : x); }();
    return v;
}

__global__ void __launch_bounds__(256)
llm_argmax_kernel(float *__restrict__ logits, float *__restrict__ keep, int V_r, int v_offset, AmaxSlot *my_slots, AmaxSlot *peer_slots,
                  uint32_t *my_flags, uint32_t *peer_flags, const uint32_t *gen, int k, int32_t *__restrict__ next_tok,
                  int32_t *__restrict__ out_tokens, const int32_t *__restrict__ out_pos, int max_new,
                  unsigned long long *__restrict__ row_key, int *__restrict__ row_cnt)
{
    __shared__ float s_val[256];
    __shared__ int s_idx[256];
    __shared__ int s_last;
    sm100::griddep_launch_dependents();
    sm100::griddep_wait();
    const int b = blockIdx.x, part = blockIdx.y, n_rows = gridDim.x;
    float *row = logits + (int64_t)b * V_r;
    const int n_split = gridDim.y;
    const int chunk = (V_r + n_split - 1) / n_split;
    const int c0 = part * chunk, c1 = min(V_r, c0 + chunk);
    float best = -INFINITY;
    int bi = 0x7fffffff;
    // eight independent loads per thread before the first use: as a load -> compare -> clear loop the compiler kept one L2 round
    // trip per element in flight (247 us for the 128 k columns of a row on one CTA)
    for (int i0 = c0 + threadIdx.x; i0 < c1; i0 += 256 * 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * 256;
            v[u] = i < c1 ? __ldcg(row + i) : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * 256;
            if (i < c1) {
                if (keep) keep[(int64_t)b * V_r + i] = v[u];
                row[i] = 0.f;
                // ascending i: first maximum per thread (a strip of -inf still names its first element)
                if (v[u] > best || (bi == 0x7fffffff && v[u] == best)) { best = v[u]; bi = i; }
            }
        }
    }
    s_val[threadIdx.x] = best;
    s_idx[threadIdx.x] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            const float v2 = s_val[threadIdx.x + o];
            const int i2 = s_idx[threadIdx.x + o];
            if (v2 > s_val[threadIdx.x] || (v2 == s_val[threadIdx.x] && i2 < s_idx[threadIdx.x])) {
                s_val[threadIdx.x] = v2;
                s_idx[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // (value, index) -> one orderable 64-bit key: larger value first, then smaller index
        const uint32_t fb = __float_as_uint(s_val[0]) == 0x80000000u ? 0u : __float_as_uint(s_val[0]);   // -0.0 ties +0.0
        const uint32_t ord = (fb & 0x80000000u) ? ~fb : (fb | 0x80000000u);
        const unsigned long long key = ((unsigned long long)ord << 32) | (unsigned long long)(0xffffffffu - (uint32_t)s_idx[0]);
        atomicMax(row_key + b, key);
        __threadfence();
        const int old = atomicAdd(row_cnt + b, 1);
        s_last = (old == n_split - 1);
        if (s_last) {
            row_cnt[b] = 0;
            const unsigned long long w = atomicExch(row_key + b, 0ull);    // read the row's winner and clear it for the next step
            const uint32_t o2 = (uint32_t)(w >> 32);
            const uint32_t f2 = (o2 & 0x80000000u) ? (o2 & 0x7fffffffu) : ~o2;
            s_val[0] = __uint_as_float(f2);
            s_idx[0] = (int)(0xffffffffu - (uint32_t)(w & 0xffffffffull));
        }
    }
    __syncthreads();
    if (!s_last) return;
    const uint32_t g = *reinterpret_cast<const volatile uint32_t *>(gen);
    const int par = (int)(g & 1u) * LLM_MAXB;
    float val = s_val[0];
    int idx = s_idx[0] + v_offset;
    if (peer_flags) {
        // every CTA publishes its own (val, idx) into the peer's slot table, then ONE flag per step is raised by
        // the last CTA to get there (grid-wide counter in my_flags[LLM_FLAGS - 1])
        if (threadIdx.x == 0) {
            AmaxSlot s;
            s.val = val;
            s.idx = idx;
            *reinterpret_cast<volatile float *>(&peer_slots[par + b].val) = s.val;
            *reinterpret_cast<volatile int32_t *>(&peer_slots[par + b].idx) = s.idx;
            __threadfence_system();
            const uint32_t done = atomicAdd(&my_flags[LLM_FLAGS - 1], 1u);
            if (done == (uint32_t)n_rows - 1) {
                my_flags[LLM_FLAGS - 1] = 0u;
                __threadfence_system();
                st_release_sys(peer_flags + k, g + 1u);
            }
            const long long t0 = clock64();
            while ((int32_t)(ld_acquire_sys(my_flags + k) - (g + 1u)) < 0) {
                if (clock64() - t0 > 20000000000ll) __trap();
                __nanosleep(64);
            }
            const float pv = *reinterpret_cast<volatile float *>(&my_slots[par + b].val);
            const int pi = *reinterpret_cast<volatile int32_t *>(&my_slots[par + b].idx);
            if (pv > val || (pv == val && pi < idx)) { val = pv; idx = pi; }
            s_idx[0] = idx;
        }
        __syncthreads();
        idx = s_idx[0];
    }
    if (threadIdx.x == 0) {
        next_tok[b] = idx;
        const int p = out_pos[b];
        if (p < max_new) out_tokens[(int64_t)b * max_new + p] = idx;
    }
}

// end of a step: the step counter advances; decode steps also advance context lengths / output positions
__global__ void llm_step_end_kernel(uint32_t *gen, int32_t *ctx_len, int32_t *out_pos, int n_seq, int is_decode, uint32_t *dstep)
{
    sm100::griddep_launch_dependents();
    sm100::griddep_wait();
    const int b = threadIdx.x;
    if (b < n_seq) {
        if (is_decode) ctx_len[b] += 1;
        out_pos[b] += 1;
    }
    if (b == 0) {
        *gen += 1u;
        if (is_decode && dstep) *dstep += 1u;     // decode steps completed: the pushed-partial counters of a TP pair advance with it
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct LlmLayer {
    __nv_bfloat16 *wqkv = nullptr, *wo = nullptr, *wgu = nullptr, *wdown = nullptr;
    float *ln1 = nullptr, *ln2 = nullptr;
    CUtensorMap m_qkv_w, m_o_w, m_gu_w, m_down_w;   // skinny-GEMM weight maps
    CUtensorMap m_kc, m_vc;                         // this layer's K / V page pool as [pages * kv_heads * 64, 128] (decode attention)
};

struct Llm {
    b2s_llm_config cfg{};
    int device = 0;
    int hq_r = 0, kvh_r = 0, qkv_n = 0, I_r = 0, V_r = 0, H = 0;
    int64_t max_tokens = 0;
    std::vector<LlmLayer> layers;
    __nv_bfloat16 *embed = nullptr, *lm_head = nullptr;
    float *final_norm = nullptr, *rope_cos = nullptr, *rope_sin = nullptr;
    __nv_bfloat16 *kcache = nullptr, *vcache = nullptr;
    int64_t kv_layer_stride = 0;
    int n_pages = 0, pages_per_seq = 0;     // paged KV: pool size, page-table row length (ceil(max_ctx / 64))
    int32_t *d_page_table = nullptr;        // [LLM_MAXB][pages_per_seq]
    std::vector<int32_t> h_page_table;
    // activations
    float *h = nullptr;
    __nv_bfloat16 *xn = nullptr, *qkv = nullptr, *attn = nullptr, *gu = nullptr, *act = nullptr, *xlast = nullptr;
    float *ws_qkv = nullptr, *ws_gu = nullptr, *ws_logits = nullptr, *keep_logits = nullptr;
    float *attn_part = nullptr;   // decode attention: (m, l, o) partials of split (sequence, kv head) segments, 2 slots per CTA
    int *attn_cnt = nullptr;      // arrivals per (sequence, kv head)
    int n_sm = 148;
    int attn_stream = 1;          // decode attention: 1 = key blocks dealt to the SMs (split sequences, merge order depends on the batch),
                                  // 0 = one CTA per (sequence, kv head): slower, bit-identical whatever else is in the batch
    // exchange block (one allocation, exported through cudaIpc)
    unsigned char *comm = nullptr, *peer_comm = nullptr;
    size_t comm_bytes = 0, off_amax = 0, off_pdec[2] = {0, 0}, off_ppre[2] = {0, 0};
    // step state
    int32_t *d_tokens = nullptr, *d_tok_seq = nullptr, *d_tok_pos = nullptr, *d_cu = nullptr, *d_slots = nullptr,
            *d_ctx_len = nullptr, *d_next_tok = nullptr, *d_out_tokens = nullptr, *d_out_pos = nullptr;
    uint32_t *d_gen = nullptr;
    unsigned long long *d_amax_key = nullptr;   // [LLM_MAXB] packed (value, index) maxima of the split argmax
    int *d_amax_cnt = nullptr;                  // [LLM_MAXB] arrivals
    uint32_t *d_dstep = nullptr;  // decode steps completed (device side)
    size_t off_mail[2] = {0, 0};  // exchange block: decode mailboxes, [32][H] fp32 each, slots hold 0xffffffff until the peer's partial lands
    size_t off_cnt = 0;           // exchange block: per exchange point, CTAs of the peer's projection that have pushed their partial
    int tp_push = 2;              // decode all-reduce (B2S_LLM_TP_PUSH): 2 = mailboxes, the value is its own arrival flag (default, 2.46 ms);
                                  // -1 = flag from the consumer kernel + peer read (2.57 ms per TP2 step); 0 = per-CTA arrival counts on the peer + peer read (2.78: 296 system-scope releases per projection
                                  // delay every CTA's exit); 1 = push, remote reductions + counts (3.21: NVLink atomics are no substitute for
                                  // one bulk read)
    uint32_t *d_idle = nullptr;   // [2] idle-HBM signals of the decode step (raised by reduce_rms / SwiGLU, polled by the next projection)
    int32_t *h_stage = nullptr;   // pinned staging for token metadata
    int max_new_cap = 0;
    int n_seq = 0;                // sequences of the current wave
    CUtensorMap m_x_xn, m_x_attn, m_x_act, m_x_last, m_lm_w;
    std::map<int, cudaGraphExec_t> decode_graphs;   // by n_seq
    std::map<int, int> decode_graph_launches;
    std::vector<void *> allocs;
    cudaStream_t stream = nullptr;        // every step of this model runs on its own stream
    cudaEvent_t events[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

    uint32_t *flags(unsigned char *base) const { return reinterpret_cast<uint32_t *>(base); }
    AmaxSlot *amax(unsigned char *base) const { return reinterpret_cast<AmaxSlot *>(base + off_amax); }
    uint32_t *pushed(unsigned char *base) const { return reinterpret_cast<uint32_t *>(base + off_cnt); }

    ~Llm()
    {
        cudaSetDevice(device);
        for (auto &g : decode_graphs) cudaGraphExecDestroy(g.second);
        if (peer_comm) cudaIpcCloseMemHandle(peer_comm);
        for (void *p : allocs) cudaFree(p);
        if (h_stage) cudaFreeHost(h_stage);
        for (cudaEvent_t e : events) if (e) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

template <typename T>
static int llm_alloc(Llm *m, T **out, size_t count, bool zero = true)
{
    void *p = nullptr;
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
    if (e != cudaSuccess) return fail_cuda(e, "cudaMalloc(llm)");
    m->allocs.push_back(p);
    if (zero) B2S_CUDA(cudaMemset(p, 0, bytes ? bytes : 16));
    *out = static_cast<T *>(p);
    return 0;
}

static int llm_create(int device, const b2s_llm_config *c, Llm **out)
{
    if (!c || !out) return fail(B2S_ERR_INVALID, "llm_create: null argument");
    if (c->head_dim != LLM_HD) return fail(B2S_ERR_INVALID, "llm: head_dim must be 128");
    if (c->tp_size != 1 && c->tp_size != 2) return fail(B2S_ERR_INVALID, "llm: tensor_parallel must be 1 or 2");
    if (c->tp_rank < 0 || c->tp_rank >= c->tp_size) return fail(B2S_ERR_INVALID, "llm: bad tp_rank");
    if (c->n_heads % c->tp_size || c->n_kv_heads % c->tp_size || c->inter % (64 * c->tp_size) || c->vocab % c->tp_size)
        return fail(B2S_ERR_INVALID, "llm: heads / kv heads / intermediate / vocab must divide by tensor_parallel");
    if (c->n_heads % c->n_kv_heads) return fail(B2S_ERR_INVALID, "llm: n_heads must be a multiple of n_kv_heads");
    if (c->hidden % 64 || c->hidden > 8192) return fail(B2S_ERR_INVALID, "llm: hidden must be a multiple of 64, <= 8192");
    if (c->max_batch < 1 || c->max_batch > LLM_MAXB) return fail(B2S_ERR_INVALID, "llm: max_batch must be 1..32");
    if (c->max_ctx < 16 || c->max_tokens < c->max_batch) return fail(B2S_ERR_INVALID, "llm: bad max_ctx / max_tokens");
    if (c->kv_pages < 0) return fail(B2S_ERR_INVALID, "llm: bad kv_pages");
    B2S_CUDA(cudaSetDevice(device));
    Llm *m = new Llm();
    m->cfg = *c;
    m->device = device;
    m->H = c->hidden;
    m->hq_r = c->n_heads / c->tp_size;
    m->kvh_r = c->n_kv_heads / c->tp_size;
    m->qkv_n = (m->hq_r + 2 * m->kvh_r) * LLM_HD;
    m->I_r = c->inter / c->tp_size;
    m->V_r = c->vocab / c->tp_size;
    m->max_tokens = c->max_tokens;
    m->max_new_cap = c->max_ctx;
    const int H = m->H, L = c->n_layers;
    const int64_t T = m->max_tokens;
    int rc = 0;
#define LA(ptr, count) if ((rc = llm_alloc(m, &(ptr), (size_t)(count))) != 0) { delete m; return rc; }
    LA(m->embed, (int64_t)c->vocab * H);
    LA(m->lm_head, (int64_t)m->V_r * H);
    LA(m->final_norm, H);
    LA(m->rope_cos, (int64_t)c->max_ctx * 64);
    LA(m->rope_sin, (int64_t)c->max_ctx * 64);
    m->layers.resize(L);
    for (int l = 0; l < L; ++l) {
        LlmLayer &y = m->layers[l];
        LA(y.wqkv, (int64_t)m->qkv_n * H);
        LA(y.wo, (int64_t)H * m->hq_r * LLM_HD);
        LA(y.wgu, (int64_t)2 * m->I_r * H);
        LA(y.wdown, (int64_t)H * m->I_r);
        LA(y.ln1, H);
        LA(y.ln2, H);
    }
    m->pages_per_seq = (c->max_ctx + 63) / 64;
    m->n_pages = c->kv_pages > 0 ? c->kv_pages : c->max_batch * m->pages_per_seq;
    m->kv_layer_stride = (int64_t)m->n_pages * m->kvh_r * 64 * LLM_HD;
    LA(m->kcache, m->kv_layer_stride * L);
    LA(m->vcache, m->kv_layer_stride * L);
    LA(m->d_page_table, (int64_t)LLM_MAXB * m->pages_per_seq);
    // default table: slot s owns pages [s * pages_per_seq, (s + 1) * pages_per_seq) while the pool is large enough (the
    // fixed-slot behaviour of b2s_llm_prefill); a host that manages pages itself overwrites rows with b2s_llm_set_pages
    m->h_page_table.assign((size_t)LLM_MAXB * m->pages_per_seq, 0);
    for (int sl = 0; sl < LLM_MAXB; ++sl)
        for (int pg = 0; pg < m->pages_per_seq; ++pg) {
            const int64_t id = (int64_t)sl * m->pages_per_seq + pg;
            m->h_page_table[(size_t)id] = id < m->n_pages ? (int32_t)id : 0;
        }
    if (cudaMemcpy(m->d_page_table, m->h_page_table.data(), m->h_page_table.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
        delete m;
        return fail(B2S_ERR_CUDA, "llm: page table upload failed");
    }
    const int64_t Tp = T > LLM_MAXB ? T : LLM_MAXB;
    LA(m->h, Tp * H);
    LA(m->xn, Tp * H);
    LA(m->qkv, Tp * m->qkv_n);
    LA(m->attn, Tp * m->hq_r * LLM_HD);
    LA(m->gu, (int64_t)128 << 20);   // 256 MiB of bf16: L2-flush scratch (the gate/up product itself never exists in memory)
    LA(m->act, Tp * m->I_r);
    LA(m->xlast, (int64_t)LLM_MAXB * H);
    LA(m->ws_qkv, (int64_t)LLM_MAXB * m->qkv_n);
    LA(m->ws_gu, (int64_t)LLM_MAXB * 2 * m->I_r);
    LA(m->ws_logits, (int64_t)LLM_MAXB * m->V_r);
    cudaDeviceGetAttribute(&m->n_sm, cudaDevAttrMultiProcessorCount, device);
    if (const char *e = getenv("B2S_LLM_ATTN_STREAM")) m->attn_stream = e[0] != '0';   // read per model, at creation
    LA(m->attn_part, (int64_t)m->n_sm * 2 * 2 * 8 * 132);   // up to 2 CTAs per SM, 2 slots each
    LA(m->attn_cnt, (int64_t)LLM_MAXB * m->kvh_r);
    // exchange block
    m->off_amax = LLM_FLAGS * 4;
    size_t off = m->off_amax + 2 * LLM_MAXB * sizeof(AmaxSlot);
    off = (size_t)round_up((int64_t)off, 256);
    for (int i = 0; i < 2; ++i) { m->off_pdec[i] = off; off += (size_t)LLM_MAXB * H * 4; }
    for (int i = 0; i < 2; ++i) { m->off_ppre[i] = off; off += (size_t)Tp * H * 2; }
    m->off_cnt = off;
    off += (size_t)LLM_FLAGS * 4;
    off = (size_t)round_up((int64_t)off, 256);
    for (int i = 0; i < 2; ++i) { m->off_mail[i] = off; off += (size_t)LLM_MAXB * H * 4; }
    m->comm_bytes = off;
    if (const char *e = getenv("B2S_LLM_TP_PUSH")) m->tp_push = atoi(e);
    LA(m->comm, off);
    for (int i = 0; i < 2; ++i) cudaMemset(m->comm + m->off_mail[i], 0xff, (size_t)LLM_MAXB * H * 4);
    LA(m->d_tokens, Tp);
    LA(m->d_tok_seq, Tp);
    LA(m->d_tok_pos, Tp);
    LA(m->d_cu, LLM_MAXB + 1);
    LA(m->d_slots, LLM_MAXB);
    LA(m->d_ctx_len, LLM_MAXB);
    LA(m->d_next_tok, LLM_MAXB);
    LA(m->d_out_pos, LLM_MAXB);
    LA(m->d_out_tokens, (int64_t)LLM_MAXB * m->max_new_cap);
    LA(m->d_gen, 4);
    LA(m->d_idle, 4);
    LA(m->d_dstep, 4);
    LA(m->d_amax_key, LLM_MAXB);
    LA(m->d_amax_cnt, LLM_MAXB);
#undef LA
    cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&m->h_stage), (size_t)(3 * Tp + 4 * LLM_MAXB + 8) * 4);
    if (e != cudaSuccess) { delete m; return fail_cuda(e, "cudaMallocHost(llm staging)"); }
    // RoPE table (fp32, as torch computes inv_freq / cos / sin in fp32)
    {
        std::vector<float> cs((size_t)c->max_ctx * 64), sn((size_t)c->max_ctx * 64);
        for (int i = 0; i < 64; ++i) {
            const float inv_freq = 1.0f / powf(c->rope_theta, (float)(2 * i) / (float)LLM_HD);
            for (int p = 0; p < c->max_ctx; ++p) {
                const float ang = (float)p * inv_freq;
                cs[(size_t)p * 64 + i] = (float)cos((double)ang);
                sn[(size_t)p * 64 + i] = (float)sin((double)ang);
            }
        }
        cudaMemcpy(m->rope_cos, cs.data(), cs.size() * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(m->rope_sin, sn.data(), sn.size() * 4, cudaMemcpyHostToDevice);
    }
    // norm weights default to 1 (nn.Module init); everything else zero until loaded / initialised
    llm_fill_const_kernel<<<8, 256>>>(m->final_norm, H, 1.0f);
    for (int l = 0; l < L; ++l) {
        llm_fill_const_kernel<<<8, 256>>>(m->layers[l].ln1, H, 1.0f);
        llm_fill_const_kernel<<<8, 256>>>(m->layers[l].ln2, H, 1.0f);
    }
    // tensor maps of the decode path (fixed buffers: graph-capturable)
    for (int l = 0; l < L && rc == 0; ++l) {
        LlmLayer &y = m->layers[l];
        rc = skinny_make_maps(&y.m_qkv_w, &m->m_x_xn, y.wqkv, m->qkv_n, H, m->xn, LLM_MAXB);
        if (!rc) rc = skinny_make_maps(&y.m_o_w, &m->m_x_attn, y.wo, H, m->hq_r * LLM_HD, m->attn, LLM_MAXB);
        if (!rc) rc = skinny_make_maps(&y.m_gu_w, &m->m_x_xn, y.wgu, 2 * m->I_r, H, m->xn, LLM_MAXB);
        if (!rc) rc = skinny_make_maps(&y.m_down_w, &m->m_x_act, y.wdown, H, m->I_r, m->act, LLM_MAXB);
        const int64_t kv_rows = (int64_t)m->n_pages * m->kvh_r * 64;
        if (!rc) rc = make_tmap_2d_kmajor(&y.m_kc, m->kcache + m->kv_layer_stride * l, kv_rows, LLM_HD, LLM_HD, 64, 1);
        if (!rc) rc = make_tmap_2d_kmajor(&y.m_vc, m->vcache + m->kv_layer_stride * l, kv_rows, LLM_HD, LLM_HD, 64, 1);
    }
    if (!rc) rc = skinny_make_maps(&m->m_lm_w, &m->m_x_last, m->lm_head, m->V_r, H, m->xlast, LLM_MAXB);
    if (rc) { delete m; return rc; }
    e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreate(&m->events[i]);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { delete m; return fail_cuda(e, "llm_create"); }
    *out = m;
    return 0;
}

static int llm_find_tensor(Llm *m, const char *name, int layer, void **ptr, int64_t *rows, int64_t *cols, int *elem)
{
    const std::string n(name ? name : "");
    const int H = m->H;
    *elem = 2;
    if (n == "embed") { *ptr = m->embed; *rows = m->cfg.vocab; *cols = H; return 0; }
    if (n == "lm_head") { *ptr = m->lm_head; *rows = m->V_r; *cols = H; return 0; }
    if (n == "final_norm") { *ptr = m->final_norm; *rows = 1; *cols = H; *elem = 4; return 0; }
    if (layer < 0 || layer >= m->cfg.n_layers) return fail(B2S_ERR_INVALID, "llm tensor '%s': layer %d out of range", name, layer);
    LlmLayer &y = m->layers[layer];
    if (n == "wqkv") { *ptr = y.wqkv; *rows = m->qkv_n; *cols = H; return 0; }
    if (n == "wo") { *ptr = y.wo; *rows = H; *cols = m->hq_r * LLM_HD; return 0; }
    if (n == "wgu") { *ptr = y.wgu; *rows = 2 * m->I_r; *cols = H; return 0; }
    if (n == "wdown") { *ptr = y.wdown; *rows = H; *cols = m->I_r; return 0; }
    if (n == "ln1") { *ptr = y.ln1; *rows = 1; *cols = H; *elem = 4; return 0; }
    if (n == "ln2") { *ptr = y.ln2; *rows = 1; *cols = H; *elem = 4; return 0; }
    return fail(B2S_ERR_INVALID, "llm: unknown tensor '%s'", name);
}

static void llm_fill(__nv_bfloat16 *w, int64_t rows, int64_t cols, uint64_t seed, uint32_t id, uint32_t row0, uint32_t col0, float std)
{
    llm_fill_kernel<<<1184, 256>>>(w, rows, cols, seed, id, row0, col0, std);
    count_launch();
}

// tensor ids of the deterministic initialiser: 0 embed, 1 lm_head, 16 + 8 * layer + {0 q, 1 k, 2 v, 3 o, 4 gate, 5 up, 6 down}
static int llm_init_random(Llm *m, uint64_t seed, float std)
{
    B2S_CUDA(cudaSetDevice(m->device));
    const int H = m->H, r = m->cfg.tp_rank;
    llm_fill(m->embed, m->cfg.vocab, H, seed, 0, 0, 0, std);
    llm_fill(m->lm_head, m->V_r, H, seed, 1, (uint32_t)(r * m->V_r), 0, std);
    for (int l = 0; l < m->cfg.n_layers; ++l) {
        LlmLayer &y = m->layers[l];
        const uint32_t id = 16 + 8 * (uint32_t)l;
        const int qr = m->hq_r * LLM_HD, kr = m->kvh_r * LLM_HD;
        llm_fill(y.wqkv, qr, H, seed, id + 0, (uint32_t)(r * qr), 0, std);
        llm_fill(y.wqkv + (int64_t)qr * H, kr, H, seed, id + 1, (uint32_t)(r * kr), 0, std);
        llm_fill(y.wqkv + (int64_t)(qr + kr) * H, kr, H, seed, id + 2, (uint32_t)(r * kr), 0, std);
        llm_fill(y.wo, H, qr, seed, id + 3, 0, (uint32_t)(r * qr), std);
        llm_fill_gate_up_kernel<<<1184, 256>>>(y.wgu, m->I_r, H, seed, id + 4, id + 5, (uint32_t)(r * m->I_r), std);
        count_launch();
        llm_fill(y.wdown, H, m->I_r, seed, id + 6, 0, (uint32_t)(r * m->I_r), std);
    }
    B2S_CUDA(cudaGetLastError());
    B2S_CUDA(cudaDeviceSynchronize());
    return 0;
}

static int llm_gemm_bf16(cudaStream_t st, const void *A, int64_t lda, const void *W, int M, int N, int K, void *C, bool swiglu = false)
{
    GemmEpilogue ep;
    ep.bias = nullptr;
    ep.residual = nullptr;
    ep.C = C;
    ep.ldc = swiglu ? N / 2 : N;
    ep.act = swiglu ? 4 : 0;   // ACT_SWIGLU: C is [M, N / 2]
    ep.out_f32 = 0;
    ep.is_bf16 = 1;
    ep.act_after = 0;
    return gemm_tn(st, A, lda, W, K, M, N, K, ep);
}

static int llm_prefill(Llm *m, cudaStream_t st, int n_seq, const int32_t *tokens, const int32_t *offsets, const int32_t *slots = nullptr)
{
    B2S_CUDA(cudaSetDevice(m->device));
    if (n_seq < 1 || n_seq > m->cfg.max_batch) return fail(B2S_ERR_INVALID, "llm prefill: n_seq %d outside 1..%d", n_seq, m->cfg.max_batch);
    const int64_t T = offsets[n_seq];
    if (offsets[0] != 0 || T < n_seq || T > m->max_tokens)
        return fail(B2S_ERR_INVALID, "llm prefill: %lld prompt tokens exceed max_tokens %lld", (long long)T, (long long)m->max_tokens);
    int max_len = 0;
    // stage token metadata: tokens | tok_seq | tok_pos | cu | slots | ctx_len | out_pos
    B2S_CUDA(cudaStreamSynchronize(st));   // staging buffer reuse
    int32_t *s_tok = m->h_stage, *s_seq = s_tok + T, *s_pos = s_seq + T, *s_cu = s_pos + T, *s_slots = s_cu + LLM_MAXB + 1,
            *s_ctx = s_slots + LLM_MAXB, *s_opos = s_ctx + LLM_MAXB;
    for (int b = 0; b < n_seq; ++b) {
        const int len = offsets[b + 1] - offsets[b];
        if (len < 1 || len >= m->cfg.max_ctx) return fail(B2S_ERR_INVALID, "llm prefill: prompt %d has %d tokens (1..%d)", b, len, m->cfg.max_ctx - 1);
        max_len = len > max_len ? len : max_len;
        for (int i = 0; i < len; ++i) {
            s_tok[offsets[b] + i] = tokens[offsets[b] + i];
            s_seq[offsets[b] + i] = b;
            s_pos[offsets[b] + i] = i;
        }
        s_cu[b] = offsets[b];
        s_slots[b] = slots ? slots[b] : b;
        if (s_slots[b] < 0 || s_slots[b] >= m->cfg.max_batch) return fail(B2S_ERR_INVALID, "llm prefill: KV slot %d outside 0..%d", s_slots[b], m->cfg.max_batch - 1);
        for (int a = 0; a < b; ++a)
            if (s_slots[a] == s_slots[b]) return fail(B2S_ERR_INVALID, "llm prefill: KV slot %d given twice", s_slots[b]);
        for (int pg = 0; pg <= (len - 1) / 64; ++pg) {   // every page the prompt touches must be a valid pool page
            const int32_t id = m->h_page_table[(size_t)s_slots[b] * m->pages_per_seq + pg];
            if (id < 0 || id >= m->n_pages) return fail(B2S_ERR_INVALID, "llm prefill: slot %d has no page for position %d", s_slots[b], pg * 64);
        }
        s_ctx[b] = len;
        s_opos[b] = 0;
    }
    s_cu[n_seq] = (int32_t)T;
    for (int b = n_seq; b < LLM_MAXB; ++b) { s_cu[b + 1] = (int32_t)T; s_slots[b] = 0; s_ctx[b] = 0; s_opos[b] = 0; }
    B2S_CUDA(cudaMemcpyAsync(m->d_tokens, s_tok, (size_t)T * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_tok_seq, s_seq, (size_t)T * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_tok_pos, s_pos, (size_t)T * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_cu, s_cu, (LLM_MAXB + 1) * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_slots, s_slots, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_ctx_len, s_ctx, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_out_pos, s_opos, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    m->n_seq = n_seq;

    const int H = m->H, L = m->cfg.n_layers, Ti = (int)T;
    const float scale = 1.0f / sqrtf((float)LLM_HD);
    uint32_t *myf = m->flags(m->comm), *peerf = m->peer_comm ? m->flags(m->peer_comm) : nullptr;
    llm_embed_rms_kernel<<<Ti, 256, 0, st>>>(m->d_tokens, m->embed, m->layers[0].ln1, m->h, m->xn, H, m->cfg.vocab, m->cfg.rms_eps);
    count_launch();
    int k = 0;
    for (int l = 0; l < L; ++l) {
        LlmLayer &y = m->layers[l];
        __nv_bfloat16 *kc = m->kcache + m->kv_layer_stride * l, *vc = m->vcache + m->kv_layer_stride * l;
        B2S_TRY(llm_gemm_bf16(st, m->xn, H, y.wqkv, Ti, m->qkv_n, H, m->qkv));
        llm_rope_cache_prefill_kernel<<<Ti, 256, 0, st>>>(m->qkv, kc, vc, m->d_tok_seq, m->d_tok_pos, m->d_slots, m->d_page_table,
                                                          m->pages_per_seq, m->rope_cos, m->rope_sin, m->hq_r, m->kvh_r, m->cfg.max_ctx);
        count_launch();
        B2S_TRY(llm_attn_prefill(st, m->qkv, m->qkv_n, kc, vc, m->d_cu, m->d_slots, m->d_page_table, m->pages_per_seq, m->attn,
                                 m->hq_r * LLM_HD, n_seq, max_len, m->hq_r, m->kvh_r, scale));
        for (int half = 0; half < 2; ++half, ++k) {
            void *mine = m->comm + m->off_ppre[k & 1];
            const void *peer = m->peer_comm ? m->peer_comm + m->off_ppre[k & 1] : nullptr;
            if (half == 0) {
                B2S_TRY(llm_gemm_bf16(st, m->attn, m->hq_r * LLM_HD, y.wo, Ti, H, m->hq_r * LLM_HD, mine));
            } else {
                B2S_TRY(llm_gemm_bf16(st, m->xn, H, y.wgu, Ti, 2 * m->I_r, H, m->act, true));   // SwiGLU in the epilogue
                B2S_TRY(llm_gemm_bf16(st, m->act, m->I_r, y.wdown, Ti, H, m->I_r, mine));
            }
            const float *w = half == 0 ? y.ln2 : (l + 1 < L ? m->layers[l + 1].ln1 : m->final_norm);
            llm_reduce_rms_kernel<false><<<Ti, 256, 0, st>>>(mine, peer, nullptr, myf, peerf, m->d_gen, k, w, m->h, m->xn, H, m->cfg.rms_eps, nullptr);
            count_launch();
        }
    }
    llm_gather_last_kernel<<<n_seq, 256, 0, st>>>(m->xn, m->d_cu, m->xlast, H);
    count_launch();
    B2S_TRY(skinny_gemm_maps(st, m->m_lm_w, m->m_x_last, m->ws_logits, m->V_r, H, n_seq));
    llm_argmax_kernel<<<dim3(n_seq, llm_amax_split()), 256, 0, st>>>(m->ws_logits, m->keep_logits, m->V_r, m->cfg.tp_rank * m->V_r, m->amax(m->comm),
                                             m->peer_comm ? m->amax(m->peer_comm) : nullptr, myf, peerf, m->d_gen, k, m->d_next_tok,
                                             m->d_out_tokens, m->d_out_pos, m->max_new_cap, m->d_amax_key, m->d_amax_cnt);
    llm_step_end_kernel<<<1, 32, 0, st>>>(m->d_gen, m->d_ctx_len, m->d_out_pos, n_seq, 0, m->d_dstep);
    count_launch(2);
    B2S_CUDA(cudaGetLastError());
    return 0;
}

// Launch as a programmatic dependent of the previous kernel in the stream: the grid may be scheduled before its
// predecessor has drained (every decode kernel begins with griddepcontrol.wait), which takes the launch latency
// of the ~9 small kernels per layer off the step's critical path.
template <typename... KArgs, typename... Args>
static cudaError_t launch_dependent(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    static const bool pdl = []() { const char *e = getenv("B2S_LLM_PDL"); return !(e && e[0] == '0'); }();
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// developer aid (b2s_llm_decode(..., use_graph = 2)): CUDA events between the kernels of eagerly launched steps
struct LlmTiming {
    std::vector<cudaEvent_t> ev;
    std::vector<int> label;
    size_t used = 0;
    void mark(cudaStream_t st, int what)
    {
        if (used == ev.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev.push_back(e);
            label.push_back(0);
        }
        label[used] = what;
        cudaEventRecord(ev[used++], st);
    }
};
static const char *const LLM_TIMING_NAMES[] = {"start", "embed_rms", "qkv_gemm", "rope_cache", "attention", "o_gemm", "reduce_rms(attn)",
                                               "gate_up_gemm", "swiglu", "down_gemm", "reduce_rms(mlp)", "lm_head_gemm", "argmax", "step_end"};

// one decode step for the current wave (enqueue only)
static int llm_decode_enqueue(Llm *m, cudaStream_t st, int *n_launch, LlmTiming *tm = nullptr)
{
#define LLM_MARK(id) do { if (tm) tm->mark(st, (id)); } while (0)
    LLM_MARK(0);
    const int H = m->H, L = m->cfg.n_layers, n_seq = m->n_seq;
    const float scale = 1.0f / sqrtf((float)LLM_HD);
    uint32_t *myf = m->flags(m->comm), *peerf = m->peer_comm ? m->flags(m->peer_comm) : nullptr;
    int nl = 0;
    // developer aid: B2S_LLM_SKIP bitmask drops kernels from the step (results are then meaningless) so that the
    // in-pipeline cost of each one can be read off the step time: 1 attention, 2 reduce_rms, 4 swiglu, 8 qkv,
    // 16 o, 32 gate/up, 64 down, 128 lm_head + argmax
    static const int skip = []() { const char *e = getenv("B2S_LLM_SKIP"); return e ? atoi(e) : 0; }();
    // The step's first kernel is a PLAIN launch: everything of this step starts after the previous step (or the prefill, or a
    // host update of slots / pages) has completed, so context lengths, slots and the page table are constant for every kernel
    // of the step -- the decode attention reads them, and streams cached K / V, before its programmatic dependency resolves.
    llm_embed_rms_kernel<<<n_seq, 256, 0, st>>>(m->d_next_tok, m->embed, m->layers[0].ln1, m->h, m->xn, H, m->cfg.vocab, m->cfg.rms_eps);
    B2S_CUDA(cudaGetLastError());
    ++nl;
    LLM_MARK(1);
    int k = 0;
    for (int l = 0; l < L; ++l) {
        LlmLayer &y = m->layers[l];
        __nv_bfloat16 *kc = m->kcache + m->kv_layer_stride * l, *vc = m->vcache + m->kv_layer_stride * l;
        // (idle-HBM signal of the kernel before each projection: reduce_rms k raises idle[0] to gen * 1024 + k + 1, SwiGLU of layer l idle[1] to + l + 1)
        if (!(skip & 8)) B2S_TRY(skinny_gemm_maps(st, y.m_qkv_w, m->m_x_xn, m->ws_qkv, m->qkv_n, H, n_seq, l > 0 ? m->d_idle : nullptr, m->d_gen, 2 * l));
        LLM_MARK(2);
        if (!(skip & 1)) B2S_TRY(llm_attn_decode(st, m->ws_qkv, kc, vc, m->d_ctx_len, m->d_slots, m->d_page_table, m->pages_per_seq, m->rope_cos,
                                m->rope_sin, m->attn, m->hq_r * LLM_HD, n_seq, m->hq_r, m->kvh_r, m->cfg.max_ctx, scale, &y.m_kc, &y.m_vc,
                                m->attn_part, m->attn_cnt, m->n_sm, m->attn_stream));
        LLM_MARK(4);
        nl += 2;
        for (int half = 0; half < 2; ++half, ++k) {
            float *mine = reinterpret_cast<float *>(m->comm + m->off_pdec[k & 1]);
            float *older = reinterpret_cast<float *>(m->comm + m->off_pdec[(k & 1) ^ 1]);
            const void *peer = m->peer_comm ? m->peer_comm + m->off_pdec[k & 1] : nullptr;
            // tensor-parallel pair, push form: this rank's projection also adds its partial into the PEER's buffer and counts
            // its CTAs there; the consumer below then reads (and clears) only local memory
            const bool push = m->peer_comm != nullptr && m->tp_push == 1, counted = m->peer_comm != nullptr && (m->tp_push == 0 || m->tp_push == 1);
            const bool mail = m->peer_comm != nullptr && m->tp_push == 2;
            float *push_to = push ? reinterpret_cast<float *>(m->peer_comm + m->off_pdec[k & 1]) : nullptr;
            uint32_t *push_cnt = counted ? m->pushed(m->peer_comm) + k : nullptr;
            int pushes = 0;
            if (half == 0) {
                if (!(skip & 16)) B2S_TRY(skinny_gemm_maps(st, y.m_o_w, m->m_x_attn, mine, H, m->hq_r * LLM_HD, n_seq, nullptr, nullptr, 0, push_to, push_cnt, &pushes));
                LLM_MARK(5);
                ++nl;
            } else {
                if (!(skip & 32)) B2S_TRY(skinny_gemm_maps(st, y.m_gu_w, m->m_x_xn, m->ws_gu, 2 * m->I_r, H, n_seq, m->d_idle, m->d_gen, 2 * l + 1));
                LLM_MARK(7);
                if (!(skip & 4)) B2S_CUDA(launch_dependent(llm_swiglu_decode_kernel, dim3((n_seq * (m->I_r / 4) + 255) / 256), dim3(256), st, m->ws_gu, m->act,
                                          (int64_t)n_seq, m->I_r, m->d_idle + 1, (const uint32_t *)m->d_gen, l + 1));
                LLM_MARK(8);
                if (!(skip & 64)) B2S_TRY(skinny_gemm_maps(st, y.m_down_w, m->m_x_act, mine, H, m->I_r, n_seq, m->d_idle + 1, m->d_gen, l + 1, push_to, push_cnt, &pushes));
                LLM_MARK(9);
                nl += 3;
            }
            const float *w = half == 0 ? y.ln2 : (l + 1 < L ? m->layers[l + 1].ln1 : m->final_norm);
            if (!(skip & 2)) B2S_CUDA(launch_dependent(llm_reduce_rms_kernel<true>, dim3(n_seq), dim3(256), st, (const void *)mine, peer, push ? mine : older,
                                      myf, peerf, (const uint32_t *)m->d_gen, k, w, m->h, m->xn, H, m->cfg.rms_eps, m->d_idle,
                                      counted ? (const uint32_t *)m->pushed(m->comm) : (const uint32_t *)nullptr, (const uint32_t *)m->d_dstep, pushes,
                                      push ? 1 : 0, mail ? reinterpret_cast<float *>(m->peer_comm + m->off_mail[k & 1]) : (float *)nullptr,
                                      mail ? reinterpret_cast<float *>(m->comm + m->off_mail[k & 1]) : (float *)nullptr));
            LLM_MARK(half == 0 ? 6 : 10);
            ++nl;
        }
    }
    // xn rows 0..n_seq-1 are the final-normed hidden states: lm_head reads them through the xn map
    if (!(skip & 128)) B2S_TRY(skinny_gemm_maps(st, m->m_lm_w, m->m_x_xn, m->ws_logits, m->V_r, H, n_seq, m->d_idle, m->d_gen, 2 * L));
    LLM_MARK(11);
    if (!(skip & 128)) B2S_CUDA(launch_dependent(llm_argmax_kernel, dim3(n_seq, llm_amax_split()), dim3(256), st, m->ws_logits, m->keep_logits, m->V_r, m->cfg.tp_rank * m->V_r,
                              m->amax(m->comm), m->peer_comm ? m->amax(m->peer_comm) : (AmaxSlot *)nullptr, myf, peerf,
                              (const uint32_t *)m->d_gen, k, m->d_next_tok, m->d_out_tokens, (const int32_t *)m->d_out_pos, m->max_new_cap,
                              m->d_amax_key, m->d_amax_cnt));
    LLM_MARK(12);
    B2S_CUDA(launch_dependent(llm_step_end_kernel, dim3(1), dim3(32), st, m->d_gen, m->d_ctx_len, m->d_out_pos, n_seq, 1, m->d_dstep));
    LLM_MARK(13);
    nl += 3;
    B2S_CUDA(cudaGetLastError());
    *n_launch = nl;
    return 0;
#undef LLM_MARK
}

static int llm_decode(Llm *m, cudaStream_t st, int n_steps, int use_graph)
{
    B2S_CUDA(cudaSetDevice(m->device));
    if (m->n_seq < 1) return fail(B2S_ERR_INVALID, "llm decode: no prefilled wave");
    if (n_steps < 0) return fail(B2S_ERR_INVALID, "llm decode: negative step count");
    if (use_graph == 2) {   // per-kernel device times of eagerly launched steps, printed to stderr
        double tot[14] = {0}, all = 0;
        int cnt[14] = {0};
        LlmTiming tm;
        for (int s = 0; s < n_steps; ++s) {
            int nl = 0;
            tm.used = 0;
            B2S_TRY(llm_decode_enqueue(m, st, &nl, &tm));
            count_launch((uint64_t)nl);
            B2S_CUDA(cudaStreamSynchronize(st));
            if (s == 0) continue;   // first step warms up
            for (size_t i = 1; i < tm.used; ++i) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, tm.ev[i - 1], tm.ev[i]);
                tot[tm.label[i]] += ms;
                cnt[tm.label[i]] += 1;
                all += ms;
            }
        }
        const int steps = n_steps > 1 ? n_steps - 1 : 1;
        fprintf(stderr, "llm decode timing (eager, %d steps, n_seq %d): %.3f ms/step\n", steps, m->n_seq, all / steps);
        for (int i = 1; i < 14; ++i)
            if (cnt[i]) fprintf(stderr, "  %-18s n/step=%4d avg=%8.2f us  per-step=%8.1f us (%4.1f%%)\n", LLM_TIMING_NAMES[i], cnt[i] / steps,
                                1e3 * tot[i] / cnt[i], 1e3 * tot[i] / steps, 100.0 * tot[i] / all);
        for (cudaEvent_t e : tm.ev) cudaEventDestroy(e);
        return 0;
    }
    if (!use_graph) {
        for (int s = 0; s < n_steps; ++s) {
            int nl = 0;
            B2S_TRY(llm_decode_enqueue(m, st, &nl));
            count_launch((uint64_t)nl);
        }
        return 0;
    }
    auto it = m->decode_graphs.find(m->n_seq);
    if (it == m->decode_graphs.end()) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        int nl = 0;
        B2S_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        const int rc = llm_decode_enqueue(m, st, &nl);
        cudaError_t e = cudaStreamEndCapture(st, &graph);
        if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) return fail_cuda(e, "cudaStreamEndCapture(llm decode)");
        e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return fail_cuda(e, "cudaGraphInstantiate(llm decode)");
        m->decode_graphs[m->n_seq] = exec;
        m->decode_graph_launches[m->n_seq] = nl;
        it = m->decode_graphs.find(m->n_seq);
    }
    const int nl = m->decode_graph_launches[m->n_seq];
    for (int s = 0; s < n_steps; ++s) {
        B2S_CUDA(cudaGraphLaunch(it->second, st));
        count_launch((uint64_t)nl);
    }
    return 0;
}

}  // namespace b2s

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
using b2s::Llm;

extern "C" {

B2S_API int b2s_llm_create(int device, const b2s_llm_config *cfg, b2s_llm **out)
{
    Llm *m = nullptr;
    const int rc = b2s::llm_create(device, cfg, &m);
    if (rc == 0) *out = reinterpret_cast<b2s_llm *>(m);
    return rc;
}

B2S_API int b2s_llm_free(b2s_llm *llm)
{
    delete reinterpret_cast<Llm *>(llm);
    return 0;
}

B2S_API int b2s_llm_init_random(b2s_llm *llm, uint64_t seed, float std)
{
    if (!llm) return b2s::fail(B2S_ERR_INVALID, "null llm");
    return b2s::llm_init_random(reinterpret_cast<Llm *>(llm), seed, std);
}

// device pointer + shape of one (per-rank) weight tensor; elem_bytes 2 = bf16, 4 = fp32
B2S_API int b2s_llm_tensor(b2s_llm *llm, const char *name, int layer, void **dptr, int64_t *rows, int64_t *cols, int *elem_bytes)
{
    if (!llm || !dptr || !rows || !cols || !elem_bytes) return b2s::fail(B2S_ERR_INVALID, "null argument");
    return b2s::llm_find_tensor(reinterpret_cast<Llm *>(llm), name, layer, dptr, rows, cols, elem_bytes);
}

B2S_API int b2s_llm_comm_export(b2s_llm *llm, unsigned char *handle64, uint64_t *bytes)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !handle64) return fail(B2S_ERR_INVALID, "null argument");
    B2S_CUDA(cudaSetDevice(m->device));
    cudaIpcMemHandle_t hnd;
    B2S_CUDA(cudaIpcGetMemHandle(&hnd, m->comm));
    static_assert(sizeof(hnd) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &hnd, 64);
    if (bytes) *bytes = m->comm_bytes;
    return 0;
}

B2S_API int b2s_llm_comm_attach(b2s_llm *llm, const unsigned char *peer_handle64)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !peer_handle64) return fail(B2S_ERR_INVALID, "null argument");
    if (m->cfg.tp_size != 2) return fail(B2S_ERR_INVALID, "llm: comm_attach needs tensor_parallel = 2");
    if (m->peer_comm) return fail(B2S_ERR_INVALID, "llm: peer already attached");
    B2S_CUDA(cudaSetDevice(m->device));
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, peer_handle64, 64);
    void *p = nullptr;
    B2S_CUDA(cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
    m->peer_comm = static_cast<unsigned char *>(p);
    return 0;
}

B2S_API int b2s_llm_prefill(b2s_llm *llm, int n_seq, const int32_t *tokens, const int32_t *offsets)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !tokens || !offsets) return fail(B2S_ERR_INVALID, "null argument");
    if (m->cfg.tp_size == 2 && !m->peer_comm) return fail(B2S_ERR_INVALID, "llm: tensor-parallel peer not attached");
    return llm_prefill(m, m->stream, n_seq, tokens, offsets);
}

B2S_API int b2s_llm_prefill_slots(b2s_llm *llm, int n_seq, const int32_t *tokens, const int32_t *offsets, const int32_t *slots)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !tokens || !offsets || !slots) return fail(B2S_ERR_INVALID, "null argument");
    if (m->cfg.tp_size == 2 && !m->peer_comm) return fail(B2S_ERR_INVALID, "llm: tensor-parallel peer not attached");
    return llm_prefill(m, m->stream, n_seq, tokens, offsets, slots);
}

B2S_API int b2s_llm_kv_info(b2s_llm *llm, int32_t *n_pages, int32_t *page_tokens, int32_t *pages_per_seq)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m) return fail(B2S_ERR_INVALID, "null argument");
    if (n_pages) *n_pages = m->n_pages;
    if (page_tokens) *page_tokens = 64;
    if (pages_per_seq) *pages_per_seq = m->pages_per_seq;
    return 0;
}

B2S_API int b2s_llm_set_pages(b2s_llm *llm, int slot, int first, int n, const int32_t *pages)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || (n > 0 && !pages)) return fail(B2S_ERR_INVALID, "null argument");
    if (slot < 0 || slot >= m->cfg.max_batch || first < 0 || n < 0 || first + n > m->pages_per_seq)
        return fail(B2S_ERR_INVALID, "llm set_pages: slot %d / logical pages [%d, %d) out of range", slot, first, first + n);
    for (int i = 0; i < n; ++i)
        if (pages[i] < 0 || pages[i] >= m->n_pages) return fail(B2S_ERR_INVALID, "llm set_pages: page %d outside the pool of %d", pages[i], m->n_pages);
    if (n == 0) return 0;
    B2S_CUDA(cudaSetDevice(m->device));
    int32_t *row = m->h_page_table.data() + (size_t)slot * m->pages_per_seq + first;
    memcpy(row, pages, (size_t)n * 4);
    // ordered on the model's stream behind the steps already enqueued (pageable source: staged before the call returns)
    B2S_CUDA(cudaMemcpyAsync(m->d_page_table + (size_t)slot * m->pages_per_seq + first, row, (size_t)n * 4, cudaMemcpyHostToDevice, m->stream));
    return 0;
}

B2S_API int b2s_llm_set_rows(b2s_llm *llm, int n_rows, const int32_t *slots, const int32_t *ctx_len, const int32_t *next_tok)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !slots || !ctx_len || !next_tok) return fail(B2S_ERR_INVALID, "null argument");
    if (n_rows < 1 || n_rows > m->cfg.max_batch) return fail(B2S_ERR_INVALID, "llm set_rows: %d rows outside 1..%d", n_rows, m->cfg.max_batch);
    int32_t h_slots[LLM_MAXB] = {0}, h_ctx[LLM_MAXB] = {0}, h_tok[LLM_MAXB] = {0}, h_pos[LLM_MAXB] = {0};
    for (int b = 0; b < n_rows; ++b) {
        if (slots[b] < 0 || slots[b] >= m->cfg.max_batch) return fail(B2S_ERR_INVALID, "llm set_rows: KV slot %d out of range", slots[b]);
        for (int a = 0; a < b; ++a)
            if (slots[a] == slots[b]) return fail(B2S_ERR_INVALID, "llm set_rows: KV slot %d given twice", slots[b]);
        if (ctx_len[b] < 1 || ctx_len[b] >= m->cfg.max_ctx) return fail(B2S_ERR_INVALID, "llm set_rows: context length %d outside 1..%d", ctx_len[b], m->cfg.max_ctx - 1);
        const int32_t id = m->h_page_table[(size_t)slots[b] * m->pages_per_seq + ctx_len[b] / 64];
        if (id < 0 || id >= m->n_pages) return fail(B2S_ERR_INVALID, "llm set_rows: slot %d has no page for position %d", slots[b], ctx_len[b]);
        h_slots[b] = slots[b];
        h_ctx[b] = ctx_len[b];
        h_tok[b] = next_tok[b];
    }
    B2S_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    B2S_CUDA(cudaMemcpyAsync(m->d_slots, h_slots, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_ctx_len, h_ctx, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_next_tok, h_tok, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    B2S_CUDA(cudaMemcpyAsync(m->d_out_pos, h_pos, LLM_MAXB * 4, cudaMemcpyHostToDevice, st));
    m->n_seq = n_rows;
    return 0;
}

B2S_API int b2s_llm_decode(b2s_llm *llm, int n_steps, int use_graph)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m) return fail(B2S_ERR_INVALID, "null argument");
    return llm_decode(m, m->stream, n_steps, use_graph);
}

// generated tokens of the current wave: out[n_seq][n] (first n per sequence); synchronises the stream
B2S_API int b2s_llm_get_tokens(b2s_llm *llm, int32_t *out, int n)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !out) return fail(B2S_ERR_INVALID, "null argument");
    if (n < 0 || n > m->max_new_cap) return fail(B2S_ERR_INVALID, "llm: at most %d generated tokens are kept", m->max_new_cap);
    B2S_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    B2S_CUDA(cudaMemcpy2DAsync(out, (size_t)n * 4, m->d_out_tokens, (size_t)m->max_new_cap * 4, (size_t)n * 4, (size_t)m->n_seq,
                               cudaMemcpyDeviceToHost, st));
    B2S_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// parity aid: keep a copy of the last step's logits shard ([n_seq][vocab / tp] fp32)
B2S_API int b2s_llm_keep_logits(b2s_llm *llm, int on)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m) return fail(B2S_ERR_INVALID, "null argument");
    B2S_CUDA(cudaSetDevice(m->device));
    if (on && !m->keep_logits) {
        B2S_TRY(llm_alloc(m, &m->keep_logits, (size_t)LLM_MAXB * m->V_r));
        for (auto &g : m->decode_graphs) cudaGraphExecDestroy(g.second);   // graphs baked the old pointer
        m->decode_graphs.clear();
    }
    return 0;
}

B2S_API int b2s_llm_get_logits(b2s_llm *llm, float *out)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !out) return fail(B2S_ERR_INVALID, "null argument");
    if (!m->keep_logits) return fail(B2S_ERR_INVALID, "llm: call b2s_llm_keep_logits(llm, 1) first");
    B2S_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    B2S_CUDA(cudaMemcpyAsync(out, m->keep_logits, (size_t)m->n_seq * m->V_r * 4, cudaMemcpyDeviceToHost, st));
    B2S_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// stream control: synchronise; record one of 8 CUDA events on the model's stream; device time between two of them
B2S_API int b2s_llm_synchronize(b2s_llm *llm)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m) return fail(B2S_ERR_INVALID, "null argument");
    B2S_CUDA(cudaSetDevice(m->device));
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    return 0;
}

B2S_API int b2s_llm_event_record(b2s_llm *llm, int which)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || which < 0 || which >= 8) return fail(B2S_ERR_INVALID, "llm event index must be 0..7");
    B2S_CUDA(cudaSetDevice(m->device));
    B2S_CUDA(cudaEventRecord(m->events[which], m->stream));
    return 0;
}

B2S_API int b2s_llm_elapsed_ms(b2s_llm *llm, int from, int to, float *ms)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m || !ms || from < 0 || from >= 8 || to < 0 || to >= 8) return fail(B2S_ERR_INVALID, "llm event index must be 0..7");
    B2S_CUDA(cudaSetDevice(m->device));
    B2S_CUDA(cudaEventSynchronize(m->events[to]));
    B2S_CUDA(cudaEventElapsedTime(ms, m->events[from], m->events[to]));
    return 0;
}

B2S_API int b2s_llm_flush_l2(b2s_llm *llm)
{
    using namespace b2s;
    Llm *m = reinterpret_cast<Llm *>(llm);
    if (!m) return fail(B2S_ERR_INVALID, "null argument");
    B2S_CUDA(cudaSetDevice(m->device));
    B2S_CUDA(cudaMemsetAsync(m->gu, 0, (size_t)256 << 20, m->stream));   // larger than the 126 MB L2
    return 0;
}

// ---- operator-level entry points of the LLM kernels (device pointers): each calls the launcher the model itself uses
B2S_API int b2s_op_llm_attn_decode(int device, void *cuda_stream, float *ws_qkv, void *k_pool, void *v_pool, int n_pages,
                                   const int32_t *ctx_len, const int32_t *slots, const int32_t *page_table, int pages_per_seq,
                                   const float *rope_cos, const float *rope_sin, int max_ctx, void *out, int n_seq, int n_heads,
                                   int n_kv_heads, int stream_form, int n_cta, float *part_ws, int *part_cnt)
{
    using namespace b2s;
    if (n_seq < 1 || n_seq > LLM_MAXB) return fail(B2S_ERR_INVALID, "llm decode attention: n_seq %d outside 1..%d", n_seq, LLM_MAXB);
    if (n_kv_heads < 1 || n_pages < 1) return fail(B2S_ERR_INVALID, "llm decode attention: bad pool shape");
    if (stream_form && (!part_ws || !part_cnt || n_cta < 1))
        return fail(B2S_ERR_INVALID, "llm decode attention: the stream form needs part_ws, part_cnt and n_cta >= 1");
    B2S_CUDA(cudaSetDevice(device));
    CUtensorMap tk, tv;
    if (stream_form) {
        const int64_t rows = (int64_t)n_pages * n_kv_heads * 64;
        B2S_TRY(make_tmap_2d_kmajor(&tk, k_pool, rows, LLM_HD, LLM_HD, 64, 1));
        B2S_TRY(make_tmap_2d_kmajor(&tv, v_pool, rows, LLM_HD, LLM_HD, 64, 1));
    }
    return llm_attn_decode(static_cast<cudaStream_t>(cuda_stream), ws_qkv, k_pool, v_pool, ctx_len, slots, page_table, pages_per_seq,
                           rope_cos, rope_sin, out, n_heads * LLM_HD, n_seq, n_heads, n_kv_heads, max_ctx, 1.0f / sqrtf((float)LLM_HD),
                           stream_form ? &tk : nullptr, stream_form ? &tv : nullptr, part_ws, part_cnt, n_cta, stream_form);
}

B2S_API int b2s_op_llm_attn_prefill(int device, void *cuda_stream, void *qkv, void *k_pool, void *v_pool, const int32_t *cu_seqlens,
                                    const int32_t *tok_seq, const int32_t *tok_pos, const int32_t *slots, const int32_t *page_table,
                                    int pages_per_seq, const float *rope_cos, const float *rope_sin, int max_ctx, void *out, int n_seq,
                                    int max_seqlen, int n_heads, int n_kv_heads)
{
    using namespace b2s;
    if (n_seq < 1 || max_seqlen < 1 || n_kv_heads < 1 || n_heads % n_kv_heads)
        return fail(B2S_ERR_INVALID, "llm prefill attention: bad shape");
    B2S_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    int32_t T = 0;   // one CTA per token for the RoPE + cache write: the token count is read back (this synchronises)
    B2S_CUDA(cudaMemcpyAsync(&T, cu_seqlens + n_seq, 4, cudaMemcpyDeviceToHost, st));
    B2S_CUDA(cudaStreamSynchronize(st));
    if (T < 1) return fail(B2S_ERR_INVALID, "llm prefill attention: no tokens");
    llm_rope_cache_prefill_kernel<<<T, 256, 0, st>>>(static_cast<__nv_bfloat16 *>(qkv), static_cast<__nv_bfloat16 *>(k_pool),
                                                     static_cast<__nv_bfloat16 *>(v_pool), tok_seq, tok_pos, slots, page_table,
                                                     pages_per_seq, rope_cos, rope_sin, n_heads, n_kv_heads, max_ctx);
    count_launch();
    B2S_CUDA(cudaGetLastError());
    return llm_attn_prefill(st, qkv, (n_heads + 2 * n_kv_heads) * LLM_HD, k_pool, v_pool, cu_seqlens, slots, page_table, pages_per_seq,
                            out, n_heads * LLM_HD, n_seq, max_seqlen, n_heads, n_kv_heads, 1.0f / sqrtf((float)LLM_HD));
}

B2S_API int b2s_op_llm_argmax(int device, void *cuda_stream, float *logits, float *keep, int n_seq, int vocab, int n_split,
                              unsigned long long *row_key, int *row_cnt, int32_t *tokens)
{
    using namespace b2s;
    if (n_seq < 1 || n_seq > 65535 || vocab < 1 || n_split < 1 || n_split > 65535)
        return fail(B2S_ERR_INVALID, "llm argmax: bad shape");
    B2S_CUDA(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    uint32_t *scratch = nullptr;   // [0]: step counter, [1, 1 + n_seq): output positions (all zero: no token buffer is written)
    B2S_CUDA(cudaMalloc(&scratch, (size_t)(n_seq + 1) * 4));
    cudaError_t e = cudaMemsetAsync(scratch, 0, (size_t)(n_seq + 1) * 4, st);
    if (e == cudaSuccess) {
        llm_argmax_kernel<<<dim3(n_seq, n_split), 256, 0, st>>>(logits, keep, vocab, 0, nullptr, nullptr, nullptr, nullptr, scratch, 0,
                                                               tokens, nullptr, reinterpret_cast<const int32_t *>(scratch + 1), 0,
                                                               row_key, row_cnt);
        count_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(scratch);
    B2S_CUDA(e);
    return 0;
}

}  // extern "C"
