// optim.cu -- Adam + AMP glue for the hash-grid table and the MLP weights in one pass (row f-4 of SURVEY.md section 8).
//
// What the reference's training step does around the kernels on the 12.2 M-parameter table, every step
// (nerf/utils.py:1474-1484 under `-O`: GradScaler + torch.optim.Adam; gridencoder/grid.py:43-44):
//     embeddings.half()                      49 MB read + 24.5 MB write
//     zeros_like(grad_embeddings)            24.5 MB write
//     fp16 grad -> fp32 .grad                24.5 MB read + 49 MB write
//     GradScaler inf check (+ unscale)       49 MB read (+ 49 MB write)
//     Adam                                   4 x 49 MB read + 3 x 49 MB write
// = ~610 MB of HBM traffic in 6+ launches.  Here: one non-finite check over the fp16 gradient the encoder backward
// accumulated (24.5 MB read, normally still in L2) and ONE update kernel that unscales, applies Adam (torch's fused
// CUDA Adam arithmetic, including its double-precision intermediate steps), writes the fp16 shadow copy the next
// forward gathers from, and clears the gradient: g16 R+W, p32 R+W, m R+W, v R+W, p16 W = 367 MB -- HBM-bound.
// Several tensors (table + both MLP weight vectors) are served by the same two launches.
#include <type_traits>

#include "common.cuh"

namespace lnrf {

constexpr int kMaxOptTensors = 8;
constexpr uint32_t kOptBlock = 256;
constexpr uint32_t kOptPerThread = 8;                      // elements per thread per chunk (one 16-byte fp16 vector)
constexpr uint32_t kOptChunk = kOptBlock * kOptPerThread;  // elements per block-iteration

struct OptTensor {
    float* p;          // fp32 master parameters
    float* m;          // exp_avg
    float* v;          // exp_avg_sq
    void* g;           // gradient (fp16 or fp32), cleared after use
    __half* p16;       // fp16 shadow copy (may be null)
    uint64_t n;
    uint32_t g_is_f16;
    uint32_t first_block;  // first block of the grid that works on this tensor
};
struct OptBatch {
    OptTensor t[kMaxOptTensors];
    uint32_t count;
};

__device__ __forceinline__ bool finite_h2(uint32_t w) {  // both halves of a packed half2 finite?
    return ((w & 0x7c00u) != 0x7c00u) && ((w & 0x7c000000u) != 0x7c000000u);
}

__device__ __forceinline__ int find_tensor(const OptBatch& b, uint32_t block) {
    int k = 0;
#pragma unroll
    for (int i = 1; i < kMaxOptTensors; i++)
        if (i < (int)b.count && block >= b.t[i].first_block) k = i;
    return k;
}

// does this block's share of the gradients hold an inf / nan?  (per thread; combine with __syncthreads_or)
__device__ __forceinline__ bool grad_block_nonfinite(const OptBatch& b) {
    const int k = find_tensor(b, blockIdx.x);
    const OptTensor& t = b.t[k];
    const uint32_t nblocks = (k + 1 < (int)b.count ? b.t[k + 1].first_block : gridDim.x) - t.first_block;
    bool bad = false;
    uint64_t base = (uint64_t)(blockIdx.x - t.first_block) * kOptChunk;
    if (t.g_is_f16) {
        // up to eight independent 16-byte loads per thread in flight (predicated): the 24.5 MB gradient is L2-resident (just written by
        // the encoder backward) and the table is ~5 chunks per block, so the whole check is ONE round trip per thread -- one load per
        // loop trip left the kernel latency-bound (10.6 us = 2.3 TB/s), four in flight + a remainder loop still took three trips
        const uint64_t stride = (uint64_t)nblocks * kOptChunk;
        const __half* g = reinterpret_cast<const __half*>(t.g);
        for (; base < t.n; base += 8 * stride) {
            uint4 w[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const uint64_t i = base + (uint64_t)u * stride + (uint64_t)threadIdx.x * kOptPerThread;
                w[u] = make_uint4(0u, 0u, 0u, 0u);
                if (i + kOptPerThread <= t.n) {
                    w[u] = *reinterpret_cast<const uint4*>(g + i);
                } else {
                    for (uint64_t j = i; j < t.n; j++) bad |= !isfinite(__half2float(g[j]));  // the ragged end of the tensor (< 8 elements)
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) bad |= !(finite_h2(w[u].x) && finite_h2(w[u].y) && finite_h2(w[u].z) && finite_h2(w[u].w));
        }
    }
    for (; base < t.n; base += (uint64_t)nblocks * kOptChunk) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kOptPerThread;
        if (i + kOptPerThread <= t.n) {
            if (t.g_is_f16) {
                const uint4 w = *reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(t.g) + i);
                bad |= !(finite_h2(w.x) && finite_h2(w.y) && finite_h2(w.z) && finite_h2(w.w));
            } else {
                const float4 a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i);
                const float4 c = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i + 4);
                bad |= !(isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w) && isfinite(c.x) && isfinite(c.y) &&
                         isfinite(c.z) && isfinite(c.w));
            }
        } else {
            for (uint64_t j = i; j < t.n; j++) {
                const float g = t.g_is_f16 ? __half2float(reinterpret_cast<const __half*>(t.g)[j]) : reinterpret_cast<const float*>(t.g)[j];
                bad |= !isfinite(g);
            }
        }
    }
    return bad;
}

// found_inf[0] = 1.0f when any gradient element is inf/nan (never cleared here: torch's GradScaler convention)
__global__ void __launch_bounds__(kOptBlock) k_grad_nonfinite(const OptBatch b, float* __restrict__ found_inf) {
    pdl_trigger();
    pdl_wait();  // nothing below may run before the kernels ahead on the stream are complete (common.cuh)
    const bool bad = grad_block_nonfinite(b);
    if (__syncthreads_or(bad) && threadIdx.x == 0) *found_inf = 1.0f;
}

// the same check; block 0 also freezes the scale and the step number of the running step (snapshot[1], snapshot[2]) for an optimizer
// kernel that updates the live words itself (lnrf_adam_step_sharded_pipelined)
__global__ void __launch_bounds__(kOptBlock)
k_grad_nonfinite_snap(const OptBatch b, float* __restrict__ flag_out, const float* __restrict__ grad_scale,
                      const float* __restrict__ step_count, float* __restrict__ snap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        snap[1] = grad_scale ? *grad_scale : 1.0f;
        snap[2] = *step_count;
    }
    const bool bad = grad_block_nonfinite(b);
    if (__syncthreads_or(bad) && threadIdx.x == 0) *flag_out = 1.0f;
}

struct AdamHyper {
    double lr, beta1, beta2, eps, weight_decay;
};

// torch/aten fused CUDA Adam (ADAM_MODE::ORIGINAL, amsgrad = false, maximize = false), statement by statement.  torch's kernel
// keeps its hyper-parameters in double, which promotes every statement to double and back: 8 float<->double conversions per
// element, all on the XU pipe (16 lanes/clk/SM) -- ncu showed this kernel at 58 % XU utilisation and 62 % issue, i.e. bound by
// the conversions rather than by HBM (profiles/r1k).  The same statements in fp32 with fused multiply-adds agree with torch's
// fused and foreach kernels to 2e-6 over several steps (tests/test_gpu_fused.py::test_adam_step_matches_torch_adam: the
// double intermediates only protect the last bit of each statement) and leave sqrt + two reciprocals on the XU pipe.
struct AdamStepConsts {
    float w1, w2, beta2;    // 1 - beta1, 1 - beta2 (formed in double on the way in), beta2
    float step_size;        // (float)(lr / bias_correction1)
    float inv_bc2_sqrt;     // 1 / sqrt(bias_correction2)
    float eps, weight_decay;
    double scale;           // GradScaler scale (1 when absent)
    float inv_scale;        // exact reciprocal when the scale is a power of two (the GradScaler default), else 0
    bool unscale;
};
__device__ __forceinline__ float adam_unscale(float g, const AdamStepConsts& c) {
    if (!c.unscale) return g;
    return c.inv_scale != 0.0f ? g * c.inv_scale : (float)((double)g / c.scale);  // both are torch's `grad /= scale`
}
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, const AdamHyper&, const AdamStepConsts& c) {
    if (c.weight_decay != 0.0f) g = fmaf(c.weight_decay, p, g);
    m = fmaf(c.w1, g - m, m);                          // lerp(exp_avg, grad, 1 - beta1)
    v = fmaf(c.w2 * g, g, c.beta2 * v);                // beta2 * v + (1 - beta2) * g * g
    // sqrt.approx / div.approx (one MUFU each, <= 2 ulp; sqrt.approx(0) = 0): the update is lr-sized, so 2.4e-7 relative on it is
    // far inside the 2e-6 agreement with torch asserted by the tests, and the IEEE fix-up paths were a tenth of the kernel's issue slots
    float sq;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
    const float denom = fmaf(sq, c.inv_bc2_sqrt, c.eps);
    p -= __fdividef(c.step_size * m, denom);
}

// STREAM: the fp32 master / moment vectors (147 MB each way, touched once per step) go through the cache with the streaming
// (evict-first) hint so that the 49 MB the NEXT step gathers from and reduces into -- the fp16 shadow this kernel writes and the
// gradient buffer it clears -- stay resident in the 126 MB L2.
// The per-step constants (two double pow() among them: ~400 double-precision instructions) are formed by ONE thread of the block
// and broadcast through shared memory -- every thread computing them cost as much as ten elements of its actual work.
__device__ __forceinline__ AdamStepConsts adam_step_consts(const AdamHyper& h, const float* grad_scale, const float* step_count) {
    __shared__ AdamStepConsts s_c;
    if (threadIdx.x == 0) {
        AdamStepConsts c;
        const double step = (double)*step_count;
        const float bc1 = (float)(1.0 - pow(h.beta1, step));
        c.w1 = (float)(1.0 - h.beta1);
        c.w2 = (float)(1.0 - h.beta2);
        c.beta2 = (float)h.beta2;
        c.eps = (float)h.eps;
        c.weight_decay = (float)h.weight_decay;
        c.step_size = (float)(h.lr / (double)bc1);
        c.inv_bc2_sqrt = (float)(1.0 / sqrt(1.0 - pow(h.beta2, step)));
        c.unscale = grad_scale != nullptr;
        const float scale_f = c.unscale ? *grad_scale : 1.0f;
        c.scale = (double)scale_f;
        int e2;
        c.inv_scale = (frexpf(scale_f, &e2) == 0.5f && e2 > -100 && e2 < 100) ? 1.0f / scale_f : 0.0f;
        s_c = c;
    }
    __syncthreads();
    return s_c;
}

template <bool STREAM>
__device__ __forceinline__ float4 ld_state(const float* p) {
    return STREAM ? __ldcs(reinterpret_cast<const float4*>(p)) : *reinterpret_cast<const float4*>(p);
}
template <bool STREAM>
__device__ __forceinline__ void st_state(float* p, float4 v) {
    if (STREAM) __stcs(reinterpret_cast<float4*>(p), v);
    else *reinterpret_cast<float4*>(p) = v;
}

template <bool STREAM>
__global__ void __launch_bounds__(kOptBlock)
k_adam_step(const OptBatch b, AdamHyper h, const float* __restrict__ grad_scale, const float* __restrict__ found_inf,
            const float* __restrict__ step_count, const float* __restrict__ lr_scale) {
    const int k = find_tensor(b, blockIdx.x);
    const OptTensor& t = b.t[k];
    const uint32_t nblocks = (k + 1 < (int)b.count ? b.t[k + 1].first_block : gridDim.x) - t.first_block;
    pdl_trigger();
    pdl_wait();  // nothing below may run before the kernels ahead on the stream are complete (common.cuh)
    const bool skip = found_inf != nullptr && *found_inf != 0.0f;  // GradScaler: the step is skipped, the gradient still cleared
    if (lr_scale) h.lr *= (double)*lr_scale;  // LambdaLR-style schedule factor kept on the device (CUDA-graph friendly)
    const AdamStepConsts c = adam_step_consts(h, grad_scale, step_count);

    for (uint64_t base = (uint64_t)(blockIdx.x - t.first_block) * kOptChunk; base < t.n; base += (uint64_t)nblocks * kOptChunk) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kOptPerThread;
        if (i >= t.n) continue;
        if (i + kOptPerThread > t.n) {  // ragged tail of the tensor: scalar path
            for (uint64_t j = i; j < t.n; j++) {
                float g;
                if (t.g_is_f16) {
                    g = __half2float(reinterpret_cast<const __half*>(t.g)[j]);
                    reinterpret_cast<__half*>(t.g)[j] = __float2half_rn(0.f);
                } else {
                    g = reinterpret_cast<const float*>(t.g)[j];
                    reinterpret_cast<float*>(t.g)[j] = 0.f;
                }
                if (skip) continue;
                float p = t.p[j], m = t.m[j], v = t.v[j];
                adam_update(p, m, v, adam_unscale(g, c), h, c);
                t.p[j] = p; t.m[j] = m; t.v[j] = v;
                if (t.p16) t.p16[j] = __float2half_rn(p);
            }
            continue;
        }
        // every load of this chunk is issued before the first store (the compiler cannot prove g / p / m / v do not alias, so
        // the order written here is the order executed): 7 x 16 B per thread in flight
        float g[kOptPerThread], p[kOptPerThread], m[kOptPerThread], v[kOptPerThread];
        uint4 gw = make_uint4(0u, 0u, 0u, 0u);
        if (t.g_is_f16) {
            gw = *reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(t.g) + i);
        } else {
            const float4* gp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i);
            *reinterpret_cast<float4*>(g) = __ldcs(gp);
            *reinterpret_cast<float4*>(g + 4) = __ldcs(gp + 1);
        }
        *reinterpret_cast<float4*>(p) = ld_state<STREAM>(t.p + i);
        *reinterpret_cast<float4*>(p + 4) = ld_state<STREAM>(t.p + i + 4);
        *reinterpret_cast<float4*>(m) = ld_state<STREAM>(t.m + i);
        *reinterpret_cast<float4*>(m + 4) = ld_state<STREAM>(t.m + i + 4);
        *reinterpret_cast<float4*>(v) = ld_state<STREAM>(t.v + i);
        *reinterpret_cast<float4*>(v + 4) = ld_state<STREAM>(t.v + i + 4);
        if (t.g_is_f16) {
            union { uint4 u; __half2 h2[4]; } w;
            w.u = gw;
#pragma unroll
            for (int j = 0; j < 4; j++) { const float2 f = __half22float2(w.h2[j]); g[2 * j] = f.x; g[2 * j + 1] = f.y; }
            *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(t.g) + i) = make_uint4(0u, 0u, 0u, 0u);
        } else {
            float* gp = reinterpret_cast<float*>(t.g) + i;
            *reinterpret_cast<float4*>(gp) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(gp + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (skip) continue;
#pragma unroll
        for (int j = 0; j < (int)kOptPerThread; j++)
            adam_update(p[j], m[j], v[j], adam_unscale(g[j], c), h, c);
        st_state<STREAM>(t.p + i, *reinterpret_cast<const float4*>(p));
        st_state<STREAM>(t.p + i + 4, *reinterpret_cast<const float4*>(p + 4));
        st_state<STREAM>(t.m + i, *reinterpret_cast<const float4*>(m));
        st_state<STREAM>(t.m + i + 4, *reinterpret_cast<const float4*>(m + 4));
        st_state<STREAM>(t.v + i, *reinterpret_cast<const float4*>(v));
        st_state<STREAM>(t.v + i + 4, *reinterpret_cast<const float4*>(v + 4));
        if (t.p16) {
            union { uint4 u; __half2 h2[4]; } w;
#pragma unroll
            for (int j = 0; j < 4; j++) w.h2[j] = __floats2half2_rn(p[2 * j], p[2 * j + 1]);
            *reinterpret_cast<uint4*>(t.p16 + i) = w.u;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// One launch for the whole optimizer step (round 2): non-finite check + Adam + GradScaler update
// ---------------------------------------------------------------------------------------------------------------------
// The three launches of the step above (k_grad_nonfinite, k_adam_step, k_amp_update) cost a 24.5 MB pass of their own for the
// check plus two launch gaps (10.6 + 3.7 us of kernels and the gaps between them in the 0.41 ms step).  Here every block first
// scans the gradient chunks it is about to update (phase 1), the blocks meet at a grid-wide barrier (the grid is capped at what is
// resident at once, so a spin barrier on a device counter cannot deadlock), read the combined flag, and run the update (phase 2) on
// the same chunks -- still in L2 from phase 1; the block that finishes last applies GradScaler.update() and re-arms the flag.
// `sync` = three zero-initialised device words owned by the optimizer: [0] arrivals, [1] barrier generation, [2] finished blocks.
struct AmpUpdateArgs {
    float* scale;
    int* growth_tracker;
    float* found_inf;
    float* step_count;
    float growth_factor, backoff_factor;
    int growth_interval;
};
__device__ __forceinline__ void amp_update_body(const AmpUpdateArgs& u, const float* found_now = nullptr) {
    if ((found_now ? *found_now : *u.found_inf) != 0.0f) {
        if (u.scale) *u.scale = *u.scale * u.backoff_factor;
        if (u.growth_tracker) *u.growth_tracker = 0;
    } else {
        if (u.scale && u.growth_tracker) {
            const int successful = *u.growth_tracker + 1;
            if (successful == u.growth_interval) {
                const float grown = *u.scale * u.growth_factor;
                if (isfinite(grown)) *u.scale = grown;
                *u.growth_tracker = 0;
            } else {
                *u.growth_tracker = successful;
            }
        }
        *u.step_count += 1.0f;
    }
    *u.found_inf = 0.0f;
}

// Non-finite check AND GradScaler.update() in one launch, ahead of Adam: the last block out (ticket) freezes what the optimizer
// kernel of THIS step must see -- snap[0] = found_inf, snap[1] = the scale the gradients carry, snap[2] = the step count before the
// increment -- and then updates scale / growth tracker / step count / found_inf for the next step.  lnrf_adam_step reads the
// snapshot instead of the live words, so the separate one-thread k_amp_update launch behind it disappears.  snap[4] is the ticket
// (zero before first use, re-armed here).
__global__ void __launch_bounds__(kOptBlock)
k_grad_nonfinite_amp(const OptBatch b, const AmpUpdateArgs u, float* __restrict__ snap) {
    pdl_trigger();
    pdl_wait();  // nothing below may run before the kernels ahead on the stream are complete (common.cuh)
    const bool bad = grad_block_nonfinite(b);
    if (__syncthreads_or(bad) && threadIdx.x == 0) *u.found_inf = 1.0f;
    if (threadIdx.x == 0) {
        unsigned int* ticket = reinterpret_cast<unsigned int*>(snap + 4);
        __threadfence();
        if (atomicAdd(ticket, 1u) == gridDim.x - 1u) {
            __threadfence();
            const float found = __ldcg(u.found_inf);
            snap[0] = found;
            snap[1] = u.scale ? *u.scale : 1.0f;
            snap[2] = *u.step_count;
            amp_update_body(u, &found);
            *ticket = 0u;
        }
    }
}

__global__ void __launch_bounds__(kOptBlock)
k_adam_amp_fused(const OptBatch b, AdamHyper h, const float* __restrict__ lr_scale, const AmpUpdateArgs u, unsigned int* __restrict__ sync) {
    const int k = find_tensor(b, blockIdx.x);
    const OptTensor& t = b.t[k];
    const uint32_t nblocks = (k + 1 < (int)b.count ? b.t[k + 1].first_block : gridDim.x) - t.first_block;
    __shared__ unsigned int s_gen;
    if (threadIdx.x == 0) s_gen = *reinterpret_cast<volatile unsigned int*>(sync + 1);
    if (lr_scale) h.lr *= (double)*lr_scale;
    const AdamStepConsts c = adam_step_consts(h, u.scale, u.step_count);   // reads scale / step_count before anybody may update them

    // ---- phase 1: non-finite check over this block's own chunks (fp16 gradients) ----
    bool bad = false;
    for (uint64_t base = (uint64_t)(blockIdx.x - t.first_block) * kOptChunk; base < t.n; base += (uint64_t)nblocks * kOptChunk) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kOptPerThread;
        if (i + kOptPerThread <= t.n) {
            if (t.g_is_f16) {
                const uint4 w = *reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(t.g) + i);
                bad |= !(finite_h2(w.x) && finite_h2(w.y) && finite_h2(w.z) && finite_h2(w.w));
            } else {
                const float4 a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i);
                const float4 d = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i + 4);
                bad |= !(isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w) && isfinite(d.x) && isfinite(d.y) &&
                         isfinite(d.z) && isfinite(d.w));
            }
        } else {
            for (uint64_t j = i; j < t.n; j++) {
                const float g = t.g_is_f16 ? __half2float(reinterpret_cast<const __half*>(t.g)[j]) : reinterpret_cast<const float*>(t.g)[j];
                bad |= !isfinite(g);
            }
        }
    }
    const bool block_bad = __syncthreads_or(bad) != 0;
    // ---- grid barrier ----
    if (threadIdx.x == 0) {
        if (block_bad) *reinterpret_cast<volatile float*>(u.found_inf) = 1.0f;
        __threadfence();
        const unsigned int arrived = atomicAdd(sync, 1u);
        if (arrived == gridDim.x - 1u) {
            sync[0] = 0u;
            __threadfence();
            atomicAdd(sync + 1, 1u);
        } else {
            const long long t0 = clock64();
            while (*reinterpret_cast<volatile unsigned int*>(sync + 1) == s_gen) {
                __nanosleep(32);
                if (clock64() - t0 > 8000000000ll) __trap();   // a barrier that cannot complete is a launch failure, not a hung GPU
            }
        }
        __threadfence();
    }
    __syncthreads();
    const bool skip = *reinterpret_cast<volatile float*>(u.found_inf) != 0.0f;

    // ---- phase 2: the update of k_adam_step on the same chunks ----
    for (uint64_t base = (uint64_t)(blockIdx.x - t.first_block) * kOptChunk; base < t.n; base += (uint64_t)nblocks * kOptChunk) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kOptPerThread;
        if (i >= t.n) continue;
        if (i + kOptPerThread > t.n) {  // ragged tail of the tensor: scalar path
            for (uint64_t j = i; j < t.n; j++) {
                float g;
                if (t.g_is_f16) {
                    g = __half2float(reinterpret_cast<const __half*>(t.g)[j]);
                    reinterpret_cast<__half*>(t.g)[j] = __float2half_rn(0.f);
                } else {
                    g = reinterpret_cast<const float*>(t.g)[j];
                    reinterpret_cast<float*>(t.g)[j] = 0.f;
                }
                if (skip) continue;
                float p = t.p[j], m = t.m[j], v = t.v[j];
                adam_update(p, m, v, adam_unscale(g, c), h, c);
                t.p[j] = p; t.m[j] = m; t.v[j] = v;
                if (t.p16) t.p16[j] = __float2half_rn(p);
            }
            continue;
        }
        float g[kOptPerThread], p[kOptPerThread], m[kOptPerThread], v[kOptPerThread];
        uint4 gw = make_uint4(0u, 0u, 0u, 0u);
        if (t.g_is_f16) {
            gw = *reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(t.g) + i);
        } else {
            const float4* gp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(t.g) + i);
            *reinterpret_cast<float4*>(g) = *gp;
            *reinterpret_cast<float4*>(g + 4) = *(gp + 1);
        }
        *reinterpret_cast<float4*>(p) = ld_state<true>(t.p + i);
        *reinterpret_cast<float4*>(p + 4) = ld_state<true>(t.p + i + 4);
        *reinterpret_cast<float4*>(m) = ld_state<true>(t.m + i);
        *reinterpret_cast<float4*>(m + 4) = ld_state<true>(t.m + i + 4);
        *reinterpret_cast<float4*>(v) = ld_state<true>(t.v + i);
        *reinterpret_cast<float4*>(v + 4) = ld_state<true>(t.v + i + 4);
        if (t.g_is_f16) {
            union { uint4 u; __half2 h2[4]; } w;
            w.u = gw;
#pragma unroll
            for (int j = 0; j < 4; j++) { const float2 f = __half22float2(w.h2[j]); g[2 * j] = f.x; g[2 * j + 1] = f.y; }
            *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(t.g) + i) = make_uint4(0u, 0u, 0u, 0u);
        } else {
            float* gp = reinterpret_cast<float*>(t.g) + i;
            *reinterpret_cast<float4*>(gp) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(gp + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (skip) continue;
#pragma unroll
        for (int j = 0; j < (int)kOptPerThread; j++) adam_update(p[j], m[j], v[j], adam_unscale(g[j], c), h, c);
        st_state<true>(t.p + i, *reinterpret_cast<const float4*>(p));
        st_state<true>(t.p + i + 4, *reinterpret_cast<const float4*>(p + 4));
        st_state<true>(t.m + i, *reinterpret_cast<const float4*>(m));
        st_state<true>(t.m + i + 4, *reinterpret_cast<const float4*>(m + 4));
        st_state<true>(t.v + i, *reinterpret_cast<const float4*>(v));
        st_state<true>(t.v + i + 4, *reinterpret_cast<const float4*>(v + 4));
        if (t.p16) {
            union { uint4 u; __half2 h2[4]; } w;
#pragma unroll
            for (int j = 0; j < 4; j++) w.h2[j] = __floats2half2_rn(p[2 * j], p[2 * j + 1]);
            *reinterpret_cast<uint4*>(t.p16 + i) = w.u;
        }
    }
    // ---- the block that finishes last applies GradScaler.update() (every block has consumed scale / step_count / found_inf) ----
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(sync + 2, 1u) == gridDim.x - 1u) {
            sync[2] = 0u;
            amp_update_body(u);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Ray-sharded training: gradient exchange + Adam + parameter broadcast as ONE kernel over NVLink peer memory
// ---------------------------------------------------------------------------------------------------------------------
// Every rank holds its full local fp16 gradient and the full fp16 shadow table in symmetric (peer-mapped) memory.  Rank r
// owns elements [lo, lo + n) of the flat parameter vector: for each of them it LOADS the gradient from all R ranks (its own
// and R-1 over NVLink), averages in fp32, applies Adam to its fp32 master slice and STORES the new fp16 value into all R
// shadow tables.  Per rank that moves (R-1)/R x 24.5 MB in and (R-1)/R x 24.5 MB out over NVLink -- the bytes of an
// all-reduce -- while the 367 MB HBM pass of Adam shrinks R-fold, and no intermediate buffer or collective launch exists.
// The skip-on-inf decision is global and identical everywhere: every rank checked its own gradient beforehand and
// published a flag next to it; the kernel reads all R flags.  (Averaging finite fp16 values in fp32 cannot overflow.)
// Synchronisation is the caller's: a cross-rank barrier before (gradients + flags complete) and after (shadows written,
// gradients may be cleared) the launch.
constexpr int kMaxPeers = 8;   // one NVSwitch domain of 8 GPUs; also bounds the registers that hold the in-flight peer loads
// G = gradient element type, P = element type of the replicated vector the kernel stores into: (__half, __half) for the NeRF's fp16
// gradients and fp16 shadow tables, (float, float) for the style network, whose fp32 parameter vector is both master and replica
template <typename G, typename P>
struct PeerPtrs {
    const G* grad[kMaxPeers];
    P* param[kMaxPeers];
    const float* flag[kMaxPeers];
};
// Per-segment learning rates of the flat vector (the style network trains its palette at 2 x lr): element e belongs to the last
// segment whose start <= e.  Starts are multiples of 8 elements, so one thread's 8-element vector never straddles two segments.
constexpr int kMaxLrSegments = 8;
struct LrSegments {
    uint64_t start[kMaxLrSegments];
    double mult[kMaxLrSegments];
    uint32_t count;
};
struct NoLrSegments {};
// the step size of every segment, formed as adam_step_consts forms it for lr x mult (shared memory of the block)
__device__ __forceinline__ float* segment_step_sizes(const AdamHyper& h, const LrSegments& segs, const float* step_count) {
    __shared__ float s_step_size[kMaxLrSegments];
    if (threadIdx.x < segs.count) {
        const float bc1 = (float)(1.0 - pow(h.beta1, (double)*step_count));
        s_step_size[threadIdx.x] = (float)(h.lr * segs.mult[threadIdx.x] / (double)bc1);
    }
    __syncthreads();
    return s_step_size;
}

// eight consecutive gradient elements of one rank, loaded as 16-byte vectors and added to g[0..7] in fp32
__device__ __forceinline__ uint4 ld_grad8(const __half* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void add_grad8(float* g, const uint4& u) {
    union { uint4 u; __half2 h2[4]; } w;
    w.u = u;
#pragma unroll
    for (int j = 0; j < 4; j++) { const float2 f = __half22float2(w.h2[j]); g[2 * j] += f.x; g[2 * j + 1] += f.y; }
}
struct Float8 { float4 a, b; };
__device__ __forceinline__ Float8 ld_grad8(const float* p) {
    return Float8{reinterpret_cast<const float4*>(p)[0], reinterpret_cast<const float4*>(p)[1]};
}
__device__ __forceinline__ void add_grad8(float* g, const Float8& u) {
    g[0] += u.a.x; g[1] += u.a.y; g[2] += u.a.z; g[3] += u.a.w;
    g[4] += u.b.x; g[5] += u.b.y; g[6] += u.b.z; g[7] += u.b.w;
}

// In-kernel rank synchronisation (ExchangeSync.epoch != nullptr).  The flag buffer of every rank is peer-mapped; words
// [kSyncArrive + r] and [kSyncDone + r] of MY buffer are written by rank r only.  Epoch e = *epoch + 1 of this step:
//   arrive: block 0 stores e into word kSyncArrive + me of every rank's buffer (system-scope release after a system fence: this
//           rank's gradient and non-finite flag are complete -- they were written by earlier kernels of the same stream), and every
//           block waits until its own words kSyncArrive + r hold >= e for all r before it touches a peer's gradient;
//   done:   after all blocks have stored their share of the new fp16 values into every rank's table (system fence per thread),
//           the block that finishes last stores e into word kSyncDone + me of every rank and publishes *epoch = e;
// k_exchange_finish (the next launch of the stream) waits for the R done-words before it clears the local gradient, and so
// orders the next forward pass behind every peer's stores.  Replaces two symmetric-memory barrier launches and a memset.
// Waits are bounded (__trap after ~4 s): a lost rank is a launch failure, not a hung GPU.
constexpr uint32_t kSyncArrive = 8, kSyncDone = 16;
struct ExchangeSync {
    uint32_t* epoch;    // local device word: last completed epoch
    uint32_t* ticket;   // local device word, zero between launches
    uint32_t me;
};
// Two gradient buffers alternate between consecutive steps (lnrf_adam_step_sharded_pipelined): while the ranks read THIS step's buffer,
// each rank clears the one the previous step used (its readers are long done: they passed this step's opening barrier), zeroes that
// step's non-finite flag word, and -- in one thread, at the very end -- performs GradScaler.update().  The separate closing launch
// (gradient clear + scale update behind barrier B) and the flag memset ahead of the inf check disappear.
struct ExchangeExtra {
    uint4* clear;       // local: the OTHER gradient buffer (null: nothing to clear)
    uint64_t clear_nvec;
    float* other_flag;  // local: the other step's non-finite flag word
    AmpUpdateArgs amp;  // amp.step_count == nullptr: no scale update here (grad_scale / step_count above must then be the snapshot)
};
__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void wait_words_ge(const uint32_t* words, uint32_t R, uint32_t e) {  // threads r < R poll word r; then barrier
    if (threadIdx.x < R) {
        const long long t0 = clock64();
        while ((int32_t)(ld_acquire_sys_u32(words + threadIdx.x) - e) < 0) {
            if (clock64() - t0 > 8000000000ll) __trap();
            __nanosleep(64);
        }
    }
    __syncthreads();
}

// fp32 form (G = P = float): `master` is this rank's slice of its own parameter vector, which the broadcast store rewrites like every
// other rank's; `segs` gives the learning rate of each part of the vector.
template <typename G, typename P, typename Segs>
__global__ void __launch_bounds__(kOptBlock)
k_adam_step_p2p(const PeerPtrs<G, P> peers, const uint32_t R, const uint64_t lo, const uint64_t n, float* __restrict__ master,
                float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, AdamHyper h, const float* __restrict__ grad_scale,
                float* __restrict__ found_inf_out, const float* __restrict__ step_count, const float* __restrict__ lr_scale,
                const ExchangeSync sync, const ExchangeExtra extra, const Segs segs) {
    constexpr bool kF32 = std::is_same<P, float>::value;
    static_assert(kF32 == std::is_same<Segs, LrSegments>::value, "segment table: fp32 form only");
    uint32_t epoch = 0;
    if (sync.epoch) {
        epoch = *sync.epoch + 1u;
        if (blockIdx.x == 0 && threadIdx.x < R) {
            __threadfence_system();
            st_release_sys_u32(reinterpret_cast<uint32_t*>(const_cast<float*>(peers.flag[threadIdx.x])) + kSyncArrive + sync.me, epoch);
        }
        wait_words_ge(reinterpret_cast<const uint32_t*>(peers.flag[sync.me]) + kSyncArrive, R, epoch);
    }
    // the R non-finite flags: thread r reads rank r's (ONE NVLink round trip per block, all in flight together -- a per-thread loop
    // over the ranks was R - 1 dependent remote reads in every warp: +7 us at N = 2, +116 us at N = 8)
    bool bad = false;
    if (threadIdx.x < R) bad = *reinterpret_cast<const volatile float*>(peers.flag[threadIdx.x]) != 0.0f;
    const bool skip = __syncthreads_or(bad) != 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) *found_inf_out = skip ? 1.0f : 0.0f;
    // GradScaler: when any rank saw a non-finite gradient nothing is updated (the gradients are cleared after the closing sync)
    if (lr_scale) h.lr *= (double)*lr_scale;
    AdamStepConsts c = adam_step_consts(h, grad_scale, step_count);
    const float inv_R = 1.0f / (float)R;
    float* s_step_size = nullptr;
    if constexpr (kF32) s_step_size = segment_step_sizes(h, segs, step_count);

    for (uint64_t base = (uint64_t)blockIdx.x * kOptChunk; base < n && !skip; base += (uint64_t)gridDim.x * kOptChunk) {
        const uint64_t i = base + (uint64_t)threadIdx.x * kOptPerThread;  // n is a multiple of 8: no ragged tail
        if (i >= n) continue;
        if constexpr (kF32) {
            uint32_t k = 0;
            for (uint32_t s = 1; s < segs.count; s++)
                if (lo + i >= segs.start[s]) k = s;
            c.step_size = s_step_size[k];
        }
        float g[kOptPerThread], p[kOptPerThread], m[kOptPerThread], v[kOptPerThread];
#pragma unroll
        for (int j = 0; j < (int)kOptPerThread; j++) g[j] = 0.0f;
        // all loads first: R gradient vectors (R-1 of them remote) + the local fp32 state
        std::conditional_t<kF32, Float8, uint4> gw[kMaxPeers];
#pragma unroll
        for (int r = 0; r < kMaxPeers; r++)
            if (r < (int)R) gw[r] = ld_grad8(peers.grad[r] + lo + i);
        *reinterpret_cast<float4*>(p) = *reinterpret_cast<const float4*>(master + i);
        *reinterpret_cast<float4*>(p + 4) = *reinterpret_cast<const float4*>(master + i + 4);
        *reinterpret_cast<float4*>(m) = *reinterpret_cast<const float4*>(exp_avg + i);
        *reinterpret_cast<float4*>(m + 4) = *reinterpret_cast<const float4*>(exp_avg + i + 4);
        *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(exp_avg_sq + i);
        *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(exp_avg_sq + i + 4);
#pragma unroll
        for (int r = 0; r < kMaxPeers; r++)   // fixed rank order 0 .. R-1: every rank forms the same sum
            if (r < (int)R) add_grad8(g, gw[r]);
#pragma unroll
        for (int j = 0; j < (int)kOptPerThread; j++) adam_update(p[j], m[j], v[j], adam_unscale(g[j] * inv_R, c), h, c);
        if constexpr (!kF32) {
            *reinterpret_cast<float4*>(master + i) = *reinterpret_cast<const float4*>(p);
            *reinterpret_cast<float4*>(master + i + 4) = *reinterpret_cast<const float4*>(p + 4);
        }
        *reinterpret_cast<float4*>(exp_avg + i) = *reinterpret_cast<const float4*>(m);
        *reinterpret_cast<float4*>(exp_avg + i + 4) = *reinterpret_cast<const float4*>(m + 4);
        *reinterpret_cast<float4*>(exp_avg_sq + i) = *reinterpret_cast<const float4*>(v);
        *reinterpret_cast<float4*>(exp_avg_sq + i + 4) = *reinterpret_cast<const float4*>(v + 4);
        if constexpr (kF32) {  // the broadcast IS the update: rank `me`'s own vector is one of the R
#pragma unroll
            for (int r = 0; r < kMaxPeers; r++) {
                if (r < (int)R) {
                    reinterpret_cast<float4*>(peers.param[r] + lo + i)[0] = *reinterpret_cast<const float4*>(p);
                    reinterpret_cast<float4*>(peers.param[r] + lo + i)[1] = *reinterpret_cast<const float4*>(p + 4);
                }
            }
        } else {
            union { uint4 u; __half2 h2[4]; } o;
#pragma unroll
            for (int j = 0; j < 4; j++) o.h2[j] = __floats2half2_rn(p[2 * j], p[2 * j + 1]);
#pragma unroll
            for (int r = 0; r < kMaxPeers; r++)
                if (r < (int)R) *reinterpret_cast<uint4*>(peers.param[r] + lo + i) = o.u;
        }
    }
    if (extra.clear) {
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < extra.clear_nvec; i += (uint64_t)gridDim.x * blockDim.x)
            extra.clear[i] = make_uint4(0u, 0u, 0u, 0u);
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            if (extra.other_flag) *extra.other_flag = 0.0f;
            if (extra.amp.step_count) {  // grad_scale / step_count of THIS kernel are the snapshot: every block may still be reading them
                const float found = skip ? 1.0f : 0.0f;
                amp_update_body(extra.amp, &found);
            }
        }
    }
    if (sync.epoch) {
        __shared__ bool s_last;
        __syncthreads();  // every store of the block happens-before thread 0's fence (fences are cumulative): ONE system fence per
        if (threadIdx.x == 0) {  // block, not one per thread (a per-thread membar.sys made the kernel 25 us slower than the barriers it replaces)
            __threadfence_system();
            s_last = atomicAdd(sync.ticket, 1u) == gridDim.x - 1u;
        }
        __syncthreads();
        if (s_last) {
            if (threadIdx.x < R) {
                __threadfence_system();
                st_release_sys_u32(reinterpret_cast<uint32_t*>(const_cast<float*>(peers.flag[threadIdx.x])) + kSyncDone + sync.me, epoch);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                *sync.ticket = 0u;
                *sync.epoch = epoch;
            }
        }
    }
}

// Closing half of the in-kernel synchronisation: wait until every rank has finished storing into MY table (done-words >= the epoch
// the exchange kernel just published), then clear the local gradient for the next step.
__global__ void __launch_bounds__(kOptBlock)
k_exchange_finish(const uint32_t* __restrict__ my_flag_words, const uint32_t R, const uint32_t* __restrict__ epoch,
                  uint4* __restrict__ grad, const uint64_t n_vec) {
    wait_words_ge(my_flag_words + kSyncDone, R, *epoch);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (uint64_t)gridDim.x * blockDim.x)
        grad[i] = make_uint4(0u, 0u, 0u, 0u);
}

// Closing launch of the barrier-bracketed sharded step: clear the local gradient (the peers have finished reading it: barrier B) and,
// in one thread, GradScaler.update() -- instead of a memset launch followed by k_amp_update.
__global__ void __launch_bounds__(kOptBlock)
k_clear_and_amp_update(uint4* __restrict__ grad, const uint64_t n_vec, const AmpUpdateArgs u) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (uint64_t)gridDim.x * blockDim.x)
        grad[i] = make_uint4(0u, 0u, 0u, 0u);
    if (blockIdx.x == 0 && threadIdx.x == 0) amp_update_body(u);
}

// GradScaler.update() (torch amp_update_scale_cuda_kernel) + the bookkeeping around it, one thread: adjust the scale,
// advance the step number when the step was not skipped, and re-arm found_inf for the next step.
__global__ void k_amp_update(float* scale, int* growth_tracker, float* found_inf, float* step_count, float growth_factor,
                             float backoff_factor, int growth_interval) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (*found_inf != 0.0f) {
        if (scale) *scale = *scale * backoff_factor;
        if (growth_tracker) *growth_tracker = 0;
    } else {
        if (scale && growth_tracker) {
            const int successful = *growth_tracker + 1;
            if (successful == growth_interval) {
                const float grown = *scale * growth_factor;
                if (isfinite(grown)) *scale = grown;
                *growth_tracker = 0;
            } else {
                *growth_tracker = successful;
            }
        }
        *step_count += 1.0f;
    }
    *found_inf = 0.0f;
}

static int make_batch(const char* who, const lnrf_opt_tensor* tensors, uint32_t count, OptBatch* b, uint32_t* grid, bool need_state,
                      uint32_t max_blocks = 0) {
    LNRF_REQUIRE(tensors && count >= 1 && count <= (uint32_t)kMaxOptTensors, "%s: 1..%d tensors per call, got %u", who, kMaxOptTensors, count);
    uint32_t blocks = 0;
    b->count = count;
    for (uint32_t i = 0; i < count; i++) {
        const lnrf_opt_tensor& s = tensors[i];
        LNRF_REQUIRE(s.grad && s.n > 0, "%s: tensor %u has no gradient / no elements", who, i);
        LNRF_REQUIRE(!need_state || (s.params && s.exp_avg && s.exp_avg_sq), "%s: tensor %u: null params / exp_avg / exp_avg_sq", who, i);
        LNRF_REQUIRE(s.grad_dtype == LNRF_F16 || s.grad_dtype == LNRF_F32, "%s: tensor %u: grad_dtype must be LNRF_F16 or LNRF_F32", who, i);
        LNRF_REQUIRE(((reinterpret_cast<uintptr_t>(s.grad) | reinterpret_cast<uintptr_t>(s.params) | reinterpret_cast<uintptr_t>(s.exp_avg) |
                       reinterpret_cast<uintptr_t>(s.exp_avg_sq) | reinterpret_cast<uintptr_t>(s.params_f16)) & 15) == 0,
                     "%s: tensor %u: buffers must be 16-byte aligned", who, i);
        OptTensor& t = b->t[i];
        t.p = s.params; t.m = s.exp_avg; t.v = s.exp_avg_sq; t.g = s.grad; t.p16 = (__half*)s.params_f16; t.n = s.n;
        t.g_is_f16 = s.grad_dtype == LNRF_F16;
        t.first_block = blocks;
        // enough blocks to fill the machine (8 resident blocks per SM), never more than the tensor has chunks
        const uint64_t chunks = (s.n + kOptChunk - 1) / kOptChunk;
        const char* ec = getenv("LNRF_ADAM_BLOCKS_PER_SM");  // A/B switch
        uint64_t cap = (uint64_t)kNumSMs * (uint64_t)(ec && atoi(ec) > 0 ? atoi(ec) : 8);
        if (max_blocks) {  // co-resident grids (k_adam_amp_fused): the tensors share max_blocks in proportion to their sizes
            uint64_t total = 0;
            for (uint32_t j = 0; j < count; j++) total += tensors[j].n;
            cap = 1ull + (uint64_t)(max_blocks > count ? max_blocks - count : 0u) * s.n / (total ? total : 1);   // sum of caps <= max_blocks
        }
        blocks += (uint32_t)(chunks < cap ? chunks : cap);
    }
    if (max_blocks && blocks > max_blocks) {
        set_error("%s: %u blocks needed but only %u can be resident at once", who, blocks, max_blocks);
        return LNRF_ERR_UNSUPPORTED;
    }
    *grid = blocks;
    return LNRF_OK;
}

}  // namespace lnrf

using namespace lnrf;

extern "C" {

int lnrf_grad_nonfinite_check(const lnrf_opt_tensor* tensors_host, uint32_t count, float* found_inf, lnrf_stream_t stream) {
    OptBatch b;
    uint32_t grid;
    if (int e = make_batch("grad_nonfinite_check", tensors_host, count, &b, &grid, false)) return e;
    LNRF_REQUIRE(found_inf, "grad_nonfinite_check: null found_inf");
    launch_pdl(k_grad_nonfinite, grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream), b, found_inf);
    LNRF_LAUNCH_CHECK("grad_nonfinite_check");
    return LNRF_OK;
}

int lnrf_adam_step(const lnrf_opt_tensor* tensors_host, uint32_t count, double lr, double beta1, double beta2, double eps,
                   double weight_decay, const float* grad_scale, const float* found_inf, const float* step_count,
                   const float* lr_scale, lnrf_stream_t stream) {
    OptBatch b;
    uint32_t grid;
    if (int e = make_batch("adam_step", tensors_host, count, &b, &grid, true)) return e;
    LNRF_REQUIRE(step_count, "adam_step: null step_count (device fp32 scalar holding the 1-based step number)");
    AdamHyper h{lr, beta1, beta2, eps, weight_decay};
    const char* es = getenv("LNRF_ADAM_STREAM");  // A/B switch (default on)
    if (!es || atoi(es) != 0)
        launch_pdl(k_adam_step<true>, grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream), b, h, grad_scale, found_inf, step_count, lr_scale);
    else
        launch_pdl(k_adam_step<false>, grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream), b, h, grad_scale, found_inf, step_count, lr_scale);
    LNRF_LAUNCH_CHECK("adam_step");
    return LNRF_OK;
}

int lnrf_adam_amp_step(const lnrf_opt_tensor* tensors_host, uint32_t count, double lr, double beta1, double beta2, double eps,
                       double weight_decay, float* grad_scale, int32_t* growth_tracker, float* found_inf, float* step_count,
                       const float* lr_scale, float growth_factor, float backoff_factor, int32_t growth_interval, uint32_t* sync_words,
                       lnrf_stream_t stream) {
    LNRF_REQUIRE(found_inf && step_count && sync_words, "adam_amp_step: null found_inf / step_count / sync_words");
    static std::atomic<int> s_per_sm{0};
    int per_sm = s_per_sm.load(std::memory_order_relaxed);
    if (per_sm == 0) {
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_adam_amp_fused, (int)kOptBlock, 0);
        if (e != cudaSuccess) return cuda_fail(e, "adam_amp_step");
        LNRF_REQUIRE(per_sm >= 1, "adam_amp_step: the kernel does not fit an SM");
        s_per_sm.store(per_sm, std::memory_order_relaxed);
    }
    if (const char* ec = getenv("LNRF_ADAM_BLOCKS_PER_SM")) {  // fewer resident blocks leave registers for a kernel on another stream
        const int want = atoi(ec);                               // (the look-ahead march of the next batch, nerf.py GraphedTrainStep)
        if (want > 0 && want < per_sm) per_sm = want;
    }
    int dev = 0, sms = kNumSMs;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    OptBatch b;
    uint32_t grid;
    // every block must be resident at once (grid-wide spin barrier): at most occupancy x SMs blocks, a count tensor-count larger
    // than the SM count keeps one block per small tensor
    if (int e = make_batch("adam_amp_step", tensors_host, count, &b, &grid, true, (uint32_t)(per_sm * sms))) return e;
    AdamHyper h{lr, beta1, beta2, eps, weight_decay};
    AmpUpdateArgs u{grad_scale, growth_tracker, found_inf, step_count, growth_factor, backoff_factor, growth_interval};
    k_adam_amp_fused<<<grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(b, h, lr_scale, u, sync_words);
    LNRF_LAUNCH_CHECK("adam_amp_step");
    return LNRF_OK;
}

int lnrf_grad_nonfinite_check_amp_update(const lnrf_opt_tensor* tensors_host, uint32_t count, float* grad_scale, int32_t* growth_tracker,
                                         float* found_inf, float* step_count, float growth_factor, float backoff_factor,
                                         int32_t growth_interval, float* snapshot, lnrf_stream_t stream) {
    LNRF_REQUIRE(found_inf && step_count && snapshot, "grad_nonfinite_check_amp_update: null found_inf / step_count / snapshot");
    OptBatch b;
    uint32_t grid;
    if (int e = make_batch("grad_nonfinite_check_amp_update", tensors_host, count, &b, &grid, false)) return e;
    AmpUpdateArgs u{grad_scale, growth_tracker, found_inf, step_count, growth_factor, backoff_factor, growth_interval};
    launch_pdl(k_grad_nonfinite_amp, grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream), b, u, snapshot);
    LNRF_LAUNCH_CHECK("grad_nonfinite_check_amp_update");
    return LNRF_OK;
}

int lnrf_amp_update(float* scale, int32_t* growth_tracker, float* found_inf, float* step_count, float growth_factor,
                    float backoff_factor, int32_t growth_interval, lnrf_stream_t stream) {
    LNRF_REQUIRE(found_inf && step_count, "amp_update: null found_inf / step_count");
    k_amp_update<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(scale, growth_tracker, found_inf, step_count, growth_factor,
                                                                       backoff_factor, growth_interval);
    LNRF_LAUNCH_CHECK("amp_update");
    return LNRF_OK;
}

static int adam_step_sharded_impl(const void* const* grad_peers_host, void* const* shadow_peers_host, const float* const* flag_peers_host,
                           uint32_t world, uint64_t lo, uint64_t n, float* master_shard, float* exp_avg_shard, float* exp_avg_sq_shard,
                           double lr, double beta1, double beta2, double eps, double weight_decay, const float* grad_scale,
                           float* found_inf_out, const float* step_count, const float* lr_scale, uint32_t rank, uint32_t* sync_epoch,
                           uint32_t* sync_ticket, lnrf_stream_t stream, const ExchangeExtra extra = ExchangeExtra{}) {
    LNRF_REQUIRE(world >= 1 && world <= (uint32_t)kMaxPeers, "adam_step_sharded: 1..%d ranks, got %u", kMaxPeers, world);
    LNRF_REQUIRE(grad_peers_host && shadow_peers_host && flag_peers_host && master_shard && exp_avg_shard && exp_avg_sq_shard &&
                     found_inf_out && step_count,
                 "adam_step_sharded: null pointer");
    LNRF_REQUIRE(n % 8 == 0 && lo % 8 == 0, "adam_step_sharded: slice offset / length must be multiples of 8 elements");
    if (n == 0) return LNRF_OK;
    PeerPtrs<__half, __half> pp{};
    for (uint32_t r = 0; r < world; r++) {
        LNRF_REQUIRE(grad_peers_host[r] && shadow_peers_host[r] && flag_peers_host[r], "adam_step_sharded: null peer pointer (rank %u)", r);
        pp.grad[r] = (const __half*)grad_peers_host[r];
        pp.param[r] = (__half*)shadow_peers_host[r];
        pp.flag[r] = flag_peers_host[r];
    }
    AdamHyper h{lr, beta1, beta2, eps, weight_decay};
    const uint64_t chunks = (n + kOptChunk - 1) / kOptChunk, cap = (uint64_t)kNumSMs * 8;
    ExchangeSync sy{sync_epoch, sync_ticket, rank};
    k_adam_step_p2p<__half, __half, NoLrSegments><<<(uint32_t)(chunks < cap ? chunks : cap), kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        pp, world, lo, n, master_shard, exp_avg_shard, exp_avg_sq_shard, h, grad_scale, found_inf_out, step_count, lr_scale, sy, extra,
        NoLrSegments{});
    LNRF_LAUNCH_CHECK("adam_step_sharded");
    return LNRF_OK;
}

int lnrf_adam_step_sharded(const void* const* grad_peers_host, void* const* shadow_peers_host, const float* const* flag_peers_host,
                           uint32_t world, uint64_t lo, uint64_t n, float* master_shard, float* exp_avg_shard, float* exp_avg_sq_shard,
                           double lr, double beta1, double beta2, double eps, double weight_decay, const float* grad_scale,
                           float* found_inf_out, const float* step_count, const float* lr_scale, lnrf_stream_t stream) {
    return adam_step_sharded_impl(grad_peers_host, shadow_peers_host, flag_peers_host, world, lo, n, master_shard, exp_avg_shard,
                                  exp_avg_sq_shard, lr, beta1, beta2, eps, weight_decay, grad_scale, found_inf_out, step_count, lr_scale, 0u,
                                  nullptr, nullptr, stream);
}

int lnrf_adam_step_sharded_sync(const void* const* grad_peers_host, void* const* shadow_peers_host, const float* const* flag_peers_host,
                                uint32_t world, uint32_t rank, uint64_t lo, uint64_t n, float* master_shard, float* exp_avg_shard,
                                float* exp_avg_sq_shard, double lr, double beta1, double beta2, double eps, double weight_decay,
                                const float* grad_scale, float* found_inf_out, const float* step_count, const float* lr_scale,
                                uint32_t* sync_state, lnrf_stream_t stream) {
    LNRF_REQUIRE(sync_state && rank < world, "adam_step_sharded_sync: null sync state / rank %u outside the world of %u", rank, world);
    return adam_step_sharded_impl(grad_peers_host, shadow_peers_host, flag_peers_host, world, lo, n, master_shard, exp_avg_shard,
                                  exp_avg_sq_shard, lr, beta1, beta2, eps, weight_decay, grad_scale, found_inf_out, step_count, lr_scale, rank,
                                  sync_state, sync_state + 1, stream);
}

int lnrf_adam_step_sharded_f32(const float* const* grad_peers_host, float* const* param_peers_host, const float* const* flag_peers_host,
                               uint32_t world, uint32_t rank, uint64_t lo, uint64_t n, const uint64_t* seg_start_host,
                               const double* seg_lr_mult_host, uint32_t n_segs, float* exp_avg_shard, float* exp_avg_sq_shard, double lr,
                               double beta1, double beta2, double eps, double weight_decay, const float* grad_scale, float* found_inf_out,
                               const float* step_count, const float* lr_scale, lnrf_stream_t stream) {
    LNRF_REQUIRE(world >= 1 && world <= (uint32_t)kMaxPeers, "adam_step_sharded_f32: 1..%d ranks, got %u", kMaxPeers, world);
    LNRF_REQUIRE(rank < world, "adam_step_sharded_f32: rank %u outside the world of %u", rank, world);
    LNRF_REQUIRE(grad_peers_host && param_peers_host && flag_peers_host && seg_start_host && seg_lr_mult_host && exp_avg_shard &&
                     exp_avg_sq_shard && found_inf_out && step_count,
                 "adam_step_sharded_f32: null pointer");
    LNRF_REQUIRE(n % 8 == 0 && lo % 8 == 0, "adam_step_sharded_f32: slice offset / length must be multiples of 8 elements");
    LNRF_REQUIRE(n_segs >= 1 && n_segs <= (uint32_t)kMaxLrSegments, "adam_step_sharded_f32: 1..%d lr segments, got %u", kMaxLrSegments, n_segs);
    LrSegments segs{};
    segs.count = n_segs;
    for (uint32_t s = 0; s < n_segs; s++) {
        LNRF_REQUIRE(s == 0 ? seg_start_host[0] == 0 : seg_start_host[s] > seg_start_host[s - 1],
                     "adam_step_sharded_f32: segment starts must begin at 0 and ascend strictly (segment %u)", s);
        LNRF_REQUIRE(seg_start_host[s] % 8 == 0, "adam_step_sharded_f32: segment %u starts off a multiple of 8 elements", s);
        LNRF_REQUIRE(seg_lr_mult_host[s] >= 0.0 && seg_lr_mult_host[s] < 1e30, "adam_step_sharded_f32: segment %u: bad lr multiplier", s);
        segs.start[s] = seg_start_host[s];
        segs.mult[s] = seg_lr_mult_host[s];
    }
    PeerPtrs<float, float> pp{};
    uintptr_t align = reinterpret_cast<uintptr_t>(exp_avg_shard) | reinterpret_cast<uintptr_t>(exp_avg_sq_shard);
    for (uint32_t r = 0; r < world; r++) {
        LNRF_REQUIRE(grad_peers_host[r] && param_peers_host[r] && flag_peers_host[r], "adam_step_sharded_f32: null peer pointer (rank %u)", r);
        pp.grad[r] = grad_peers_host[r];
        pp.param[r] = param_peers_host[r];
        pp.flag[r] = flag_peers_host[r];
        align |= reinterpret_cast<uintptr_t>(grad_peers_host[r]) | reinterpret_cast<uintptr_t>(param_peers_host[r]);
    }
    LNRF_REQUIRE((align & 15) == 0, "adam_step_sharded_f32: buffers must be 16-byte aligned");
    if (n == 0) return LNRF_OK;
    AdamHyper h{lr, beta1, beta2, eps, weight_decay};
    const uint64_t chunks = (n + kOptChunk - 1) / kOptChunk, cap = (uint64_t)kNumSMs * 8;
    k_adam_step_p2p<float, float, LrSegments><<<(uint32_t)(chunks < cap ? chunks : cap), kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        pp, world, lo, n, param_peers_host[rank] + lo, exp_avg_shard, exp_avg_sq_shard, h, grad_scale, found_inf_out, step_count, lr_scale,
        ExchangeSync{nullptr, nullptr, rank}, ExchangeExtra{}, segs);
    LNRF_LAUNCH_CHECK("adam_step_sharded_f32");
    return LNRF_OK;
}

int lnrf_adam_step_sharded_pipelined(const void* const* grad_peers_host, void* const* shadow_peers_host, const float* const* flag_peers_host,
                                     uint32_t world, uint64_t lo, uint64_t n, float* master_shard, float* exp_avg_shard,
                                     float* exp_avg_sq_shard, double lr, double beta1, double beta2, double eps, double weight_decay,
                                     const float* snapshot, const float* lr_scale, void* other_grad_f16, uint64_t other_n,
                                     float* other_flag, float* grad_scale, int32_t* growth_tracker, float* found_inf, float* step_count,
                                     float growth_factor, float backoff_factor, int32_t growth_interval, lnrf_stream_t stream) {
    LNRF_REQUIRE(snapshot && other_grad_f16 && other_flag && found_inf && step_count, "adam_step_sharded_pipelined: null pointer");
    LNRF_REQUIRE(other_n % 8 == 0 && (reinterpret_cast<uintptr_t>(other_grad_f16) & 15) == 0,
                 "adam_step_sharded_pipelined: the gradient buffers must be 16-byte vectors");
    ExchangeExtra ex{reinterpret_cast<uint4*>(other_grad_f16), other_n / 8, other_flag,
                     AmpUpdateArgs{grad_scale, growth_tracker, found_inf, step_count, growth_factor, backoff_factor, growth_interval}};
    // scale and step of THIS step come from the snapshot the inf check took (snapshot[1], snapshot[2]): the live words change under the kernel
    return adam_step_sharded_impl(grad_peers_host, shadow_peers_host, flag_peers_host, world, lo, n, master_shard, exp_avg_shard,
                                  exp_avg_sq_shard, lr, beta1, beta2, eps, weight_decay, grad_scale ? snapshot + 1 : nullptr, found_inf,
                                  snapshot + 2, lr_scale, 0u, nullptr, nullptr, stream, ex);
}

int lnrf_grad_nonfinite_check_snapshot(const lnrf_opt_tensor* tensors_host, uint32_t count, float* flag_out, const float* grad_scale,
                                       const float* step_count, float* snapshot, lnrf_stream_t stream) {
    LNRF_REQUIRE(flag_out && step_count && snapshot, "grad_nonfinite_check_snapshot: null pointer");
    OptBatch b;
    uint32_t grid;
    if (int e = make_batch("grad_nonfinite_check_snapshot", tensors_host, count, &b, &grid, false)) return e;
    k_grad_nonfinite_snap<<<grid, kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(b, flag_out, grad_scale, step_count, snapshot);
    LNRF_LAUNCH_CHECK("grad_nonfinite_check_snapshot");
    return LNRF_OK;
}

int lnrf_exchange_tail(void* grad_f16, uint64_t n, float* scale, int32_t* growth_tracker, float* found_inf, float* step_count,
                       float growth_factor, float backoff_factor, int32_t growth_interval, lnrf_stream_t stream) {
    LNRF_REQUIRE(grad_f16 && found_inf && step_count, "exchange_tail: null pointer");
    LNRF_REQUIRE(n % 8 == 0 && (reinterpret_cast<uintptr_t>(grad_f16) & 15) == 0, "exchange_tail: the gradient must be 16-byte vectors");
    const uint64_t n_vec = n / 8;
    const uint64_t want = (n_vec + kOptBlock - 1) / kOptBlock, cap = (uint64_t)kNumSMs * 8;
    AmpUpdateArgs u{scale, growth_tracker, found_inf, step_count, growth_factor, backoff_factor, growth_interval};
    k_clear_and_amp_update<<<(uint32_t)(want < cap ? (want ? want : 1) : cap), kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<uint4*>(grad_f16), n_vec, u);
    LNRF_LAUNCH_CHECK("exchange_tail");
    return LNRF_OK;
}

int lnrf_exchange_finish(const float* my_flags, uint32_t world, const uint32_t* sync_state, void* grad_f16, uint64_t n,
                         lnrf_stream_t stream) {
    LNRF_REQUIRE(my_flags && sync_state && grad_f16 && world >= 1 && world <= (uint32_t)kMaxPeers, "exchange_finish: bad arguments");
    LNRF_REQUIRE(n % 8 == 0 && (reinterpret_cast<uintptr_t>(grad_f16) & 15) == 0, "exchange_finish: the gradient must be 16-byte vectors");
    const uint64_t n_vec = n / 8;
    const uint64_t want = (n_vec + kOptBlock - 1) / kOptBlock, cap = (uint64_t)kNumSMs * 8;
    k_exchange_finish<<<(uint32_t)(want < cap ? (want ? want : 1) : cap), kOptBlock, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint32_t*>(my_flags), world, sync_state, reinterpret_cast<uint4*>(grad_f16), n_vec);
    LNRF_LAUNCH_CHECK("exchange_finish");
    return LNRF_OK;
}

}  // extern "C"
