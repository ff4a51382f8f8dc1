// occupancy.cu -- occupancy-grid maintenance (row f-2 of SURVEY.md section 8): NeRFRenderer.update_extra_state
// (nerf/renderer.py:556-649), which the reference runs every 16 training steps as Python loops over ~25 small torch
// launches per cascade (meshgrid, cat, morton3D, five elementwise passes to build the jittered points, density(), indexed
// assignment, masked EMA, mean + .item(), packbits).  Here, per cascade:
//     lnrf_occupancy_points   cell coordinates (or the full-grid enumeration) + caller-supplied uniforms -> jittered world
//                             points and Morton indices, one pass, the reference's rounding sequence
//     [hash-grid encode + sigma net: lnrf_grid_encode_forward_world + lnrf_nerf_density]
//     lnrf_occupancy_scatter  tmp_grid[cas, idx] = sigma
// and once per update:
//     lnrf_occupancy_ema      density_grid = max(density_grid * decay, tmp_grid) where both are >= 0, tmp_grid re-armed to -1,
//                             mean(clamp(density_grid, 0)) reduced on the device (two-stage, deterministic)
//     lnrf_packbits_dev       bitfield from min(mean, density_thresh) read on the device -- no .item() on the path
// The random numbers stay with the caller (torch.rand / torch.randint, consumed in the reference's order), so a run with
// the same seed visits the same cells and jitters as the reference's update.
#include "common.cuh"
#include "march_core.cuh"

namespace lnrf {

// xyz = (2 * c / (H - 1) - 1) * (bound - hgs) + (u * 2 - 1) * hgs with every intermediate rounded to fp32 as torch does it
// (`t / python_scalar` is t * fl32(1 / scalar), renderer.py:585-597).  coords == nullptr: the full grid in meshgrid('ij')
// order, i = (x * H + y) * H + z.
__global__ void __launch_bounds__(256)
k_occ_points(const int* __restrict__ coords, const float* __restrict__ uniforms, const uint32_t N, const uint32_t H, const float inv_hm1,
             const float scale, const float hgs, float* __restrict__ xyzs, int* __restrict__ indices) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    uint32_t c[3];
    if (coords) {
        c[0] = (uint32_t)coords[(size_t)i * 3]; c[1] = (uint32_t)coords[(size_t)i * 3 + 1]; c[2] = (uint32_t)coords[(size_t)i * 3 + 2];
    } else {
        c[2] = i % H; c[1] = (i / H) % H; c[0] = i / (H * H);
    }
    indices[i] = (int)morton3d(c[0], c[1], c[2]);
#pragma unroll
    for (int d = 0; d < 3; d++) {
        const float x = f_add(f_mul(f_mul(2.0f, (float)c[d]), inv_hm1), -1.0f);
        const float u = uniforms[(size_t)i * 3 + d];
        const float jit = f_mul(f_add(f_mul(u, 2.0f), -1.0f), hgs);
        xyzs[(size_t)i * 3 + d] = f_add(f_mul(x, scale), jit);
    }
}

__global__ void __launch_bounds__(256)
k_occ_scatter(const float* __restrict__ sigmas, const int* __restrict__ indices, const uint32_t N, float* __restrict__ tmp_cas) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) tmp_cas[indices[i]] = sigmas[i];
}

// Duplicate indices resolved as torch's deterministic `tmp[idx] = sigma` does (the last occurrence wins): the largest sample index per
// cell is found with an integer max, then only that sample stores.  `winner` (int32 per cell) is -1 on entry and re-armed on exit.
__global__ void __launch_bounds__(256)
k_occ_scatter_claim(const int* __restrict__ indices, const uint32_t N, const uint32_t cells, int* __restrict__ winner) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N && (uint32_t)indices[i] < cells) atomicMax(winner + indices[i], (int)i);
}
__global__ void __launch_bounds__(256)
k_occ_scatter_store(const float* __restrict__ sigmas, const int* __restrict__ indices, const uint32_t N, const uint32_t cells,
                    int* __restrict__ winner, float* __restrict__ tmp_cas) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int idx = indices[i];
    if ((uint32_t)idx < cells && winner[idx] == (int)i) {  // a loser never reads its own index back, re-armed or not
        tmp_cas[idx] = sigmas[i];
        winner[idx] = -1;
    }
}

__global__ void __launch_bounds__(256) k_occ_fill(float* __restrict__ p, const uint32_t n, const float v) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = v;
}

// EMA (renderer.py:625-626) + per-block partial sums of clamp(grid, 0); tmp is reset to -1 for the next update
constexpr uint32_t kEmaBlocks = 1024;
__global__ void __launch_bounds__(256)
k_occ_ema(float* __restrict__ grid, float* __restrict__ tmp, const uint32_t n, const float decay, float* __restrict__ partial) {
    __shared__ float red[8];
    float acc = 0.0f;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float g = grid[i];
        const float t = tmp[i];
        if (g >= 0.0f && t >= 0.0f) {
            g = fmaxf(f_mul(g, decay), t);
            grid[i] = g;
        }
        tmp[i] = -1.0f;
        acc += fmaxf(g, 0.0f);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
        for (int w = 0; w < 8; w++) s += red[w];
        partial[blockIdx.x] = s;
    }
}
// mean_out[0] = mean(clamp(grid, 0)), mean_out[1] = min(mean, density_thresh) = the packbits threshold
__global__ void __launch_bounds__(256)
k_occ_mean(const float* __restrict__ partial, const uint32_t nblocks, const uint32_t n, const float density_thresh, float* __restrict__ mean_out) {
    __shared__ double red[8];
    double acc = 0.0;
    for (uint32_t i = threadIdx.x; i < nblocks; i += 256) acc += (double)partial[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; w++) s += red[w];
        const float mean = (float)(s / (double)n);
        mean_out[0] = mean;
        mean_out[1] = fminf(mean, density_thresh);
    }
}

// packbits (raymarching.cu:267-289) with the threshold read from device memory
__global__ void __launch_bounds__(256)
k_packbits_dev(const float* __restrict__ grid, const uint32_t N, const float* __restrict__ thresh_dev, uint8_t* __restrict__ bitfield) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float thresh = *thresh_dev;
    const float4 a = *reinterpret_cast<const float4*>(grid + (size_t)n * 8), b = *reinterpret_cast<const float4*>(grid + (size_t)n * 8 + 4);
    const uint32_t bits = (a.x > thresh ? 1u : 0u) | (a.y > thresh ? 2u : 0u) | (a.z > thresh ? 4u : 0u) | (a.w > thresh ? 8u : 0u) |
                          (b.x > thresh ? 16u : 0u) | (b.y > thresh ? 32u : 0u) | (b.z > thresh ? 64u : 0u) | (b.w > thresh ? 128u : 0u);
    bitfield[n] = (uint8_t)bits;
}

}  // namespace lnrf

using namespace lnrf;
static inline cudaStream_t S(lnrf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

namespace lnrf {
// Box around the occupied cells (lnrf_render_desc.occupied_box): per cascade the min / max cell coordinate of the set bits (bit index =
// cascade * H^3 + morton(x, y, z)), then the union of the cascades' boxes in world space with two cells of margin.  One launch:
// integer atomics into `work` (6 ints per cascade: min xyz, max xyz; + a ticket), the last block out converts and re-arms `work`.
__global__ void __launch_bounds__(256)
k_occupied_box(const uint8_t* __restrict__ bits, const uint32_t C, const uint32_t H, const float bound, int* __restrict__ work,
               float* __restrict__ box) {
    const uint32_t per = H * H * H / 8u;  // bytes per cascade
    __shared__ bool s_last;
    for (uint32_t c = 0; c < C; c++) {
        int lo[3] = {(int)H, (int)H, (int)H}, hi[3] = {-1, -1, -1};
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < per; i += gridDim.x * blockDim.x) {
            uint32_t b = bits[(size_t)c * per + i];
            while (b) {
                const uint32_t k = (uint32_t)__ffs((int)b) - 1u;
                b &= b - 1u;
                const uint32_t m = i * 8u + k;
                const int x = (int)morton3d_invert(m), y = (int)morton3d_invert(m >> 1), z = (int)morton3d_invert(m >> 2);
                lo[0] = min(lo[0], x); lo[1] = min(lo[1], y); lo[2] = min(lo[2], z);
                hi[0] = max(hi[0], x); hi[1] = max(hi[1], y); hi[2] = max(hi[2], z);
            }
        }
#pragma unroll
        for (int a = 0; a < 3; a++) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo[a] = min(lo[a], __shfl_xor_sync(kFull, lo[a], o));
                hi[a] = max(hi[a], __shfl_xor_sync(kFull, hi[a], o));
            }
            if ((threadIdx.x & 31) == 0) {
                if (lo[a] < (int)H) atomicMin(work + c * 6 + a, lo[a]);
                if (hi[a] >= 0) atomicMax(work + c * 6 + 3 + a, hi[a]);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(reinterpret_cast<unsigned int*>(work + 6 * C), 1u) == gridDim.x - 1u;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        float wlo[3] = {INFINITY, INFINITY, INFINITY}, whi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (uint32_t c = 0; c < C; c++) {
            const float half = fminf((float)(1u << c), bound);  // mip_bound of the cascade (march_probe)
            const float cell = 2.0f * half / (float)H;
            for (int a = 0; a < 3; a++) {
                const int l = __ldcg(work + c * 6 + a), h = __ldcg(work + c * 6 + 3 + a);
                if (h >= 0) {
                    wlo[a] = fminf(wlo[a], -half + ((float)l - 2.0f) * cell);
                    whi[a] = fmaxf(whi[a], -half + ((float)h + 3.0f) * cell);
                }
                work[c * 6 + a] = (int)H;
                work[c * 6 + 3 + a] = -1;
            }
        }
        for (int a = 0; a < 3; a++) { box[a] = wlo[a]; box[3 + a] = whi[a]; }
        work[6 * C] = 0;
    }
}

}  // namespace lnrf

extern "C" {

int lnrf_occupancy_points(const int32_t* coords, const float* uniforms, uint32_t N, uint32_t H, float cascade_bound, float* xyzs,
                          int32_t* indices, lnrf_stream_t stream) {
    if (N == 0) return LNRF_OK;
    LNRF_REQUIRE(uniforms && xyzs && indices, "occupancy_points: null pointer");
    LNRF_REQUIRE(H >= 2 && H <= 1024 && cascade_bound > 0.0f, "occupancy_points: H=%u / bound out of range", H);
    LNRF_REQUIRE(coords || (uint64_t)N == (uint64_t)H * H * H, "occupancy_points: the full-grid enumeration needs N == H^3");
    // python: half_grid_size = bound / H (double); the tensor ops see fl32(bound - hgs), fl32(hgs), fl32(1 / (H - 1))
    const double hgs = (double)cascade_bound / (double)H;
    k_occ_points<<<div_up(N, 256u), 256, 0, S(stream)>>>(coords, uniforms, N, H, (float)(1.0 / (double)(H - 1)),
                                                         (float)((double)cascade_bound - hgs), (float)hgs, xyzs, indices);
    LNRF_LAUNCH_CHECK("occupancy_points");
    return LNRF_OK;
}

int lnrf_occupancy_scatter(const float* sigmas, const int32_t* indices, uint32_t N, float* tmp_grid_cascade, lnrf_stream_t stream) {
    if (N == 0) return LNRF_OK;
    LNRF_REQUIRE(sigmas && indices && tmp_grid_cascade, "occupancy_scatter: null pointer");
    k_occ_scatter<<<div_up(N, 256u), 256, 0, S(stream)>>>(sigmas, indices, N, tmp_grid_cascade);
    LNRF_LAUNCH_CHECK("occupancy_scatter");
    return LNRF_OK;
}

int lnrf_occupancy_scatter_det(const float* sigmas, const int32_t* indices, uint32_t N, float* tmp_grid_cascade, int32_t* winner,
                               uint32_t cells, lnrf_stream_t stream) {
    if (N == 0) return LNRF_OK;
    LNRF_REQUIRE(sigmas && indices && tmp_grid_cascade && winner, "occupancy_scatter_det: null pointer");
    LNRF_REQUIRE(cells > 0 && N <= 0x7fffffffu, "occupancy_scatter_det: cells must be > 0 and N < 2^31");
    k_occ_scatter_claim<<<div_up(N, 256u), 256, 0, S(stream)>>>(indices, N, cells, winner);
    LNRF_LAUNCH_CHECK("occupancy_scatter_det(claim)");
    k_occ_scatter_store<<<div_up(N, 256u), 256, 0, S(stream)>>>(sigmas, indices, N, cells, winner, tmp_grid_cascade);
    LNRF_LAUNCH_CHECK("occupancy_scatter_det");
    return LNRF_OK;
}

int lnrf_occupancy_fill(float* grid, uint32_t n, float value, lnrf_stream_t stream) {
    if (n == 0) return LNRF_OK;
    LNRF_REQUIRE(grid, "occupancy_fill: null pointer");
    const uint32_t want = div_up(n, 256u), cap = (uint32_t)kNumSMs * 8u;
    k_occ_fill<<<want < cap ? want : cap, 256, 0, S(stream)>>>(grid, n, value);
    LNRF_LAUNCH_CHECK("occupancy_fill");
    return LNRF_OK;
}

size_t lnrf_occupancy_scratch_bytes(void) { return sizeof(float) * kEmaBlocks; }

int lnrf_occupancy_ema(float* density_grid, float* tmp_grid, uint32_t n, float decay, float density_thresh, float* mean_out,
                       void* scratch, size_t scratch_bytes, lnrf_stream_t stream) {
    LNRF_REQUIRE(density_grid && tmp_grid && mean_out && n > 0, "occupancy_ema: null pointer / empty grid");
    if (!scratch || scratch_bytes < lnrf_occupancy_scratch_bytes()) {
        set_error("occupancy_ema: scratch too small (%zu < %zu)", scratch_bytes, lnrf_occupancy_scratch_bytes());
        return LNRF_ERR_SCRATCH_TOO_SMALL;
    }
    const uint32_t want = div_up(n, 256u);
    const uint32_t blocks = want < kEmaBlocks ? want : kEmaBlocks;
    k_occ_ema<<<blocks, 256, 0, S(stream)>>>(density_grid, tmp_grid, n, decay, (float*)scratch);
    LNRF_LAUNCH_CHECK("occupancy_ema");
    k_occ_mean<<<1, 256, 0, S(stream)>>>((const float*)scratch, blocks, n, density_thresh, mean_out);
    LNRF_LAUNCH_CHECK("occupancy_ema(mean)");
    return LNRF_OK;
}

int lnrf_packbits_dev(const float* grid, uint32_t N, const float* thresh_dev, uint8_t* bitfield, lnrf_stream_t stream) {
    if (N == 0) return LNRF_OK;
    LNRF_REQUIRE(grid && bitfield && thresh_dev, "packbits_dev: null pointer");
    LNRF_REQUIRE((reinterpret_cast<uintptr_t>(grid) & 15) == 0, "packbits_dev: grid must be 16-byte aligned");
    k_packbits_dev<<<div_up(N, 256u), 256, 0, S(stream)>>>(grid, N, thresh_dev, bitfield);
    LNRF_LAUNCH_CHECK("packbits_dev");
    return LNRF_OK;
}

size_t lnrf_occupied_box_work_ints(uint32_t C) { return 6 * (size_t)C + 1; }

int lnrf_occupied_box(const uint8_t* bitfield, uint32_t C, uint32_t H, float bound, int32_t* work, float* box, lnrf_stream_t stream) {
    LNRF_REQUIRE(bitfield && work && box, "occupied_box: null pointer");
    LNRF_REQUIRE(C >= 1 && C <= 16 && H >= 2 && H <= 1024 && (H & (H - 1)) == 0, "occupied_box: cascades must be in [1, 16] and H a power of two <= 1024");
    k_occupied_box<<<kNumSMs * 2, 256, 0, S(stream)>>>(bitfield, C, H, bound, work, box);
    LNRF_LAUNCH_CHECK("occupied_box");
    return LNRF_OK;
}

}  // extern "C"
