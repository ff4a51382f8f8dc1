// gridenc.cu -- multiresolution hash/tiled grid encoder for sm_100a (forward, backward, TV gradient).
//
// Replaces gridencoder/src/gridencoder.cu of the reference (kernel_grid :87-245, kernel_grid_backward :248-340,
// kernel_input_backward :343-369, kernel_grad_tv :506-610).  Design (DESIGN.md section 4):
//   * hot shape (D = 3, C = 2, no dy_dx, [B, L*C] output): a CTA owns a tile of 128 consecutive samples for ALL
//     levels.  A warp always works on 32 consecutive samples of ONE level (samples of a ray are spatially
//     coherent, so the 8 corner gathers of neighbouring lanes share sectors / L1 lines), the 8 gathers of an item
//     are issued back to back, and the per-level results are transposed through shared memory so that the
//     [B, L*C] row-major output the Python API returns is written directly and fully coalesced -- the reference
//     writes [L, B, C] and then pays a permute+reshape copy (grid.py:57).  Interpolation accumulates in fp32 and
//     rounds once (the reference rounds to scalar_t after each of the 8 corners).
//   * backward: same tiling; gradient rows are staged through shared memory (coalesced 64-byte rows), corner
//     weights are recomputed, and each corner is one packed f16x2 (or v2.f32) reduction that never returns a value.
//   * everything else (D = 2, C in {1,4,8}, dy_dx, [L,B,C] layout) takes a generic thread-per-(sample, level) path.
// Index arithmetic is uint32 and bit-identical to the reference (gridencoder.cu:50-84), including the per-level
// scale evaluated on the device as fma(exp2f(level * S), H, -1).
#include <cfloat>

#include "common.cuh"

namespace lnrf {

constexpr uint32_t kPrime1 = 2654435761u, kPrime2 = 805459861u;  // gridencoder.cu:54 (primes[0] == 1)
constexpr int kMaxLevels = 32;

struct GridOffsets {
    uint32_t v[kMaxLevels + 1];
};

struct Level {
    float scale;
    uint32_t res, hs, base;
    uint32_t str1, str2;  // strides of dims 1 and 2 when they take part in the dense index, else 0
    uint32_t hashed;
    uint32_t mask;        // hs - 1 when hs is a power of two (every hashed level of a 2^k table), else 0
};

// gridencoder.cu:66-84 + :138-139, for one level
template <int D>
__device__ __forceinline__ Level make_level(uint32_t level, float S, uint32_t H, const GridOffsets& off, uint32_t gridtype,
                                            bool align_corners) {
    Level lv;
    lv.scale = __fmaf_rn(exp2f(__fmul_rn((float)level, S)), (float)H, -1.0f);
    lv.res = (uint32_t)ceilf(lv.scale) + 1u;
    lv.base = off.v[level];
    lv.hs = off.v[level + 1] - off.v[level];
    const uint32_t step = align_corners ? lv.res : lv.res + 1u;
    uint32_t stride = 1;
    lv.str1 = lv.str2 = 0;
    // d = 0 always contributes (stride 1 <= hashmap_size)
    stride *= step;
    if (D > 1 && stride <= lv.hs) {
        lv.str1 = stride;
        stride *= step;
        if (D > 2 && stride <= lv.hs) {
            lv.str2 = stride;
            stride *= step;
        }
    }
    lv.hashed = (gridtype == 0u && stride > lv.hs) ? 1u : 0u;
    lv.mask = (lv.hs & (lv.hs - 1u)) == 0u ? lv.hs - 1u : 0u;
    return lv;
}

template <int D>
__device__ __forceinline__ uint32_t grid_index(const Level& lv, const uint32_t* pg) {
    uint32_t index;
    if (lv.hashed) {
        index = pg[0];
        if (D > 1) index ^= pg[1] * kPrime1;
        if (D > 2) index ^= pg[2] * kPrime2;
    } else {
        index = pg[0];
        if (D > 1) index += pg[1] * lv.str1;
        if (D > 2) index += pg[2] * lv.str2;
    }
    // index % hashmap_size (gridencoder.cu:83) without the integer division on the hot shapes: a mask for
    // power-of-two tables, nothing at all when a dense index is already in range (the reference sizes dense levels
    // as (res+1)^D rounded up, so this is the common case), the real remainder otherwise
    if (lv.mask) return index & lv.mask;
    return index < lv.hs ? index : index % lv.hs;
}

// The 8 corner indices of a 3-D cell (same values as 8 grid_index<3> calls).  `lv` is warp-uniform in the tile kernels, so the
// branch is taken once per item instead of once per corner: hashed power-of-two tables need two multiplies and eight xor/and
// (uint32 wrap-around: (y + 1) * P == y * P + P); dense levels are base + stride sums, in range whenever the far corner is.
__device__ __forceinline__ void corner_indices3(const Level& lv, const uint32_t* pg, uint32_t* idx) {
    if (lv.hashed && lv.mask) {
        const uint32_t x0 = pg[0], x1 = pg[0] + 1u;
        const uint32_t y0 = pg[1] * kPrime1, y1 = y0 + kPrime1;
        const uint32_t z0 = pg[2] * kPrime2, z1 = z0 + kPrime2;
        const uint32_t a00 = y0 ^ z0, a10 = y1 ^ z0, a01 = y0 ^ z1, a11 = y1 ^ z1;
        idx[0] = (x0 ^ a00) & lv.mask; idx[1] = (x1 ^ a00) & lv.mask;
        idx[2] = (x0 ^ a10) & lv.mask; idx[3] = (x1 ^ a10) & lv.mask;
        idx[4] = (x0 ^ a01) & lv.mask; idx[5] = (x1 ^ a01) & lv.mask;
        idx[6] = (x0 ^ a11) & lv.mask; idx[7] = (x1 ^ a11) & lv.mask;
    } else if (!lv.hashed) {
        const uint32_t b = pg[0] + pg[1] * lv.str1 + pg[2] * lv.str2;
        idx[0] = b; idx[1] = b + 1u;
        idx[2] = b + lv.str1; idx[3] = idx[2] + 1u;
        idx[4] = b + lv.str2; idx[5] = idx[4] + 1u;
        idx[6] = idx[4] + lv.str1; idx[7] = idx[6] + 1u;
        if (idx[7] >= lv.hs) {  // only when a caller hands in a table smaller than the level (index % hashmap_size, gridencoder.cu:83)
#pragma unroll
            for (int c = 0; c < 8; c++) idx[c] = lv.mask ? (idx[c] & lv.mask) : (idx[c] < lv.hs ? idx[c] : idx[c] % lv.hs);
        }
    } else {
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const uint32_t pgl[3] = {pg[0] + (c & 1), pg[1] + ((c >> 1) & 1), pg[2] + ((c >> 2) & 1)};
            idx[c] = grid_index<3>(lv, pgl);
        }
    }
}

template <typename T> struct Vec2;
template <> struct Vec2<__half> { using type = __half2; };
template <> struct Vec2<float> { using type = float2; };

__device__ __forceinline__ float2 ld2(const __half2* p) { return __half22float2(__ldg(p)); }
__device__ __forceinline__ float2 ld2(const float2* p) { return __ldg(p); }
__device__ __forceinline__ void cvt2(float2 v, __half2& o) { o = __floats2half2_rn(v.x, v.y); }
__device__ __forceinline__ void cvt2(float2 v, float2& o) { o = v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ void from_f(float v, __half& o) { o = __float2half_rn(v); }
__device__ __forceinline__ void from_f(float v, float& o) { o = v; }

// packed reductions without a return value (RED.E.ADD.F16x2.RN / RED.E.ADD.v2.F32)
__device__ __forceinline__ void red2(__half2* p, float2 v) {
    const __half2 h = __floats2half2_rn(v.x, v.y);
    asm volatile("red.global.add.noftz.f16x2 [%0], %1;" ::"l"(p), "r"(*reinterpret_cast<const uint32_t*>(&h)) : "memory");
}
__device__ __forceinline__ void red2(float2* p, float2 v) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
// Two table entries that share an aligned 8-byte (16-byte for fp32) slot in ONE reduction (REDG.E.ADD.F16x4): the x / x+1 corners of
// a cell are such a pair whenever the first index is even -- always adjacent on dense levels, and on hashed levels exactly when
// pg[0] is even (x ^ h and (x + 1) ^ h then differ in bit 0 only).  Same per-lane fp16 adds as two separate reductions.
__device__ __forceinline__ void red4(__half2* p, float2 a, float2 b) {
    const __half2 ha = __floats2half2_rn(a.x, a.y), hb = __floats2half2_rn(b.x, b.y);
    asm volatile("red.global.add.noftz.v2.f16x2 [%0], {%1, %2};" ::"l"(p), "r"(*reinterpret_cast<const uint32_t*>(&ha)),
                 "r"(*reinterpret_cast<const uint32_t*>(&hb)) : "memory");
}
__device__ __forceinline__ void red4(float2* p, float2 a, float2 b) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y) : "memory");
}
__device__ __forceinline__ void ld2x2(const __half2* p, float2& a, float2& b) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
    b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
}
__device__ __forceinline__ void ld2x2(const float2* p, float2& a, float2& b) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    a = make_float2(v.x, v.y);
    b = make_float2(v.z, v.w);
}
__device__ __forceinline__ void red1(__half* p, float v) { atomicAdd(p, __float2half_rn(v)); }
__device__ __forceinline__ void red1(float* p, float v) { atomicAdd(p, v); }

// Deterministic table gradient (torch.use_deterministic_algorithms; DESIGN.md section 4, "Deterministic backward").  The fp32 value
// a thread flushes depends only on the sample indices it owns (fixed 128-sample tile, fixed 8-sample run, fixed carry rule), never
// on which CTA runs the tile; only the float reductions at L2 make the sum order-dependent.  Here a flush adds round(p / q) to an
// int64 fixed-point sum instead, and integer addition is associative.  q = 2^qexp, qexp = E + ceil(log2 B) + 1 - 62 with 2^E >=
// max |g| over the rows read: the corner weights of a sample sum to 1 within a level, so |sum| <= B * 2^E (1 + eps) < 2^62 q and
// no int64 sum wraps.  A non-finite p sets its entry's flag instead (the finish kernel writes NaN there).
struct DetSink {
    unsigned long long* acc;  // [entries, C] two's-complement fixed-point sums, zero between calls (k_det_finish re-arms them)
    uint32_t* flag;           // [entries] non-zero: a contribution was non-finite; zero between calls
    const uint32_t* gmax;     // fp32 gradients: bit pattern of max finite |g| (k_det_absmax); nullptr: fp16, |g| < 2^16
    int lb;                   // ceil(log2 B), B = the row capacity of the call
};
constexpr int kDetMinExp = -60;  // E for an all-zero gradient: keeps 2^-qexp a normal float

__device__ __forceinline__ int det_qexp(const DetSink& d) {
    int E = 16;
    if (d.gmax) {
        const uint32_t m = *d.gmax;  // 2^((m >> 23) - 126) > m for every finite non-negative float
        E = m == 0u ? kDetMinExp : max((int)(m >> 23) - 126, kDetMinExp);
    }
    return E + d.lb + 1 - 62;
}
__device__ __forceinline__ float det_inv_q(const DetSink& d) { return __int_as_float((127 - det_qexp(d)) << 23); }  // exact 2^-qexp

__device__ __forceinline__ void det_red(unsigned long long* p, float v, float inv_q) {
    const long long q = __float2ll_rn(__fmul_rn(v, inv_q));  // the multiply by a power of two is exact
    if (q) asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(q) : "memory");
}
// entry e of a C = 2 table
__device__ __forceinline__ void det_add2(const DetSink& d, size_t e, float2 v, float inv_q) {
    if (!isfinite(v.x) || !isfinite(v.y)) { d.flag[e] = 1u; return; }
    det_red(d.acc + e * 2, v.x, inv_q);
    det_red(d.acc + e * 2 + 1, v.y, inv_q);
}

// position inside the level: cell + interpolation weights (gridencoder.cu:141-163)
template <int D, bool SMOOTH>
__device__ __forceinline__ void cell_of(const Level& lv, const float* x, bool align_corners, uint32_t* pg, float* pos,
                                        float* pos_deriv) {
#pragma unroll
    for (int d = 0; d < D; d++) {
        const float p = __fmaf_rn(x[d], lv.scale, align_corners ? 0.0f : 0.5f);
        const float fl = floorf(p);
        pg[d] = (uint32_t)fl;
        float f = __fadd_rn(p, -(float)pg[d]);
        if (SMOOTH) {
            if (pos_deriv) pos_deriv[d] = 6.0f * f * (1.0f - f);
            f = f * f * (3.0f - 2.0f * f);
        } else if (pos_deriv) {
            pos_deriv[d] = 1.0f;
        }
        pos[d] = f;
    }
}

// =========================================================================================================
// hot path: D = 3, C = 2, tile of 128 samples x all levels per CTA
// =========================================================================================================
constexpr int kTile = 128;
constexpr int kGridThreads = 256;

template <typename T, bool SMOOTH, bool PAIR>
__global__ void __launch_bounds__(kGridThreads)
k_grid_fwd_tile(const float* __restrict__ inputs, const typename Vec2<T>::type* __restrict__ emb,
                typename Vec2<T>::type* __restrict__ outputs, uint32_t B, const uint32_t L, const float S,
                const uint32_t H, const uint32_t gridtype, const bool align_corners, const GridOffsets off,
                uint32_t ntiles, const float in_bound, const int* __restrict__ B_dev) {
    using T2 = typename Vec2<T>::type;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ Level s_lv[kMaxLevels];
    __shared__ float s_in[kTile * 3];
    T2* s_out = reinterpret_cast<T2*>(s_raw);
    pdl_trigger();
    pdl_wait();  // nothing below may run before the kernels ahead on the stream are complete (common.cuh)
    if (B_dev) {  // device-side sample count (render control block, row f-3; the training marcher's counter): whole 128-row tiles up
                  // to the capacity B -- the rows between the count and the tile end are the marcher's zero padding, encoded like any
                  // other point (the network kernels work on the same 128-row tiles)
        const uint32_t live = div_up((uint32_t)max(*B_dev, 0), (uint32_t)kTile) * (uint32_t)kTile;
        B = live < B ? live : B;
        ntiles = div_up(B, (uint32_t)kTile);
    }
    // torch evaluates `t / python_scalar` as t * (1 / scalar) with the reciprocal rounded to fp32 (div_true_kernel_cuda), and that
    // is what the reference's grid.py:147 runs; the same two roundings here
    const float in_inv = in_bound > 0.0f ? __fdiv_rn(1.0f, __fmul_rn(2.0f, in_bound)) : 0.0f;
    const uint32_t LP = L | 1u;  // odd row pitch: conflict-free transposition
    const int tid = threadIdx.x;
    if (tid < (int)L) s_lv[tid] = make_level<3>(tid, S, H, off, gridtype, align_corners);

    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const size_t b0 = (size_t)tile * kTile;
        const uint32_t rows = (uint32_t)min((size_t)kTile, (size_t)B - b0);
        __syncthreads();  // previous tile's copy-out finished with s_out / s_in (also publishes s_lv)
        // in_bound > 0: the caller passes world coordinates and GridEncoder.forward's (x + bound) / (2 * bound) (grid.py:147) is
        // applied here with the same two roundings instead of two elementwise passes over [B, 3]
        for (uint32_t i = tid; i < rows * 3; i += kGridThreads) {
            const float x = __ldcs(inputs + b0 * 3 + i);
            s_in[i] = in_bound > 0.0f ? __fmul_rn(__fadd_rn(x, in_bound), in_inv) : x;
        }
        __syncthreads();
        const uint32_t nitems = L * kTile;
#pragma unroll 2
        for (uint32_t i = tid; i < nitems; i += kGridThreads) {
            const uint32_t level = i >> 7, s = i & (kTile - 1);
            if (s >= rows) continue;
            const Level lv = s_lv[level];
            const float x[3] = {s_in[s * 3], s_in[s * 3 + 1], s_in[s * 3 + 2]};
            float2 acc = make_float2(0.f, 0.f);
            const bool inside = !(x[0] < 0.f || x[0] > 1.f || x[1] < 0.f || x[1] > 1.f || x[2] < 0.f || x[2] > 1.f);
            if (inside) {
                uint32_t pg[3];
                float pos[3];
                cell_of<3, SMOOTH>(lv, x, align_corners, pg, pos, nullptr);
                const T2* grid = emb + lv.base;
                uint32_t idx[8];
                corner_indices3(lv, pg, idx);
                float2 v[8];
                if (PAIR && (reinterpret_cast<uintptr_t>(grid) & (2 * sizeof(T2) - 1)) == 0 && !(lv.hs & 1u)) {
                    // x / x+1 corners that share an aligned slot (see red4) come in with ONE load, without a divergent branch:
                    // every lane loads the aligned slot of its x corner; only lanes whose x+1 corner lives elsewhere issue the
                    // second (predicated) load.  Level sizes are even (multiples of 8 entries in grid.py:114), so the slot stays inside the level.
#pragma unroll
                    for (int c = 0; c < 8; c += 2) {
                        float2 lo, hi;
                        ld2x2(grid + (idx[c] & ~1u), lo, hi);
                        const bool odd = idx[c] & 1u;
                        v[c] = odd ? hi : lo;
                        v[c + 1] = hi;
                        if (odd || idx[c + 1] != idx[c] + 1u) v[c + 1] = ld2(grid + idx[c + 1]);
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < 8; c++) v[c] = ld2(grid + idx[c]);
                }
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    const float w = ((c & 1) ? pos[0] : 1.0f - pos[0]) * ((c & 2) ? pos[1] : 1.0f - pos[1]) *
                                    ((c & 4) ? pos[2] : 1.0f - pos[2]);
                    acc.x = fmaf(w, v[c].x, acc.x);
                    acc.y = fmaf(w, v[c].y, acc.y);
                }
            }
            T2 o;
            cvt2(acc, o);
            s_out[s * LP + level] = o;
        }
        __syncthreads();
        T2* out = outputs + b0 * L;
        for (uint32_t j = tid; j < rows * L; j += kGridThreads) {
            const uint32_t s = j / L, l = j - s * L;
            __stcs(out + j, s_out[s * LP + l]);
        }
    }
}

// Backward of the hot shape.  A thread owns ONE level and a run of kRun = 8 CONSECUTIVE samples of the tile (16 runs x
// L levels = 256 work items for L = 16).  Samples of a ray are ordered along the ray, so on the coarse levels several
// consecutive samples fall into the same grid cell (dt = 1/592 of the normalised cube vs. a cell of 1/16 .. 1/80 on
// levels 0-5): their 8 corner contributions are summed in registers and flushed as ONE packed reduction per corner
// when the cell changes.  That removes up to 8x of the same-address atomics that serialise in L2 on the small dense
// levels (level 0 has 4920 entries for 2.3e5 samples x 8 corners) -- the reference issues every one of them.
constexpr int kRun = 8;

// DET: the flushes go to the fixed-point sums of `det` (see DetSink) instead of reductions into grad_emb.
template <typename T, bool SMOOTH, bool PAIR, bool DET>
__global__ void __launch_bounds__(kGridThreads)
k_grid_bwd_tile(const typename Vec2<T>::type* __restrict__ grad, const float* __restrict__ inputs,
                typename Vec2<T>::type* __restrict__ grad_emb, const uint32_t B, const uint32_t L, const float S,
                const uint32_t H, const uint32_t gridtype, const bool align_corners, const GridOffsets off,
                uint32_t ntiles, const float in_bound, const int* __restrict__ B_dev, const DetSink det) {
    using T2 = typename Vec2<T>::type;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ Level s_lv[kMaxLevels];
    __shared__ float s_in[kTile * 3];
    T2* s_g = reinterpret_cast<T2*>(s_raw);
    pdl_trigger();
    pdl_wait();
    if (B_dev) {  // rows at or beyond the device-side count carry no gradient (and may be unwritten memory): skipped by whole tiles
        const uint32_t live = div_up((uint32_t)max(*B_dev, 0), (uint32_t)kTile);
        ntiles = live < ntiles ? live : ntiles;
    }
    // torch evaluates `t / python_scalar` as t * (1 / scalar) with the reciprocal rounded to fp32 (div_true_kernel_cuda), and that
    // is what the reference's grid.py:147 runs; the same two roundings here
    const float in_inv = in_bound > 0.0f ? __fdiv_rn(1.0f, __fmul_rn(2.0f, in_bound)) : 0.0f;
    const uint32_t LP = L | 1u;
    const int tid = threadIdx.x;
    if (tid < (int)L) s_lv[tid] = make_level<3>(tid, S, H, off, gridtype, align_corners);
    float inv_q = 0.0f;
    if constexpr (DET) inv_q = det_inv_q(det);  // after pdl_wait: the max pre-pass ran ahead on the stream

    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const size_t b0 = (size_t)tile * kTile;
        const uint32_t rows = (uint32_t)min((size_t)kTile, (size_t)B - b0);
        __syncthreads();
        for (uint32_t i = tid; i < rows * 3; i += kGridThreads) {
            const float x = __ldcs(inputs + b0 * 3 + i);
            s_in[i] = in_bound > 0.0f ? __fmul_rn(__fadd_rn(x, in_bound), in_inv) : x;
        }
        const T2* g = grad + b0 * L;
        for (uint32_t j = tid; j < rows * L; j += kGridThreads) {
            const uint32_t s = j / L, l = j - s * L;
            s_g[s * LP + l] = __ldcs(g + j);
        }
        __syncthreads();
        const uint32_t nitems = L * (kTile / kRun);
        for (uint32_t item = tid; item < nitems; item += kGridThreads) {
            const uint32_t level = item / (kTile / kRun), s0 = (item % (kTile / kRun)) * kRun;
            const Level lv = s_lv[level];
            T2* gg = grad_emb + lv.base;
            uint32_t cell[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};
            uint32_t idx[8];
            float2 acc[8];
            bool open = false;
            const bool slot_ok = PAIR && (reinterpret_cast<uintptr_t>(gg) & (2 * sizeof(T2) - 1)) == 0;
            // flush the corners c with (c & kmask) != kval: all of them for kmask = 0, kval = 1
            auto flush = [&](uint32_t kmask, uint32_t kval) {
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    const bool f0 = ((uint32_t)c & kmask) != kval, f1 = ((uint32_t)(c + 1) & kmask) != kval;
                    const bool nz0 = acc[c].x != 0.f || acc[c].y != 0.f, nz1 = acc[c + 1].x != 0.f || acc[c + 1].y != 0.f;
                    if constexpr (DET) {  // no 64-bit vector reduction exists: one per corner and channel
                        if (f0 && nz0) det_add2(det, (size_t)lv.base + idx[c], acc[c], inv_q);
                        if (f1 && nz1) det_add2(det, (size_t)lv.base + idx[c + 1], acc[c + 1], inv_q);
                    } else if (f0 && f1 && slot_ok && !(idx[c] & 1u) && idx[c + 1] == idx[c] + 1u) {
                        if (nz0 || nz1) red4(gg + idx[c], acc[c], acc[c + 1]);
                    } else {
                        if (f0 && nz0) red2(gg + idx[c], acc[c]);
                        if (f1 && nz1) red2(gg + idx[c + 1], acc[c + 1]);
                    }
                }
            };
#pragma unroll 1
            for (uint32_t j = 0; j < (uint32_t)kRun; j++) {
                const uint32_t s = s0 + j;
                if (s >= rows) break;
                const float x[3] = {s_in[s * 3], s_in[s * 3 + 1], s_in[s * 3 + 2]};
                if (x[0] < 0.f || x[0] > 1.f || x[1] < 0.f || x[1] > 1.f || x[2] < 0.f || x[2] > 1.f) continue;
                const T2 gt = s_g[s * LP + level];
                const float2 gv = make_float2(to_f(gt.x), to_f(gt.y));
                if (gv.x == 0.f && gv.y == 0.f) continue;  // adding +-0 changes nothing (padding rows, dead samples)
                uint32_t pg[3];
                float pos[3];
                cell_of<3, SMOOTH>(lv, x, align_corners, pg, pos, nullptr);
                if (!open || pg[0] != cell[0] || pg[1] != cell[1] || pg[2] != cell[2]) {
                    // A neighbouring cell (every axis moved by at most one) shares a face, an edge or a vertex with the open one: those
                    // corners are the same grid points, hence the same table entries, so their sums stay in registers instead of being
                    // flushed.  Old corner c is kept iff (c & kmask) == kval, and becomes corner c ^ kmask of the new cell.
                    uint32_t kmask = 0u, kval = 1u;  // nothing kept
                    if (open) {
                        uint32_t m = 0u, v = 0u;
                        bool near = true;
#pragma unroll
                        for (int a = 0; a < 3; a++) {
                            if (pg[a] == cell[a] + 1u) { m |= 1u << a; v |= 1u << a; }
                            else if (pg[a] + 1u == cell[a]) m |= 1u << a;
                            else if (pg[a] != cell[a]) near = false;
                        }
                        if (near) { kmask = m; kval = v; }
                        flush(kmask, kval);
                    }
#pragma unroll
                    for (int a = 0; a < 3; a++) {
                        if (kmask & (1u << a)) {
#pragma unroll
                            for (int c = 0; c < 8; c++) {
                                if (c & (1 << a)) continue;
                                const float2 t = acc[c]; acc[c] = acc[c | (1 << a)]; acc[c | (1 << a)] = t;
                            }
                        }
                    }
#pragma unroll
                    for (int c = 0; c < 8; c++)
                        if (((uint32_t)c & kmask) != (kval ^ kmask)) acc[c] = make_float2(0.f, 0.f);
                    open = true;
                    cell[0] = pg[0]; cell[1] = pg[1]; cell[2] = pg[2];
                    corner_indices3(lv, pg, idx);
                }
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    const float w = ((c & 1) ? pos[0] : 1.0f - pos[0]) * ((c & 2) ? pos[1] : 1.0f - pos[1]) *
                                    ((c & 4) ? pos[2] : 1.0f - pos[2]);
                    acc[c].x = fmaf(w, gv.x, acc[c].x);
                    acc[c].y = fmaf(w, gv.y, acc[c].y);
                }
            }
            if (open) flush(0u, 1u);
        }
    }
}

// =========================================================================================================
// generic path: thread per (sample, level); any D in {2,3}, C in {1,2,4,8}, both layouts, optional dy_dx
// =========================================================================================================
template <typename T, int D, int C, bool SMOOTH>
__global__ void __launch_bounds__(256)
k_grid_fwd_generic(const float* __restrict__ inputs, const T* __restrict__ emb, T* __restrict__ outputs, const uint32_t B,
                   const uint32_t L, const float S, const uint32_t H, T* __restrict__ dy_dx, const uint32_t gridtype,
                   const bool align_corners, const GridOffsets off, const int layout) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t level = blockIdx.y;
    if (b >= B) return;
    const Level lv = make_level<D>(level, S, H, off, gridtype, align_corners);
    T* out = layout == LNRF_GRID_LBC ? outputs + ((size_t)level * B + b) * C : outputs + ((size_t)b * L + level) * C;
    T* dd = dy_dx ? dy_dx + ((size_t)b * L + level) * D * C : nullptr;
    float x[D];
    bool inside = true;
#pragma unroll
    for (int d = 0; d < D; d++) {
        x[d] = inputs[(size_t)b * D + d];
        if (x[d] < 0.f || x[d] > 1.f) inside = false;
    }
    if (!inside) {
#pragma unroll
        for (int ch = 0; ch < C; ch++) from_f(0.f, out[ch]);
        if (dd)
            for (int i = 0; i < D * C; i++) from_f(0.f, dd[i]);
        return;
    }
    uint32_t pg[D];
    float pos[D], pos_deriv[D];
    cell_of<D, SMOOTH>(lv, x, align_corners, pg, pos, pos_deriv);
    const T* grid = emb + (size_t)lv.base * C;
    float res[C];
#pragma unroll
    for (int ch = 0; ch < C; ch++) res[ch] = 0.f;
#pragma unroll
    for (int c = 0; c < (1 << D); c++) {
        float w = 1.f;
        uint32_t pgl[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            if (c & (1 << d)) { w *= pos[d]; pgl[d] = pg[d] + 1; }
            else { w *= 1.0f - pos[d]; pgl[d] = pg[d]; }
        }
        const size_t index = (size_t)grid_index<D>(lv, pgl) * C;
#pragma unroll
        for (int ch = 0; ch < C; ch++) res[ch] = fmaf(w, to_f(__ldg(grid + index + ch)), res[ch]);
    }
#pragma unroll
    for (int ch = 0; ch < C; ch++) from_f(res[ch], out[ch]);
    if (dd) {  // gridencoder.cu:205-243
#pragma unroll
        for (int gd = 0; gd < D; gd++) {
            float rg[C];
#pragma unroll
            for (int ch = 0; ch < C; ch++) rg[ch] = 0.f;
#pragma unroll
            for (int c = 0; c < (1 << (D - 1)); c++) {
                float w = lv.scale;
                uint32_t pgl[D];
#pragma unroll
                for (int nd = 0; nd < D - 1; nd++) {
                    const int d = (nd >= gd) ? (nd + 1) : nd;
                    if (c & (1 << nd)) { w *= pos[d]; pgl[d] = pg[d] + 1; }
                    else { w *= 1.0f - pos[d]; pgl[d] = pg[d]; }
                }
                pgl[gd] = pg[gd];
                const size_t il = (size_t)grid_index<D>(lv, pgl) * C;
                pgl[gd] = pg[gd] + 1;
                const size_t ir = (size_t)grid_index<D>(lv, pgl) * C;
#pragma unroll
                for (int ch = 0; ch < C; ch++)
                    rg[ch] += w * (to_f(__ldg(grid + ir + ch)) - to_f(__ldg(grid + il + ch))) * pos_deriv[gd];
            }
#pragma unroll
            for (int ch = 0; ch < C; ch++) from_f(rg[ch], dd[gd * C + ch]);
        }
    }
}

template <typename T, int D, int C, bool SMOOTH, bool DET>
__global__ void __launch_bounds__(256)
k_grid_bwd_generic(const T* __restrict__ grad, const float* __restrict__ inputs, T* __restrict__ grad_emb, const uint32_t B,
                   const uint32_t L, const float S, const uint32_t H, const uint32_t gridtype, const bool align_corners,
                   const GridOffsets off, const int layout, const DetSink det) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t level = blockIdx.y;
    if (b >= B) return;
    const Level lv = make_level<D>(level, S, H, off, gridtype, align_corners);
    const T* g = layout == LNRF_GRID_LBC ? grad + ((size_t)level * B + b) * C : grad + ((size_t)b * L + level) * C;
    float x[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        x[d] = inputs[(size_t)b * D + d];
        if (x[d] < 0.f || x[d] > 1.f) return;
    }
    uint32_t pg[D];
    float pos[D];
    cell_of<D, SMOOTH>(lv, x, align_corners, pg, pos, nullptr);
    float gv[C];
#pragma unroll
    for (int ch = 0; ch < C; ch++) gv[ch] = to_f(g[ch]);
    T* gg = grad_emb + (size_t)lv.base * C;
#pragma unroll
    for (int c = 0; c < (1 << D); c++) {
        float w = 1.f;
        uint32_t pgl[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            if (c & (1 << d)) { w *= pos[d]; pgl[d] = pg[d] + 1; }
            else { w *= 1.0f - pos[d]; pgl[d] = pg[d]; }
        }
        const uint32_t entry = grid_index<D>(lv, pgl);
        const size_t index = (size_t)entry * C;
        if constexpr (DET) {
            const size_t e = (size_t)lv.base + entry;
            const float inv_q = det_inv_q(det);
#pragma unroll
            for (int ch = 0; ch < C; ch++) {
                const float v = w * gv[ch];
                if (!isfinite(v)) det.flag[e] = 1u;
                else det_red(det.acc + e * C + ch, v, inv_q);
            }
        } else if (C % 2 == 0) {
            using T2 = typename Vec2<T>::type;
#pragma unroll
            for (int ch = 0; ch < C; ch += 2) red2(reinterpret_cast<T2*>(gg + index + ch), make_float2(w * gv[ch], w * gv[ch + 1]));
        } else {
#pragma unroll
            for (int ch = 0; ch < C; ch++) red1(gg + index + ch, w * gv[ch]);
        }
    }
}

// gridencoder.cu:343-369
template <typename T>
__global__ void __launch_bounds__(256)
k_grid_input_bwd(const T* __restrict__ grad, const T* __restrict__ dy_dx, T* __restrict__ grad_inputs, const uint32_t B,
                 const uint32_t D, const uint32_t C, const uint32_t L, const int layout) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * D) return;
    const uint32_t b = t / D, d = t - b * D;
    float result = 0.f;
    for (uint32_t l = 0; l < L; l++)
        for (uint32_t ch = 0; ch < C; ch++) {
            const float g = to_f(layout == LNRF_GRID_LBC ? grad[((size_t)l * B + b) * C + ch] : grad[((size_t)b * L + l) * C + ch]);
            result += g * to_f(dy_dx[(((size_t)b * L + l) * D + d) * C + ch]);
        }
    from_f(result, grad_inputs[t]);
}

// gridencoder.cu:506-610 (inputs arrive in the embedding dtype there; no caller exists in the reference tree)
template <typename T, int D, int C>
__global__ void __launch_bounds__(256)
k_grid_grad_tv(const T* __restrict__ inputs, const T* __restrict__ emb, T* __restrict__ grad, const float weight,
               const uint32_t B, const uint32_t L, const float S, const uint32_t H, const uint32_t gridtype,
               const bool align_corners, const GridOffsets off) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t level = blockIdx.y;
    if (b >= B) return;
    const Level lv = make_level<D>(level, S, H, off, gridtype, align_corners);
    float x[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        x[d] = to_f(inputs[(size_t)b * D + d]);
        if (x[d] < 0.f || x[d] > 1.f) return;
    }
    uint32_t pg[D];
#pragma unroll
    for (int d = 0; d < D; d++) pg[d] = (uint32_t)floorf(__fmaf_rn(x[d], lv.scale, align_corners ? 0.0f : 0.5f));
    const T* grid = emb + (size_t)lv.base * C;
    T* gg = grad + (size_t)lv.base * C;
    const size_t index = (size_t)grid_index<D>(lv, pg) * C;
    float results[C], idelta[C];
#pragma unroll
    for (int ch = 0; ch < C; ch++) results[ch] = idelta[ch] = 0.f;
    const float w = weight / (2 * D);
#pragma unroll
    for (int d = 0; d < D; d++) {
        const uint32_t cur = pg[d];
        if (cur < lv.res) {
            pg[d] = cur + 1;
            const size_t ir = (size_t)grid_index<D>(lv, pg) * C;
#pragma unroll
            for (int ch = 0; ch < C; ch++) {
                const float gv = to_f(grid[index + ch]) - to_f(grid[ir + ch]);
                results[ch] += gv; idelta[ch] += gv * gv;
            }
        }
        if (cur > 0) {
            pg[d] = cur - 1;
            const size_t il = (size_t)grid_index<D>(lv, pg) * C;
#pragma unroll
            for (int ch = 0; ch < C; ch++) {
                const float gv = to_f(grid[index + ch]) - to_f(grid[il + ch]);
                results[ch] += gv; idelta[ch] += gv * gv;
            }
        }
        pg[d] = cur;
    }
#pragma unroll
    for (int ch = 0; ch < C; ch++) red1(gg + index + ch, w * results[ch] * rsqrtf(idelta[ch] + 1e-9f));
}

// max finite |g| over the first n elements (n cut to the live 128-row tiles when B_dev is given), as float bits: non-negative floats
// order like their bit patterns, so one integer max per warp; *gmax must be zero on entry.  Order-independent.
__global__ void __launch_bounds__(256)
k_det_absmax(const float* __restrict__ g, size_t n, const uint32_t row_elems, const int* __restrict__ B_dev, uint32_t* __restrict__ gmax) {
    if (B_dev) {
        const size_t live = (size_t)div_up((uint32_t)max(*B_dev, 0), (uint32_t)kTile) * kTile * row_elems;
        n = live < n ? live : n;
    }
    float m = 0.0f;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = fabsf(__ldcs(g + i));
        if (v <= FLT_MAX) m = fmaxf(m, v);  // non-finite values set flags, they do not scale the quantum
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(gmax, __float_as_uint(m));
}

__device__ __forceinline__ void from_d(double v, __half& o) { o = __double2half(v); }
__device__ __forceinline__ void from_d(double v, float& o) { o = __double2float_rn(v); }

// out[e, ch] = RN_T(out[e, ch] + acc[e, ch] * q), or NaN for a flagged entry; the acc / flag words read are zeroed for the next call.
// Entries with nothing to add are left untouched (out + 0 is out).
template <typename T>
__global__ void __launch_bounds__(256)
k_det_finish(const DetSink d, T* __restrict__ out, const uint32_t n_entries, const uint32_t C) {
    const int qexp = det_qexp(d);
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n_entries; e += gridDim.x * blockDim.x) {
        const bool bad = d.flag[e] != 0u;
        if (bad) d.flag[e] = 0u;
        for (uint32_t ch = 0; ch < C; ch++) {
            const size_t i = (size_t)e * C + ch;
            const long long a = (long long)d.acc[i];
            if (a) d.acc[i] = 0ull;
            if (bad) from_f(__int_as_float(0x7fffffff), out[i]);
            else if (a) from_d((double)to_f(out[i]) + ldexp((double)a, qexp), out[i]);
        }
    }
}

__global__ void k_grid_level_scales(uint32_t L, float S, uint32_t H, float* __restrict__ scales) {
    const uint32_t l = threadIdx.x;
    if (l < L) scales[l] = __fmaf_rn(exp2f(__fmul_rn((float)l, S)), (float)H, -1.0f);
}

}  // namespace lnrf

using namespace lnrf;

static inline cudaStream_t S_(lnrf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// CTAs for `ntiles` tiles: at most kNumSMs * per_sm (LNRF_GRID_CAP = "fwd,bwd" blocks per SM overrides the default for A/B runs)
static uint32_t tile_grid(uint32_t ntiles, int which) {
    int per_sm[2] = {16, 16};  // one tile per CTA up to 2368 CTAs: the block scheduler balances better than a 2-vs-1 tile split (-5 us per step)
    if (const char* e = getenv("LNRF_GRID_CAP")) sscanf(e, "%d,%d", &per_sm[0], &per_sm[1]);
    const uint32_t cap = (uint32_t)kNumSMs * (uint32_t)(per_sm[which] > 0 ? per_sm[which] : 16);
    return ntiles < cap ? ntiles : cap;
}

// x-pair merged table accesses (bit 0: forward gathers, bit 1: backward reductions); LNRF_GRID_PAIR overrides for A/B measurement.
// Default 2: the merged reductions cut the L2 atomic operations of the backward by ~20 % (118.8 -> 99.7 us at 228k samples); the
// merged forward gathers measured no gain (the forward is issue-bound, not sector-bound: 50.9 us unmerged vs 53-55 us merged).
static int pair_mode() {
    const char* e = getenv("LNRF_GRID_PAIR");  // read per call: tests flip it inside one process
    return e ? atoi(e) : 2;
}

static int check_grid_args(const char* who, const int32_t* offsets_host, uint32_t D, uint32_t C, uint32_t L, uint32_t gridtype,
                           uint32_t interp, GridOffsets* off) {
    LNRF_REQUIRE(offsets_host, "%s: offsets_host is null", who);
    LNRF_REQUIRE(D == 2 || D == 3, "%s: input_dim D=%u unsupported (2 or 3)", who, D);
    LNRF_REQUIRE(C == 1 || C == 2 || C == 4 || C == 8, "GridEncoding: C must be 1, 2, 4, or 8.");  // gridencoder.cu:381
    LNRF_REQUIRE(L >= 1 && L <= (uint32_t)kMaxLevels, "%s: num_levels L=%u out of range [1,%d]", who, L, kMaxLevels);
    LNRF_REQUIRE(gridtype <= 1 && interp <= 1, "%s: gridtype/interpolation id out of range", who);
    for (uint32_t l = 0; l <= L; l++) {
        LNRF_REQUIRE(offsets_host[l] >= 0 && (l == 0 || offsets_host[l] > offsets_host[l - 1]), "%s: offsets must be increasing", who);
        off->v[l] = (uint32_t)offsets_host[l];
    }
    return LNRF_OK;
}

template <typename T, int D, int C>
static void launch_fwd_generic(bool smooth, dim3 g, cudaStream_t st, const float* in, const T* emb, T* out, uint32_t B, uint32_t L,
                               float S, uint32_t H, T* dy_dx, uint32_t gridtype, bool ac, const GridOffsets& off, int layout) {
    if (smooth) k_grid_fwd_generic<T, D, C, true><<<g, 256, 0, st>>>(in, emb, out, B, L, S, H, dy_dx, gridtype, ac, off, layout);
    else k_grid_fwd_generic<T, D, C, false><<<g, 256, 0, st>>>(in, emb, out, B, L, S, H, dy_dx, gridtype, ac, off, layout);
}
template <typename T, int D, int C>
static void launch_bwd_generic(bool smooth, dim3 g, cudaStream_t st, const T* grad, const float* in, T* ge, uint32_t B, uint32_t L,
                               float S, uint32_t H, uint32_t gridtype, bool ac, const GridOffsets& off, int layout, const DetSink* det) {
    const DetSink d = det ? *det : DetSink{};
    if (det) {
        if (smooth) k_grid_bwd_generic<T, D, C, true, true><<<g, 256, 0, st>>>(grad, in, ge, B, L, S, H, gridtype, ac, off, layout, d);
        else k_grid_bwd_generic<T, D, C, false, true><<<g, 256, 0, st>>>(grad, in, ge, B, L, S, H, gridtype, ac, off, layout, d);
    } else {
        if (smooth) k_grid_bwd_generic<T, D, C, true, false><<<g, 256, 0, st>>>(grad, in, ge, B, L, S, H, gridtype, ac, off, layout, d);
        else k_grid_bwd_generic<T, D, C, false, false><<<g, 256, 0, st>>>(grad, in, ge, B, L, S, H, gridtype, ac, off, layout, d);
    }
}

#define LNRF_DISPATCH_DC(D, C, CALL)                                                       \
    do {                                                                                   \
        if (D == 2) {                                                                      \
            if (C == 1) { CALL(2, 1); } else if (C == 2) { CALL(2, 2); } else if (C == 4) { CALL(2, 4); } else { CALL(2, 8); } \
        } else {                                                                           \
            if (C == 1) { CALL(3, 1); } else if (C == 2) { CALL(3, 2); } else if (C == 4) { CALL(3, 4); } else { CALL(3, 8); } \
        }                                                                                  \
    } while (0)

template <typename T>
static int grid_forward_t(const float* inputs, const T* emb, const GridOffsets& off, T* outputs, uint32_t B, uint32_t D, uint32_t C,
                          uint32_t L, float S, uint32_t H, T* dy_dx, uint32_t gridtype, bool ac, uint32_t interp, int layout,
                          cudaStream_t st, float in_bound = 0.0f, const int* B_dev = nullptr) {
    using T2 = typename Vec2<T>::type;
    const bool smooth = interp == 1;
    const bool hot = D == 3 && C == 2 && !dy_dx && layout == LNRF_GRID_BLC && (reinterpret_cast<uintptr_t>(emb) % sizeof(T2)) == 0 &&
                     (reinterpret_cast<uintptr_t>(outputs) % sizeof(T2)) == 0;
    if ((in_bound > 0.0f || B_dev) && !hot) {
        set_error("grid_encode_forward: in_bound / device-side B need the D=3, C=2, [B, L*C] kernel");
        return LNRF_ERR_UNSUPPORTED;
    }
    if (hot) {
        const uint32_t ntiles = div_up(B, (uint32_t)kTile);  // with B_dev: B is the capacity, the kernel re-derives both
        const uint32_t grid = tile_grid(ntiles, 0);
        const size_t smem = (size_t)kTile * (L | 1u) * sizeof(T2);
        auto kern = smooth ? (pair_mode() & 1 ? k_grid_fwd_tile<T, true, true> : k_grid_fwd_tile<T, true, false>)
                           : (pair_mode() & 1 ? k_grid_fwd_tile<T, false, true> : k_grid_fwd_tile<T, false, false>);
        launch_pdl(kern, grid, kGridThreads, smem, st, inputs, reinterpret_cast<const T2*>(emb), reinterpret_cast<T2*>(outputs), B, L, S, H, gridtype,
                                               ac, off, ntiles, in_bound, B_dev);
    } else {
        const dim3 g(div_up(B, 256u), L, 1);
#define CALL_(DD, CC) launch_fwd_generic<T, DD, CC>(smooth, g, st, inputs, emb, outputs, B, L, S, H, dy_dx, gridtype, ac, off, layout)
        LNRF_DISPATCH_DC(D, C, CALL_);
#undef CALL_
    }
    LNRF_LAUNCH_CHECK("grid_encode_forward");
    return LNRF_OK;
}

// det != nullptr: the table gradient goes to det's fixed-point sums (grad_emb is not touched; k_det_finish writes it)
template <typename T>
static int grid_backward_t(const T* grad, const float* inputs, const GridOffsets& off, T* grad_emb, uint32_t B, uint32_t D, uint32_t C,
                           uint32_t L, float S, uint32_t H, const T* dy_dx, T* grad_inputs, uint32_t gridtype, bool ac, uint32_t interp,
                           int layout, cudaStream_t st, float in_bound = 0.0f, const int* B_dev = nullptr, const DetSink* det = nullptr) {
    using T2 = typename Vec2<T>::type;
    const bool smooth = interp == 1;
    const bool hot = D == 3 && C == 2 && layout == LNRF_GRID_BLC && (det || (reinterpret_cast<uintptr_t>(grad_emb) % sizeof(T2)) == 0) &&
                     (reinterpret_cast<uintptr_t>(grad) % sizeof(T2)) == 0;
    if ((in_bound > 0.0f || B_dev) && (!hot || dy_dx)) {
        set_error("grid_encode_backward: in_bound / device-side B need the D=3, C=2, [B, L*C] kernel without input gradients");
        return LNRF_ERR_UNSUPPORTED;
    }
    if (det && det->gmax) {  // fp32 gradients: the quantum follows max |g| over the rows the backward reads (no host round trip)
        cudaError_t e = cudaMemsetAsync(const_cast<uint32_t*>(det->gmax), 0, sizeof(uint32_t), st);
        if (e != cudaSuccess) return cuda_fail(e, "grid_encode_backward(det)");
        const size_t n = (size_t)B * L * C;
        const size_t want = (n + 255) / 256, cap = (size_t)kNumSMs * 4;
        k_det_absmax<<<(uint32_t)(want < cap ? want : cap), 256, 0, st>>>(reinterpret_cast<const float*>(grad), n, L * C, B_dev,
                                                                         const_cast<uint32_t*>(det->gmax));
        LNRF_LAUNCH_CHECK("grid_encode_backward(max |g|)");
    }
    if (hot) {
        const uint32_t ntiles = div_up(B, (uint32_t)kTile);
        const uint32_t grid = tile_grid(ntiles, 1);
        const size_t smem = (size_t)kTile * (L | 1u) * sizeof(T2);
        auto kern = det ? (smooth ? k_grid_bwd_tile<T, true, false, true> : k_grid_bwd_tile<T, false, false, true>)
                  : smooth ? (pair_mode() & 2 ? k_grid_bwd_tile<T, true, true, false> : k_grid_bwd_tile<T, true, false, false>)
                           : (pair_mode() & 2 ? k_grid_bwd_tile<T, false, true, false> : k_grid_bwd_tile<T, false, false, false>);
        launch_pdl(kern, grid, kGridThreads, smem, st, reinterpret_cast<const T2*>(grad), inputs, reinterpret_cast<T2*>(grad_emb), B, L, S, H, gridtype,
                                               ac, off, ntiles, in_bound, B_dev, det ? *det : DetSink{});
    } else {
        const dim3 g(div_up(B, 256u), L, 1);
#define CALL_(DD, CC) launch_bwd_generic<T, DD, CC>(smooth, g, st, grad, inputs, grad_emb, B, L, S, H, gridtype, ac, off, layout, det)
        LNRF_DISPATCH_DC(D, C, CALL_);
#undef CALL_
    }
    LNRF_LAUNCH_CHECK("grid_encode_backward");
    if (dy_dx && grad_inputs) {
        k_grid_input_bwd<T><<<div_up(B * D, 256u), 256, 0, st>>>(grad, dy_dx, grad_inputs, B, D, C, L, layout);
        LNRF_LAUNCH_CHECK("grid_encode_backward(inputs)");
    }
    return LNRF_OK;
}

template <typename T>
static int grid_tv_t(const T* inputs, const T* emb, T* grad, const GridOffsets& off, float weight, uint32_t B, uint32_t D, uint32_t C,
                     uint32_t L, float S, uint32_t H, uint32_t gridtype, bool ac, cudaStream_t st) {
    const dim3 g(div_up(B, 256u), L, 1);
#define CALL_(DD, CC) k_grid_grad_tv<T, DD, CC><<<g, 256, 0, st>>>(inputs, emb, grad, weight, B, L, S, H, gridtype, ac, off)
    LNRF_DISPATCH_DC(D, C, CALL_);
#undef CALL_
    LNRF_LAUNCH_CHECK("grad_total_variation");
    return LNRF_OK;
}

extern "C" {

int lnrf_grid_encode_forward(const float* inputs, const void* embeddings, const int32_t* offsets_host, void* outputs, uint32_t B,
                             uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, void* dy_dx, uint32_t gridtype,
                             int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_grid_layout out_layout,
                             lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_forward", offsets_host, D, C, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(inputs && embeddings && outputs, "grid_encode_forward: null pointer");
    LNRF_REQUIRE((uint64_t)B * L * C < (1ull << 40), "grid_encode_forward: batch too large");
    if (emb_dtype == LNRF_F16)
        return grid_forward_t<__half>(inputs, (const __half*)embeddings, off, (__half*)outputs, B, D, C, L, S, H, (__half*)dy_dx, gridtype,
                                      align_corners != 0, interp, (int)out_layout, S_(stream));
    if (emb_dtype == LNRF_F32)
        return grid_forward_t<float>(inputs, (const float*)embeddings, off, (float*)outputs, B, D, C, L, S, H, (float*)dy_dx, gridtype,
                                     align_corners != 0, interp, (int)out_layout, S_(stream));
    set_error("grid_encode_forward: unsupported embedding dtype %d", (int)emb_dtype);
    return LNRF_ERR_UNSUPPORTED;
}

int lnrf_grid_encode_forward_world(const float* inputs_world, float bound, const void* embeddings, const int32_t* offsets_host,
                                   void* outputs, uint32_t B, const int32_t* B_dev, uint32_t L, float S, uint32_t H, uint32_t gridtype,
                                   int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_forward_world", offsets_host, 3, 2, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(inputs_world && embeddings && outputs && bound > 0.0f, "grid_encode_forward_world: null pointer / bound <= 0");
    if (emb_dtype == LNRF_F16)
        return grid_forward_t<__half>(inputs_world, (const __half*)embeddings, off, (__half*)outputs, B, 3, 2, L, S, H, nullptr, gridtype,
                                      align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev);
    if (emb_dtype == LNRF_F32)
        return grid_forward_t<float>(inputs_world, (const float*)embeddings, off, (float*)outputs, B, 3, 2, L, S, H, nullptr, gridtype,
                                     align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev);
    set_error("grid_encode_forward_world: unsupported embedding dtype %d", (int)emb_dtype);
    return LNRF_ERR_UNSUPPORTED;
}

int lnrf_grid_encode_backward_world(const void* grad, const float* inputs_world, float bound, const int32_t* offsets_host,
                                    void* grad_embeddings, uint32_t B, const int32_t* B_dev, uint32_t L, float S, uint32_t H,
                                    uint32_t gridtype, int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_backward_world", offsets_host, 3, 2, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(grad && inputs_world && grad_embeddings && bound > 0.0f, "grid_encode_backward_world: null pointer / bound <= 0");
    if (emb_dtype == LNRF_F16)
        return grid_backward_t<__half>((const __half*)grad, inputs_world, off, (__half*)grad_embeddings, B, 3, 2, L, S, H, nullptr, nullptr,
                                       gridtype, align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev);
    if (emb_dtype == LNRF_F32)
        return grid_backward_t<float>((const float*)grad, inputs_world, off, (float*)grad_embeddings, B, 3, 2, L, S, H, nullptr, nullptr,
                                      gridtype, align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev);
    set_error("grid_encode_backward_world: unsupported embedding dtype %d", (int)emb_dtype);
    return LNRF_ERR_UNSUPPORTED;
}

int lnrf_grid_encode_backward(const void* grad, const float* inputs, const void* embeddings, const int32_t* offsets_host,
                              void* grad_embeddings, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H,
                              const void* dy_dx, void* grad_inputs, uint32_t gridtype, int align_corners, uint32_t interp,
                              lnrf_dtype emb_dtype, lnrf_grid_layout grad_layout, lnrf_stream_t stream) {
    (void)embeddings;  // the reference passes it but never reads it in the backward kernels either
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_backward", offsets_host, D, C, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(grad && inputs && grad_embeddings, "grid_encode_backward: null pointer");
    if (emb_dtype == LNRF_F16)
        return grid_backward_t<__half>((const __half*)grad, inputs, off, (__half*)grad_embeddings, B, D, C, L, S, H, (const __half*)dy_dx,
                                       (__half*)grad_inputs, gridtype, align_corners != 0, interp, (int)grad_layout, S_(stream));
    if (emb_dtype == LNRF_F32)
        return grid_backward_t<float>((const float*)grad, inputs, off, (float*)grad_embeddings, B, D, C, L, S, H, (const float*)dy_dx,
                                      (float*)grad_inputs, gridtype, align_corners != 0, interp, (int)grad_layout, S_(stream));
    set_error("grid_encode_backward: unsupported embedding dtype %d", (int)emb_dtype);
    return LNRF_ERR_UNSUPPORTED;
}

// ---- deterministic table gradient (DetSink) ----
static int det_sink(const char* who, void* acc, void* flags, void* gmax, uint32_t B, lnrf_dtype dt, DetSink* d) {
    LNRF_REQUIRE(acc && flags, "%s: acc / flags is null", who);
    LNRF_REQUIRE(dt == LNRF_F16 || dt == LNRF_F32, "%s: unsupported dtype %d", who, (int)dt);
    LNRF_REQUIRE(dt == LNRF_F16 || gmax, "%s: fp32 gradients need the gmax word", who);
    LNRF_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "%s: acc must be 16-byte aligned", who);
    LNRF_REQUIRE(B >= 1, "%s: B must be >= 1", who);
    int lb = 0;
    while ((1ull << lb) < (unsigned long long)B) lb++;
    *d = DetSink{(unsigned long long*)acc, (uint32_t*)flags, dt == LNRF_F32 ? (const uint32_t*)gmax : nullptr, lb};
    return LNRF_OK;
}

int lnrf_grid_encode_backward_det(const void* grad, const float* inputs, const int32_t* offsets_host, void* acc, void* flags, void* gmax,
                                  uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, const void* dy_dx, void* grad_inputs,
                                  uint32_t gridtype, int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_grid_layout grad_layout,
                                  lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_backward_det", offsets_host, D, C, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(grad && inputs, "grid_encode_backward_det: null pointer");
    LNRF_REQUIRE((uint64_t)B * L * C < (1ull << 40), "grid_encode_backward_det: batch too large");
    DetSink d;
    if (int e = det_sink("grid_encode_backward_det", acc, flags, gmax, B, emb_dtype, &d)) return e;
    if (emb_dtype == LNRF_F16)
        return grid_backward_t<__half>((const __half*)grad, inputs, off, nullptr, B, D, C, L, S, H, (const __half*)dy_dx, (__half*)grad_inputs,
                                       gridtype, align_corners != 0, interp, (int)grad_layout, S_(stream), 0.0f, nullptr, &d);
    return grid_backward_t<float>((const float*)grad, inputs, off, nullptr, B, D, C, L, S, H, (const float*)dy_dx, (float*)grad_inputs,
                                  gridtype, align_corners != 0, interp, (int)grad_layout, S_(stream), 0.0f, nullptr, &d);
}

int lnrf_grid_encode_backward_world_det(const void* grad, const float* inputs_world, float bound, const int32_t* offsets_host, void* acc,
                                        void* flags, void* gmax, uint32_t B, const int32_t* B_dev, uint32_t L, float S, uint32_t H,
                                        uint32_t gridtype, int align_corners, uint32_t interp, lnrf_dtype emb_dtype, lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grid_encode_backward_world_det", offsets_host, 3, 2, L, gridtype, interp, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(grad && inputs_world && bound > 0.0f, "grid_encode_backward_world_det: null pointer / bound <= 0");
    DetSink d;
    if (int e = det_sink("grid_encode_backward_world_det", acc, flags, gmax, B, emb_dtype, &d)) return e;
    if (emb_dtype == LNRF_F16)
        return grid_backward_t<__half>((const __half*)grad, inputs_world, off, nullptr, B, 3, 2, L, S, H, nullptr, nullptr, gridtype,
                                       align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev, &d);
    return grid_backward_t<float>((const float*)grad, inputs_world, off, nullptr, B, 3, 2, L, S, H, nullptr, nullptr, gridtype,
                                  align_corners != 0, interp, (int)LNRF_GRID_BLC, S_(stream), bound, B_dev, &d);
}

int lnrf_grid_det_finish(void* acc, void* flags, const void* gmax, uint32_t B, void* grad_embeddings, uint32_t n_entries, uint32_t C,
                         lnrf_dtype emb_dtype, lnrf_stream_t stream) {
    LNRF_REQUIRE(C == 1 || C == 2 || C == 4 || C == 8, "grid_det_finish: C must be 1, 2, 4, or 8");
    LNRF_REQUIRE(grad_embeddings || n_entries == 0, "grid_det_finish: grad_embeddings is null");
    DetSink d;
    if (int e = det_sink("grid_det_finish", acc, flags, const_cast<void*>(gmax), B, emb_dtype, &d)) return e;
    if (n_entries == 0) return LNRF_OK;
    const uint32_t want = div_up(n_entries, 256u), cap = (uint32_t)kNumSMs * 16u;
    const uint32_t g = want < cap ? want : cap;
    if (emb_dtype == LNRF_F16) k_det_finish<__half><<<g, 256, 0, S_(stream)>>>(d, (__half*)grad_embeddings, n_entries, C);
    else k_det_finish<float><<<g, 256, 0, S_(stream)>>>(d, (float*)grad_embeddings, n_entries, C);
    LNRF_LAUNCH_CHECK("grid_det_finish");
    return LNRF_OK;
}

int lnrf_grad_total_variation(const void* inputs, const void* embeddings, void* grad, const int32_t* offsets_host, float weight,
                              uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, uint32_t gridtype,
                              int align_corners, lnrf_dtype emb_dtype, lnrf_stream_t stream) {
    GridOffsets off;
    if (int e = check_grid_args("grad_total_variation", offsets_host, D, C, L, gridtype, 0, &off)) return e;
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(inputs && embeddings && grad, "grad_total_variation: null pointer");
    if (emb_dtype == LNRF_F16)
        return grid_tv_t<__half>((const __half*)inputs, (const __half*)embeddings, (__half*)grad, off, weight, B, D, C, L, S, H, gridtype,
                                 align_corners != 0, S_(stream));
    if (emb_dtype == LNRF_F32)
        return grid_tv_t<float>((const float*)inputs, (const float*)embeddings, (float*)grad, off, weight, B, D, C, L, S, H, gridtype,
                                align_corners != 0, S_(stream));
    set_error("grad_total_variation: unsupported embedding dtype %d", (int)emb_dtype);
    return LNRF_ERR_UNSUPPORTED;
}

int lnrf_grid_level_scales(uint32_t L, float S, uint32_t H, float* scales, lnrf_stream_t stream) {
    LNRF_REQUIRE(L >= 1 && L <= (uint32_t)kMaxLevels && scales, "grid_level_scales: bad arguments");
    k_grid_level_scales<<<1, 32, 0, S_(stream)>>>(L, S, H, scales);
    LNRF_LAUNCH_CHECK("grid_level_scales");
    return LNRF_OK;
}

}  // extern "C"
