// ffmlp.cu -- fully fused 64-wide MLP on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a only.
//
// Replaces ffmlp/src/ffmlp.cu of the reference: kernel_mlp_fused (:331-407, wmma fp16-accumulate),
// kernel_mlp_fused_backward (:410-518) and the CUTLASS 2.8 split-K weight-gradient GEMMs (:783-887).
//
// Design (DESIGN.md section 5):
//   * a CTA of 128 threads owns tiles of 128 batch rows = the native tcgen05.mma M.  Every operand tile lives in
//     shared memory as 128-byte rows (64 fp16) in the SWIZZLE_128B canonical layout, so the SAME tile can be read
//     as a K-major operand (forward / dgrad: K = feature axis) and as an MN-major operand (wgrad: K = batch rows).
//   * all weight matrices stay resident in shared memory for the life of the CTA (forward: W_m as [N, K] K-major;
//     backward: W_m^T), accumulators live in TMEM (fp32), one elected thread issues the MMAs and signals an
//     mbarrier through tcgen05.commit, the 128 threads read their accumulator row back with tcgen05.ld
//     (thread r <-> TMEM lane r), apply the activation and write the fp16 row of the next layer's A operand.
//   * backward: dL/dhidden is chained on chip the same way (ReLU mask from the saved activations), and every
//     layer's weight gradient is ONE TMEM accumulator that is summed over all tiles the CTA processes
//     (dW = sum over tiles of X_tile^T . G_tile, M = feature, N = feature, K = 128 rows), flushed once per CTA
//     with coalesced fp32 reductions into a scratch vector -- no split-K workspace, no side streams.
//   Accumulation is fp32 everywhere (the reference accumulates in fp16); activations are rounded to fp16 exactly
//   where the reference stores them (forward_buffer, backward chain, outputs).
#include "mlp_core.cuh"
#include <string.h>

namespace lnrf {

// =========================================================================================================
// forward / inference
// =========================================================================================================
// shared memory: W_0..W_{NL-1} (8 KB each), W_NL (out_dim rows), X double buffer (next tile prefetched with
// cp.async while this one is computed), two activation tiles (ping-pong), mbarrier + TMEM slot
template <bool TRAIN, int ACT>
__global__ void __launch_bounds__(128)
k_ffmlp_fwd(const __half* __restrict__ inputs, const __half* __restrict__ weights, __half* __restrict__ fwd_buf,
            __half* __restrict__ outputs, const uint32_t B, const MlpShape sh, const uint32_t ntiles) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_raw + (((smem_u32(smem_raw) + 1023u) & ~1023u) - smem_u32(smem_raw));
    const uint32_t NL = sh.n_layers, in_dim = sh.in_dim, out_dim = sh.out_dim;
    uint8_t* sW = sm;
    uint8_t* sX = sW + NL * kWBytes + ((out_dim * 128u + 1023u) & ~1023u);
    uint8_t* sA = sX + 2 * kTileBytes;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sA + 2 * kTileBytes);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(mbar + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t row = tid;  // this thread's row of the tile == its TMEM lane

    // everything the first tile needs is requested at once; TMEM allocation overlaps the copies
    load_rows_async(smem_u32(sW), weights, 64, in_dim, tid);
    for (uint32_t m = 1; m < NL; m++) load_rows_async(smem_u32(sW + m * kWBytes), weights + 64 * in_dim + (m - 1) * 4096, 64, 64, tid);
    load_rows_async(smem_u32(sW + NL * kWBytes), weights + 64 * in_dim + (NL - 1) * 4096, out_dim, 64, tid);
    load_rows_async(smem_u32(sX), inputs + (size_t)blockIdx.x * kRows * in_dim, kRows, in_dim, tid);
    cp_async_commit();
    if (warp == 0) tmem_alloc(tslot, 64);
    if (tid == 32) { mbar_init(mbar, 1); fence_mbar_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0, it = 0;

    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
        const size_t r0 = (size_t)tile * kRows;
        uint8_t* X = sX + (it & 1u) * kTileBytes;
        cp_async_wait_all();
        fence_proxy_async();
        __syncthreads();  // X (and on the first pass the weights) landed; the previous tile is completely done
        if (tile + gridDim.x < ntiles) {
            load_rows_async(smem_u32(sX + ((it + 1u) & 1u) * kTileBytes), inputs + (size_t)(tile + gridDim.x) * kRows * in_dim, kRows, in_dim, tid);
            cp_async_commit();
        }
        for (uint32_t m = 0; m <= NL; m++) {
            uint8_t* cur = m == 0 ? X : sA + ((m - 1u) & 1u) * kTileBytes;
            uint8_t* nxt = sA + (m & 1u) * kTileBytes;
            if (warp == 0) {  // uniformly; one elected lane issues (see umma_chain in mlp_core.cuh)
                tc_fence_after();
                const uint32_t K = m == 0 ? in_dim : 64u, N = m == NL ? out_dim : 64u;
                const uint32_t idesc = make_idesc(128, N, false, false);
                const uint64_t a = desc_sw128(smem_u32(cur), 16), b = desc_sw128(smem_u32(sW + m * kWBytes), 16);
                if (elect_one()) {
                    umma_chain_k(K / 16, tmem, a, b, idesc);
                    umma_commit(mbar);
                }
                __syncwarp();
            }
            if (TRAIN && m > 0) {  // save H_{m-1} (== cur) while the tensor core works: coalesced 16-byte pieces
                uint4* dst = reinterpret_cast<uint4*>(fwd_buf + ((size_t)(m - 1) * B + r0) * 64);
#pragma unroll
                for (uint32_t i = 0; i < 8; i++) {
                    const uint32_t c = tid + i * 128;
                    __stcs(dst + c, *reinterpret_cast<const uint4*>(cur + sw128(c >> 3, c & 7u)));
                }
            }
            mbar_wait(mbar, phase);
            phase ^= 1u;
            tc_fence_after();
            if (m < NL) {
                uint32_t r[64];
                tmem_ld32_nowait(taddr, r);
                tmem_ld32_nowait(taddr + 32, r + 32);
                tmem_wait_ld();
#pragma unroll
                for (uint32_t q = 0; q < 8; q++) {
                    float v[8];
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const float a = __uint_as_float(r[q * 8 + i]);
                        v[i] = ACT == 0 ? fmaxf(a, 0.0f) : act_fwd(sh.act, a);
                    }
                    *reinterpret_cast<uint4*>(nxt + sw128(row, q)) = pack8(v);
                }
                tc_fence_before();
                fence_proxy_async();
                __syncthreads();
            } else {
                __half* o = outputs + (r0 + row) * out_dim;
                for (uint32_t q = 0; q < out_dim / 16; q++) {
                    float v[16];
                    tmem_ld16(taddr + q * 16, v);
#pragma unroll
                    if (sh.out_act != 6u) {
#pragma unroll
                        for (int i = 0; i < 16; i++) v[i] = act_fwd(sh.out_act, v[i]);
                    }
                    __stcs(reinterpret_cast<uint4*>(o + q * 16), pack8(v));
                    __stcs(reinterpret_cast<uint4*>(o + q * 16) + 1, pack8(v + 8));
                }
                tc_fence_before();
            }
        }
    }
    cp_async_wait_all();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 64);
}

// =========================================================================================================
// backward: dL/dhidden chain + all weight gradients + optional dL/dinput, one kernel
// =========================================================================================================
__device__ __host__ inline uint32_t bwd_tmem_cols(uint32_t in_dim, uint32_t out_dim, uint32_t NL) {
    const uint32_t need = 64 + out_dim + 64 * (NL - 1) + in_dim;
    uint32_t c = 32;
    while (c < need) c <<= 1;
    return c;
}

// shared memory: W_m^T tiles (m = 1..NL, then W_0^T), the G ping-pong pair, and NBUF input sets
// {X, H_0..H_{NL-1}, dY}: with NBUF = 2 the next tile's 60-76 KB are prefetched (cp.async) during this tile's chain.
// Every tile that serves as an M=128 MN-major A operand (H_l, G_0) is followed by another tile: the "second atom"
// the MMA reads for D rows 64..127, which are never used.
//
// GLUE = true is the colour net of NeRFNetwork.forward (nerf/network_ff.py:51-79) with the elementwise glue of its backward
// fused in: dL/dY is built on the fly from dL/drgb and the saved sigmoid outputs (fp16 sigmoid backward), and instead of
// dL/dinput [B,32] the kernel writes dL/dh [B,16] of the sigma net: column 0 = dL/dsigma * density_scale * exp(clamp(h0,
// -15, 15)) (trunc_exp backward, activation.py:13-16), columns 1..15 = dL/dgeo_feat = dL/dinput[:, 16:31].
template <int ACT, bool GLUE>
__global__ void __launch_bounds__(128)
k_ffmlp_bwd(const __half* __restrict__ grad, const __half* __restrict__ inputs, const __half* __restrict__ weights,
            const __half* __restrict__ fwd_buf, __half* __restrict__ grad_inputs, float* __restrict__ wgrad, const uint32_t B,
            const MlpShape sh, const uint32_t ntiles, const int calc_grad_inputs, const uint32_t nbuf, const BwdGlue glue) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_raw + (((smem_u32(smem_raw) + 1023u) & ~1023u) - smem_u32(smem_raw));
    const uint32_t NL = sh.n_layers, in_dim = sh.in_dim, out_dim = sh.out_dim;
    uint8_t* sWT = sm;                         // index m-1 for m = 1..NL: [64 rows = input feature][K = n_m]
    uint8_t* sWT0 = sWT + NL * kWBytes;        // W_0^T: [in rows][K = 64]
    uint8_t* sG = sWT0 + kWBytes;              // G_m (m < NL) lives in sG[m & 1]
    uint8_t* sIN = sG + 2 * kTileBytes;
    const uint32_t in_bytes = (NL + 2) * kTileBytes;  // X, H_0..H_{NL-1}, dY
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sIN + nbuf * in_bytes);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(mbar + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t row = tid;
    const uint32_t ncols = bwd_tmem_cols(in_dim, out_dim, NL);

    auto load_inputs = [&](uint32_t tile, uint32_t buf) {
        const size_t r0 = (size_t)tile * kRows;
        const uint32_t base = smem_u32(sIN + buf * in_bytes);
        load_rows_async(base, inputs + r0 * in_dim, kRows, in_dim, tid);
        for (uint32_t l = 0; l < NL; l++) load_rows_async(base + (1 + l) * kTileBytes, fwd_buf + ((size_t)l * B + r0) * 64, kRows, 64, tid);
        if (!GLUE) load_rows_async(base + (1 + NL) * kTileBytes, grad + r0 * out_dim, kRows, out_dim, tid);
    };
    // GLUE: this thread's row of dL/dY (16 columns, 3 real) = fp16 sigmoid backward of dL/drgb, written straight into the tile
    auto glue_dy = [&](uint32_t tile, uint32_t buf) {
        const size_t r = (size_t)tile * kRows + row;
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const float g = __half2float(__float2half_rn(__ldcs(glue.grad_rgb + r * 3 + c)));  // the grad of the .float() cast
            const float sgm = __ldg(glue.rgb + r * 3 + c);
            v[c] = g * ((1.0f - sgm) * sgm);
        }
        uint8_t* t = sIN + buf * in_bytes + (1 + NL) * kTileBytes;
        *reinterpret_cast<uint4*>(t + sw128(row, 0)) = pack8(v);
        *reinterpret_cast<uint4*>(t + sw128(row, 1)) = make_uint4(0u, 0u, 0u, 0u);
    };

    // stage the raw weights in the (still unused) first input set, request the first tile, then transpose in shared memory
    const uint32_t nparams = 64 * (in_dim + 64 * (NL - 1) + out_dim);
    uint8_t* stage = sG;  // 32 KB >= 2 * nparams for every supported shape (<= 22.5 KB)
    copy_raw_async(smem_u32(stage), weights, nparams * 2 / 16, tid);
    cp_async_commit();
    load_inputs(blockIdx.x, 0);
    cp_async_commit();
    if (GLUE) glue_dy(blockIdx.x, 0);
    if (warp == 0) tmem_alloc(tslot, ncols);
    if (tid == 32) { mbar_init(mbar, 1); fence_mbar_init(); }
    asm volatile("cp.async.wait_group 1;" ::: "memory");  // the weights (first group) have landed
    __syncthreads();
    {
        const __half* w = reinterpret_cast<const __half*>(stage);
        transpose_to_tile(sWT + (NL - 1) * kWBytes, w + 64 * in_dim + (NL - 1) * 4096, out_dim, 64, tid);  // W_NL [out,64] -> [64][out]
        for (uint32_t m = 1; m < NL; m++) transpose_to_tile(sWT + (m - 1) * kWBytes, w + 64 * in_dim + (m - 1) * 4096, 64, 64, tid);
        if (calc_grad_inputs) transpose_to_tile(sWT0, w, 64, in_dim, tid);  // W_0 [64,in] -> [in][64]
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    // TMEM columns: [0,64) dgrad accumulator; then dW_NL (out_dim), dW_{NL-1}..dW_1 (64 each), dW_0 (in_dim)
    auto acc_col = [&](uint32_t m) -> uint32_t {
        if (m == NL) return 64u;
        if (m == 0) return 64u + out_dim + 64u * (NL - 1);
        return 64u + out_dim + 64u * (NL - 1 - m);
    };
    uint32_t phase = 0, iter = 0;

    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, iter++) {
        const size_t r0 = (size_t)tile * kRows;
        const uint32_t buf = nbuf == 2 ? (iter & 1u) : 0u;
        uint8_t* sX = sIN + buf * in_bytes;
        uint8_t* sH = sX + kTileBytes;
        uint8_t* sDY = sH + NL * kTileBytes;
        cp_async_wait_all();
        fence_proxy_async();
        __syncthreads();
        if (nbuf == 2 && tile + gridDim.x < ntiles) {
            load_inputs(tile + gridDim.x, buf ^ 1u);
            cp_async_commit();
            if (GLUE) glue_dy(tile + gridDim.x, buf ^ 1u);  // made visible by the fences + barriers of this tile's chain
        }
        float glue_gs = 0.f, glue_h0 = 0.f;
        if (GLUE) {
            glue_gs = __ldcs(glue.grad_sigma + r0 + row);
            glue_h0 = __half2float(glue.h0[r0 + row]);
        }
        for (uint32_t m = NL; m >= 1; m--) {
            uint8_t* Gm = m == NL ? sDY : sG + (m & 1u) * kTileBytes;
            uint8_t* Gp = sG + ((m - 1u) & 1u) * kTileBytes;
            uint8_t* Hp = sH + (m - 1) * kTileBytes;  // H_{m-1}: activation mask AND the input of matmul m
            const uint32_t n_m = m == NL ? out_dim : 64u;
            if (tid == 0) {
                tc_fence_after();
                // dgrad: D[128,64] = G_m[128,n_m] . W_m[n_m,64]
                const uint64_t a = desc_sw128(smem_u32(Gm), 16), b = desc_sw128(smem_u32(sWT + (m - 1) * kWBytes), 16);
                const uint32_t idesc = make_idesc(128, 64, false, false);
                for (uint32_t k = 0; k < n_m / 16; k++) umma_f16(tmem, a + 2 * k, b + 2 * k, idesc, k > 0);
                umma_commit(mbar);
                // wgrad: acc_m[feature i][neuron j] += H_{m-1}^T . G_m  (K = the 128 rows, 16 per MMA = 2048 B)
                const uint64_t wa = desc_sw128(smem_u32(Hp), kTileBytes), wb = desc_sw128(smem_u32(Gm), kTileBytes);
                const uint32_t widesc = make_idesc(128, n_m, true, true);
                for (uint32_t k = 0; k < 8; k++) umma_f16(tmem + acc_col(m), wa + 128 * k, wb + 128 * k, widesc, (iter | k) > 0);
            }
            // the saved activations of this row, fetched while the tensor core works
            uint4 hrow[8];
#pragma unroll
            for (uint32_t q = 0; q < 8; q++) hrow[q] = *reinterpret_cast<const uint4*>(Hp + sw128(row, q));
            mbar_wait(mbar, phase);
            phase ^= 1u;
            tc_fence_after();
            uint32_t r[64];
            tmem_ld32_nowait(taddr, r);
            tmem_ld32_nowait(taddr + 32, r + 32);
            tmem_wait_ld();
#pragma unroll
            for (uint32_t q = 0; q < 8; q++) {
                float v[8], h[8];
                unpack8(hrow[q], h);
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const float gacc = __uint_as_float(r[q * 8 + i]);
                    v[i] = ACT == 0 ? (h[i] > 0.0f ? gacc : 0.0f) : act_bwd(sh.act, gacc, h[i]);
                }
                *reinterpret_cast<uint4*>(Gp + sw128(row, q)) = pack8(v);
            }
            tc_fence_before();
            fence_proxy_async();
            __syncthreads();
        }
        // input layer: dW_0[neuron j][feature i] += G_0^T . X ; optionally dX = G_0 . W_0
        if (tid == 0) {
            tc_fence_after();
            if (calc_grad_inputs) {
                const uint64_t a = desc_sw128(smem_u32(sG), 16), b = desc_sw128(smem_u32(sWT0), 16);
                const uint32_t idesc = make_idesc(128, in_dim, false, false);
                for (uint32_t k = 0; k < 4; k++) umma_f16(tmem, a + 2 * k, b + 2 * k, idesc, k > 0);
            }
            const uint64_t wa = desc_sw128(smem_u32(sG), kTileBytes), wb = desc_sw128(smem_u32(sX), kTileBytes);
            const uint32_t widesc = make_idesc(128, in_dim, true, true);
            for (uint32_t k = 0; k < 8; k++) umma_f16(tmem + acc_col(0), wa + 128 * k, wb + 128 * k, widesc, (iter | k) > 0);
            umma_commit(mbar);
        }
        mbar_wait(mbar, phase);  // every MMA of this tile has finished: its shared-memory tiles may be overwritten
        phase ^= 1u;
        tc_fence_after();
        if (GLUE) {
            float v[16], o[16];
            tmem_ld16(taddr + 16, v);  // dL/dinput[:, 16:32] = dL/dgeo_feat (15) and the zero-pad column
            o[0] = glue_gs * glue.density_scale * expf(fminf(fmaxf(glue_h0, -15.0f), 15.0f));
#pragma unroll
            for (int i = 1; i < 16; i++) o[i] = v[i - 1];
            __half* d = glue.dh + (r0 + row) * 16;
            *reinterpret_cast<uint4*>(d) = pack8(o);
            *(reinterpret_cast<uint4*>(d) + 1) = pack8(o + 8);
        } else if (calc_grad_inputs) {
            __half* gi = grad_inputs + (r0 + row) * in_dim;
            for (uint32_t q = 0; q < in_dim / 16; q++) {
                float v[16];
                tmem_ld16(taddr + q * 16, v);
                __stcs(reinterpret_cast<uint4*>(gi + q * 16), pack8(v));
                __stcs(reinterpret_cast<uint4*>(gi + q * 16) + 1, pack8(v + 8));
            }
        }
        tc_fence_before();
        if (nbuf == 1 && tile + gridDim.x < ntiles) {
            __syncthreads();
            load_inputs(tile + gridDim.x, 0);
            cp_async_commit();
            if (GLUE) glue_dy(tile + gridDim.x, 0);
        }
    }

    // ---- flush the weight-gradient accumulators (rows 0..63 are real; lanes 64..127 hold the ignored atom) ----
    cp_async_wait_all();
    __syncthreads();
    tc_fence_after();
    if (iter > 0 && warp < 2) {
        const uint32_t w_first = 64 * in_dim;
        for (uint32_t m = 1; m <= NL; m++) {  // acc_m[i][j] = dW_m[j][i]; lane = i -> coalesced over i
            const uint32_t n_m = m == NL ? out_dim : 64u;
            float* dst = wgrad + w_first + (m - 1) * 4096;
            for (uint32_t q = 0; q < n_m / 16; q++) {
                float v[16];
                tmem_ld16(taddr + acc_col(m) + q * 16, v);
#pragma unroll
                for (int j = 0; j < 16; j++) atomicAdd(dst + (q * 16 + j) * 64 + row, v[j]);
            }
        }
        for (uint32_t q = 0; q < in_dim / 16; q++) {  // acc_0[j][i] = dW_0[j][i]; lane = j
            float v[16];
            tmem_ld16(taddr + acc_col(0) + q * 16, v);
#pragma unroll
            for (int i = 0; i < 16; i++) atomicAdd(wgrad + row * in_dim + q * 16 + i, v[i]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, ncols);
}

// =========================================================================================================
// backward, ReLU nets: two tiles in flight per CTA, dL/dhidden chained IN PLACE through the saved activations
// =========================================================================================================
// ncu (profiles/r1c) showed the kernel above at 6 % warps active / 10 % tensor pipe: one 128-thread CTA per SM (TMEM- and
// shared-memory-bound) walking a serial chain.  This variant runs kBwdGroups = 2 warpgroups per CTA, each with its own tile
// set {X, H_0..H_{NL-1}, dY}, 64 dgrad columns + its own weight-gradient accumulators in TMEM, mbarrier and named barrier,
// sharing the transposed weights.  G_{m-1} = dgrad .* relu'(H_{m-1}) is written over H_{m-1} itself (dead once its mask is
// applied and matmul m's weight gradient has consumed it -- both MMAs are covered by the commit the epilogue waits on), so
// a tile set is NL+2 tiles and two sets fit; one group's cp.async loads overlap the other group's chain.
constexpr uint32_t kBwdGroups = 2;

__device__ __host__ inline uint32_t bwd2_group_cols(uint32_t in_dim, uint32_t out_dim, uint32_t NL) {
    return 64 + out_dim + 64 * (NL - 1) + in_dim;
}

template <bool GLUE>
__global__ void __launch_bounds__(128 * kBwdGroups, 1)
k_mlp_bwd2(const __half* __restrict__ grad, const __half* __restrict__ inputs, const __half* __restrict__ weights,
           const __half* __restrict__ fwd_buf, __half* __restrict__ grad_inputs, float* __restrict__ wgrad, const uint32_t B,
           const MlpShape sh, const uint32_t ntiles, const int calc_grad_inputs, const BwdGlue glue) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = smem_raw + (((smem_u32(smem_raw) + 1023u) & ~1023u) - smem_u32(smem_raw));
    const uint32_t NL = sh.n_layers, in_dim = sh.in_dim, out_dim = sh.out_dim;
    uint8_t* sWT = sm;                         // index m-1 for m = 1..NL: [64 rows = input feature][K = n_m]
    uint8_t* sWT0 = sWT + NL * kWBytes;        // W_0^T: [in rows][K = 64]
    uint8_t* sSets = sWT0 + kWBytes;
    const uint32_t set_bytes = (NL + 2) * kTileBytes;  // X, H_0..H_{NL-1}, dY  (+ one spare tile after the last set: the
    uint64_t* mbars = reinterpret_cast<uint64_t*>(sSets + kBwdGroups * set_bytes + kTileBytes);  //  "second atom" of dY)
    uint32_t* tslot = reinterpret_cast<uint32_t*>(mbars + kBwdGroups);
    const uint32_t tid = threadIdx.x, warp = tid >> 5, g = tid >> 7, gt = tid & 127u;
    const uint32_t row = gt;
    uint8_t* sX = sSets + g * set_bytes;
    uint8_t* sH = sX + kTileBytes;
    uint8_t* sDY = sH + NL * kTileBytes;
    uint64_t* mbar = mbars + g;
    const uint32_t gcols = bwd2_group_cols(in_dim, out_dim, NL);
    const uint32_t stride = gridDim.x * kBwdGroups, first = blockIdx.x * kBwdGroups + g;

    // ---- streaming loads: the tile a chain step frees is exactly the one the NEXT tile of this group needs at the same step,
    // so its rows are requested (cp.async, one commit group per step, issued even when empty) as soon as the step's MMAs have
    // completed.  Groups complete in order and NL+1 are issued per tile, so "at most NL-1 groups pending" at the end of a step
    // is precisely "what the next step reads has landed"; load latency never sits on the chain.
    auto wait_loads = [&]() {
        switch (NL) {
            case 2: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
            case 3: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
            case 4: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
            default: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
        }
    };
    // unit m of a tile: m == NL -> dY; 1 <= m < NL -> H_m; m == 0 -> H_0 and X
    auto load_unit = [&](uint32_t tile, uint32_t m) {
        if (tile < ntiles) {
            const size_t r0 = (size_t)tile * kRows;
            if (m == NL) {
                if (!GLUE) load_rows_async_n(smem_u32(sDY), grad + r0 * out_dim, kRows, out_dim, gt, 128);
            } else {
                load_rows_async_n(smem_u32(sH + m * kTileBytes), fwd_buf + ((size_t)m * B + r0) * 64, kRows, 64, gt, 128);
                if (m == 0) load_rows_async_n(smem_u32(sX), inputs + r0 * in_dim, kRows, in_dim, gt, 128);
            }
        }
        cp_async_commit();
    };
    // GLUE: this row of dL/dY (16 columns, 3 real) = fp16 sigmoid backward of dL/drgb, as three fp16 values in two registers
    auto glue_dy_regs = [&](uint32_t tile, uint32_t* pk) {
        pk[0] = pk[1] = 0u;
        if (tile < ntiles) {
            const size_t r = (size_t)tile * kRows + row;
            float v[3];
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const float gg = __half2float(__float2half_rn(__ldcs(glue.grad_rgb + r * 3 + c)));  // the grad of the .float() cast
                const float sgm = __ldg(glue.rgb + r * 3 + c);
                v[c] = gg * (1.0f - sgm) * sgm;
            }
            pk[0] = pack_h2(v[0], v[1]);
            pk[1] = pack_h2(v[2], 0.0f);
        }
    };
    auto glue_dy_store = [&](const uint32_t* pk) {
        *reinterpret_cast<uint4*>(sDY + sw128(row, 0)) = make_uint4(pk[0], pk[1], 0u, 0u);
        *reinterpret_cast<uint4*>(sDY + sw128(row, 1)) = make_uint4(0u, 0u, 0u, 0u);
    };

    // stage the raw weights in group 0's (still unused) tile set, transpose them into the resident W^T tiles
    const uint32_t nparams = 64 * (in_dim + 64 * (NL - 1) + out_dim);
    uint8_t* stage = sSets;  // >= 64 KB, the weights are <= 22.5 KB
    for (uint32_t c = tid; c < nparams * 2 / 16; c += 128 * kBwdGroups)
        cp_async16(smem_u32(stage) + c * 16u, reinterpret_cast<const uint4*>(weights) + c);
    cp_async_commit();
    if (warp == 0) tmem_alloc(tslot, 512);
    if (tid == 32) {
        for (uint32_t i = 0; i < kBwdGroups; i++) mbar_init(mbars + i, 1);
        fence_mbar_init();
    }
    cp_async_wait_all();
    __syncthreads();
    {
        const __half* w = reinterpret_cast<const __half*>(stage);
        auto transpose = [&](uint8_t* tile, const __half* src, uint32_t rows, uint32_t K) {  // (r, k) -> tile row k, column r
            for (uint32_t e = tid; e < rows * K; e += 128 * kBwdGroups) {
                const uint32_t r = e / K, k = e - r * K;
                *reinterpret_cast<__half*>(tile + sw128(k, r >> 3) + (r & 7u) * 2u) = src[e];
            }
        };
        transpose(sWT + (NL - 1) * kWBytes, w + 64 * in_dim + (NL - 1) * 4096, out_dim, 64);  // W_NL [out,64] -> [64][out]
        for (uint32_t m = 1; m < NL; m++) transpose(sWT + (m - 1) * kWBytes, w + 64 * in_dim + (m - 1) * 4096, 64, 64);
        if (calc_grad_inputs) transpose(sWT0, w, 64, in_dim);  // W_0 [64,in] -> [in][64]
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();   // transposes done (the staging area may be overwritten), TMEM allocated, mbarriers initialised
    tc_fence_after();
    const uint32_t tmem = *tslot + g * gcols;                               // this group's columns
    const uint32_t taddr = tmem + ((uint32_t)((warp & 3u) * 32u) << 16);
    // group-relative TMEM columns: [0,64) dgrad accumulator; then dW_NL (out_dim), dW_{NL-1}..dW_1 (64 each), dW_0 (in_dim)
    auto acc_col = [&](uint32_t m) -> uint32_t {
        if (m == NL) return 64u;
        if (m == 0) return 64u + out_dim + 64u * (NL - 1);
        return 64u + out_dim + 64u * (NL - 1 - m);
    };
    uint32_t phase = 0, it = 0;

    // first tile of this group: all of its units, in the order the chain consumes them
    uint32_t dy_next[2] = {0u, 0u};
    for (uint32_t u = 0; u <= NL; u++) load_unit(first, NL - u);
    if (GLUE) {
        glue_dy_regs(first, dy_next);
        glue_dy_store(dy_next);
    }
    wait_loads();
    fence_proxy_async();
    group_barrier(g);

    for (uint32_t tile = first; tile < ntiles; tile += stride, it++) {
        const size_t r0 = (size_t)tile * kRows;
        const uint32_t next = tile + stride;
        float glue_gs = 0.f, glue_h0 = 0.f;
        if (GLUE) {  // the trunc_exp backward inputs of this row, used by the epilogue at the end of the chain
            glue_gs = __ldcs(glue.grad_sigma + r0 + row);
            glue_h0 = __half2float(glue.h0[r0 + row]);
        }
        for (uint32_t m = NL; m >= 1; m--) {
            uint8_t* Gm = m == NL ? sDY : sH + m * kTileBytes;   // G_m lives in H_m's tile (in place), dY for the output layer
            uint8_t* Hp = sH + (m - 1) * kTileBytes;             // H_{m-1}: input of matmul m, ReLU mask, and the home of G_{m-1}
            const uint32_t n_m = m == NL ? out_dim : 64u;
            if ((gt >> 5) == 0) {  // the group's first warp, uniformly; one elected lane issues (see umma_chain)
                tc_fence_after();
                // wgrad: acc_m[feature i][neuron j] += H_{m-1}^T . G_m  (K = the 128 rows, 16 per MMA = 2048 B)
                const uint64_t wa = desc_sw128(smem_u32(Hp), kTileBytes), wb = desc_sw128(smem_u32(Gm), kTileBytes);
                const uint32_t widesc = make_idesc(128, n_m, true, true);
                // dgrad: D[128,64] = G_m[128,n_m] . W_m[n_m,64]
                const uint64_t a = desc_sw128(smem_u32(Gm), 16), b = desc_sw128(smem_u32(sWT + (m - 1) * kWBytes), 16);
                const uint32_t idesc = make_idesc(128, 64, false, false);
                if (elect_one()) {
                    umma_chain<8>(tmem + acc_col(m), wa, wb, 128, 128, widesc, it > 0);
                    if (m == NL) umma_chain<1>(tmem, a, b, 2, 2, idesc, false);   // n_m = out_dim = 16
                    else umma_chain<4>(tmem, a, b, 2, 2, idesc, false);           // n_m = 64
                    umma_commit(mbar);  // covers both: H_{m-1} may be overwritten once it fires
                }
                __syncwarp();
            }
            // the saved activations of this row, fetched while the tensor core works
            uint4 hrow[8];
#pragma unroll
            for (uint32_t q = 0; q < 8; q++) hrow[q] = *reinterpret_cast<const uint4*>(Hp + sw128(row, q));
            mbar_wait_hot(mbar, phase);
            phase ^= 1u;
            tc_fence_after();
            uint32_t r[64];
            tmem_ld32_nowait(taddr, r);
            tmem_ld32_nowait(taddr + 32, r + 32);
            tmem_wait_ld();
            const __half2 zero2 = __float2half2_rn(0.0f);
#pragma unroll
            for (uint32_t q = 0; q < 8; q++) {
                const uint32_t hw[4] = {hrow[q].x, hrow[q].y, hrow[q].z, hrow[q].w};
                uint32_t o[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {  // round to fp16, then keep where the saved activation is positive
                    const uint32_t pk = pack_h2(__uint_as_float(r[q * 8 + 2 * j]), __uint_as_float(r[q * 8 + 2 * j + 1]));
                    o[j] = pk & __hgt2_mask(*reinterpret_cast<const __half2*>(&hw[j]), zero2);
                }
                *reinterpret_cast<uint4*>(Hp + sw128(row, q)) = make_uint4(o[0], o[1], o[2], o[3]);
            }
            // G_m's tile is free (both MMAs that read it have completed): stream in the next tile's rows for the same step
            load_unit(next, m);
            if (GLUE) {
                if (m == NL) glue_dy_regs(next, dy_next);          // global loads issued now ...
                else if (m == NL - 1) glue_dy_store(dy_next);      // ... consumed one step later
            }
            wait_loads();
            tc_fence_before();
            fence_proxy_async();
            group_barrier(g);
        }
        // input layer: dW_0[neuron j][feature i] += G_0^T . X ; optionally dX = G_0 . W_0   (G_0 lives in H_0's tile)
        if ((gt >> 5) == 0) {
            tc_fence_after();
            const uint64_t a = desc_sw128(smem_u32(sH), 16), b = desc_sw128(smem_u32(sWT0), 16);
            const uint32_t idesc = make_idesc(128, in_dim, false, false);
            const uint64_t wa = desc_sw128(smem_u32(sH), kTileBytes), wb = desc_sw128(smem_u32(sX), kTileBytes);
            const uint32_t widesc = make_idesc(128, in_dim, true, true);
            if (elect_one()) {
                if (calc_grad_inputs) umma_chain<4>(tmem, a, b, 2, 2, idesc, false);
                umma_chain<8>(tmem + acc_col(0), wa, wb, 128, 128, widesc, it > 0);
                umma_commit(mbar);
            }
            __syncwarp();
        }
        mbar_wait_hot(mbar, phase);  // every MMA of this tile has finished: its shared-memory tiles may be overwritten
        phase ^= 1u;
        tc_fence_after();
        if (GLUE) {
            float v[16], o[16];
            tmem_ld16(taddr + 16, v);  // dL/dinput[:, 16:32] = dL/dgeo_feat (15) and the zero-pad column
            o[0] = glue_gs * glue.density_scale * expf(fminf(fmaxf(glue_h0, -15.0f), 15.0f));
#pragma unroll
            for (int i = 1; i < 16; i++) o[i] = v[i - 1];
            uint32_t pk[8];
#pragma unroll
            for (int i = 0; i < 8; i++) pk[i] = pack_h2(o[2 * i], o[2 * i + 1]);
            st_global_32B(glue.dh + (r0 + row) * 16, pk);
        } else if (calc_grad_inputs) {
            __half* gi = grad_inputs + (r0 + row) * in_dim;
            for (uint32_t q = 0; q < in_dim / 16; q++) {
                float v[16];
                tmem_ld16(taddr + q * 16, v);
                uint32_t pk[8];
#pragma unroll
                for (int i = 0; i < 8; i++) pk[i] = pack_h2(v[2 * i], v[2 * i + 1]);
                st_global_32B(gi + q * 16, pk);
            }
        }
        load_unit(next, 0);  // H_0 (holding G_0) and X are free: the last unit of the next tile
        wait_loads();
        tc_fence_before();
        fence_proxy_async();
        group_barrier(g);  // all TMEM reads of this tile are done and the next tile's first units are visible
    }
    cp_async_wait_all();

    // ---- flush the weight-gradient accumulators (rows 0..63 are real; lanes 64..127 hold the ignored atom) ----
    // No atomics: group 1 parks its sums in shared memory, group 0 adds its own and writes this CTA's slice of the partial-sum
    // buffer with plain coalesced stores; k_wgrad_reduce adds the <= 148 slices in a fixed order (deterministic gradients).
    cp_async_wait_all();
    tc_fence_after();
    __syncthreads();
    float* park = reinterpret_cast<float*>(sSets);  // [column][64 rows] fp32, <= 45 KB of the (now idle) tile sets
    const uint32_t wcols = gcols - 64;               // accumulator columns after the dgrad block
    const bool other_has = blockIdx.x * kBwdGroups + 1 < ntiles;  // did group 1 process any tile?
    if (g == 1 && it > 0 && (warp & 3u) < 2) {
        for (uint32_t c = 0; c < wcols; c += 16) {
            float v[16];
            tmem_ld16(taddr + 64 + c, v);
#pragma unroll
            for (int j = 0; j < 16; j++) park[(c + j) * 64 + row] = v[j];
        }
    }
    __syncthreads();
    if (g == 0 && (warp & 3u) < 2) {
        float* slice = wgrad + (size_t)blockIdx.x * nparams;
        const uint32_t w_first = 64 * in_dim;
        for (uint32_t m = 1; m <= NL; m++) {  // acc_m[i][j] = dW_m[j][i]; lane = i -> coalesced over i
            const uint32_t n_m = m == NL ? out_dim : 64u;
            float* dst = slice + w_first + (m - 1) * 4096;
            for (uint32_t q = 0; q < n_m / 16; q++) {
                float v[16];
                tmem_ld16(taddr + acc_col(m) + q * 16, v);
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    const float o = other_has ? park[(acc_col(m) - 64 + q * 16 + j) * 64 + row] : 0.0f;
                    dst[(q * 16 + j) * 64 + row] = v[j] + o;
                }
            }
        }
        for (uint32_t q = 0; q < in_dim / 16; q++) {  // acc_0[j][i] = dW_0[j][i]; lane = j
            float v[16];
            tmem_ld16(taddr + acc_col(0) + q * 16, v);
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const float o = other_has ? park[(acc_col(0) - 64 + q * 16 + i) * 64 + row] : 0.0f;
                slice[row * in_dim + q * 16 + i] = v[i] + o;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(*tslot, 512);
}

// gw[i] = sum over slices of partial[s][i] (fixed order), rounded to fp16 (optionally added to the existing value).
// 256 threads = 32 parameters (one 128-byte line per slice) x 8 slice lanes.
// One launch serves up to two networks (blocks [0, ceil(a.n/32)) reduce `a`, the rest `b`): the fused NeRF backward finishes
// the colour net's and the sigma net's weight gradients together instead of with a launch each.
__global__ void __launch_bounds__(256)
k_wgrad_reduce(const WgradPending a, const WgradPending b) {
    __shared__ float red[8][32];
    pdl_trigger();
    pdl_wait();  // nothing below may run before the kernels ahead on the stream are complete (common.cuh)
    const uint32_t blocks_a = (a.n + 31u) / 32u;
    const bool first = blockIdx.x < blocks_a;
    const float* __restrict__ partial = first ? a.partial : b.partial;
    __half* __restrict__ gw = first ? a.gw : b.gw;
    const uint32_t nslices = first ? a.nslices : b.nslices, n = first ? a.n : b.n;
    const int accumulate = first ? a.accumulate : b.accumulate;
    const uint32_t c = threadIdx.x & 31u, l = threadIdx.x >> 5;
    const uint32_t p = (first ? blockIdx.x : blockIdx.x - blocks_a) * 32 + c;
    float acc = 0.0f;
    if (p < n) {
#pragma unroll 5
        for (uint32_t sidx = l; sidx < nslices; sidx += 8) acc += __ldcs(partial + (size_t)sidx * n + p);
    }
    red[l][c] = acc;
    __syncthreads();
    if (l == 0 && p < n) {
        const float t = ((red[0][c] + red[1][c]) + (red[2][c] + red[3][c])) + ((red[4][c] + red[5][c]) + (red[6][c] + red[7][c]));
        gw[p] = __float2half_rn(accumulate ? __half2float(gw[p]) + t : t);
    }
}

static size_t bwd2_smem_bytes(const MlpShape& sh) {
    return 1024 + (sh.n_layers + 1) * kWBytes + kTileBytes * (kBwdGroups * (sh.n_layers + 2) + 1) + 128;
}


}  // namespace lnrf

using namespace lnrf;

static int check_mlp(const char* who, uint32_t B, uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers,
                     uint32_t activation, uint32_t output_activation, MlpShape* sh) {
    if (!(hidden_dim == 16 || hidden_dim == 32 || hidden_dim == 64 || hidden_dim == 128 || hidden_dim == 256)) {
        set_error("hidden_dim should in [16, 32, 64, 128, 256]");  // ffmlp.cu:657
        return LNRF_ERR_INVALID_ARGUMENT;
    }
    if (hidden_dim != 64) {
        set_error("%s: hidden_dim %u not built (this library implements the 64-wide nets LAENeRF uses)", who, hidden_dim);
        return LNRF_ERR_UNSUPPORTED;
    }
    LNRF_REQUIRE(input_dim > 0 && input_dim % 16 == 0, "FFMLP input_dim should be 16 * m (m > 0), but got %u", input_dim);
    LNRF_REQUIRE(output_dim > 0 && output_dim % 16 == 0, "%s: (padded) output_dim should be 16 * m, but got %u", who, output_dim);
    LNRF_REQUIRE(num_layers >= 2, "FFMLP num_layers should be larger than 2 (3 matmuls), but got %u", num_layers);
    LNRF_REQUIRE(B % 128 == 0, "ffmlp batch size must be 128 * m (m > 0), but got %u.", B);
    if (input_dim > 64 || output_dim > 64 || num_layers > kMaxLayers) {
        set_error("%s: input_dim %u / output_dim %u / num_layers %u outside the built range (<=64, <=64, <=%u)", who, input_dim,
                  output_dim, num_layers, kMaxLayers);
        return LNRF_ERR_UNSUPPORTED;
    }
    LNRF_REQUIRE(activation <= 6 && output_activation <= 6, "%s: activation id out of range", who);
    sh->in_dim = input_dim; sh->out_dim = output_dim; sh->n_layers = num_layers; sh->act = activation; sh->out_act = output_activation;
    return LNRF_OK;
}

static size_t fwd_smem_bytes(const MlpShape& sh) {
    return 1024 + sh.n_layers * kWBytes + ((sh.out_dim * 128u + 1023u) & ~1023u) + 4 * kTileBytes + 64;
}
static size_t bwd_smem_bytes(const MlpShape& sh, uint32_t nbuf) {
    return 1024 + (sh.n_layers + 1) * kWBytes + kTileBytes * (2 + nbuf * (sh.n_layers + 2)) + 64;
}

template <bool TRAIN>
static int ffmlp_fwd_launch(const char* who, const void* inputs, const void* weights, uint32_t B, const MlpShape& sh, void* fwd_buf,
                            void* outputs, cudaStream_t st) {
    if (B == 0) return LNRF_OK;
    LNRF_REQUIRE(inputs && weights && outputs && (!TRAIN || fwd_buf), "%s: null pointer", who);
    LNRF_REQUIRE(((reinterpret_cast<uintptr_t>(inputs) | reinterpret_cast<uintptr_t>(weights) | reinterpret_cast<uintptr_t>(outputs) |
                   reinterpret_cast<uintptr_t>(fwd_buf)) & 15) == 0, "%s: tensors must be 16-byte aligned", who);
    const size_t smem = fwd_smem_bytes(sh);
    auto kern = sh.act == 0 ? k_ffmlp_fwd<TRAIN, 0> : k_ffmlp_fwd<TRAIN, kActRuntime>;
    static std::atomic<size_t> s_max_smem[2] = {{0}, {0}};  // per instantiation: raise the opt-in limit only when it grows
    std::atomic<size_t>& mx = s_max_smem[sh.act == 0 ? 0 : 1];
    if (smem > mx.load(std::memory_order_relaxed)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, who);
        mx.store(smem, std::memory_order_relaxed);
    }
    const uint32_t ntiles = B / kRows;
    const uint32_t per_sm = (uint32_t)((227 * 1024) / (smem + 1024));
    const uint32_t cap = (uint32_t)kNumSMs * (per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm));
    const uint32_t grid = ntiles < cap ? ntiles : cap;
    kern<<<grid, 128, smem, st>>>((const __half*)inputs, (const __half*)weights, (__half*)fwd_buf, (__half*)outputs, B, sh, ntiles);
    LNRF_LAUNCH_CHECK(who);
    return LNRF_OK;
}

namespace lnrf {

// cuTensorMapEncodeTiled through the runtime's driver entry point table (the library links only cudart).
// `cols` x `rows` fp16 row-major with `row_bytes` between rows; box = box_cols x box_rows; SWIZZLE_128B; out-of-bounds elements of a
// box read as zero (a 64-column box over a 32-column tensor lands as full 128-byte rows whose upper half is zero).
int make_tensor_map_2d(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t row_bytes, uint32_t box_cols,
                       uint32_t box_rows, const char* who) {
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static std::atomic<encode_fn> s_encode{nullptr};
    encode_fn enc = s_encode.load(std::memory_order_acquire);
    if (!enc) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess) return cuda_fail(e, who);
        if (!fn || qres != cudaDriverEntryPointSuccess) {
            set_error("%s: cuTensorMapEncodeTiled is not available from this driver", who);
            return LNRF_ERR_CUDA;
        }
        enc = reinterpret_cast<encode_fn>(fn);
        s_encode.store(enc, std::memory_order_release);
    }
    memset(map, 0, sizeof(*map));
    const cuuint64_t gdim[2] = {cols, rows};
    const cuuint64_t gstride[1] = {row_bytes};   // bytes between rows
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("%s: cuTensorMapEncodeTiled failed (CUresult %d)", who, (int)r);
        return LNRF_ERR_CUDA;
    }
    return LNRF_OK;
}

// [rows, 64] fp16 row-major global tensor, box = one 128-row x 128-byte tile
int make_tile_tensor_map(CUtensorMap* map, const void* base, uint64_t rows, const char* who) {
    return make_tensor_map_2d(map, base, 64, rows, 128, 64, kRows, who);
}

int mlp_shape(const char* who, uint32_t B, uint32_t input_dim, uint32_t output_dim, uint32_t num_layers, MlpShape* sh) {
    return check_mlp(who, B, input_dim, output_dim, 64, num_layers, 0, 6, sh);
}

// The two-tile ReLU kernel writes per-CTA slices that k_wgrad_reduce adds in a fixed order; every other net takes k_ffmlp_bwd, whose
// weight gradient is a float atomicAdd per element (order-dependent).
static bool bwd_fixed_order(const MlpShape& sh) {
    const uint32_t nparams = 64u * (sh.in_dim + 64u * (sh.n_layers - 1) + sh.out_dim);
    return sh.act == 0 && kBwdGroups * bwd2_group_cols(sh.in_dim, sh.out_dim, sh.n_layers) <= 512 && bwd2_smem_bytes(sh) <= 227 * 1024 &&
           (kBwdGroups * (sh.n_layers + 2)) * kTileBytes >= 2 * nparams;
}

// One launch for the whole backward of a 64-wide net (+ the fp32 -> fp16 finalize of the weight gradients).  `glue` non-null
// selects the colour-net variant with the NeRFNetwork glue fused in (see k_ffmlp_bwd).
int ffmlp_bwd_run(const char* who, const void* grad_f16, const void* inputs_f16, const void* weights_f16, const void* forward_buffer_f16,
                  uint32_t B, const MlpShape& sh, int calc_grad_inputs, void* grad_inputs_f16, void* grad_weights_f16,
                  void* wgrad_scratch, size_t wgrad_scratch_bytes, const BwdGlue* glue, int accumulate, cudaStream_t st,
                  WgradPending* defer) {
    const uint32_t input_dim = sh.in_dim, output_dim = sh.out_dim, num_layers = sh.n_layers;
    LNRF_REQUIRE(inputs_f16 && weights_f16 && forward_buffer_f16 && grad_weights_f16, "%s: null pointer", who);
    LNRF_REQUIRE(glue || !calc_grad_inputs || grad_inputs_f16, "%s: calc_grad_inputs without grad_inputs", who);
    const size_t need = lnrf_ffmlp_wgrad_scratch_bytes(input_dim, output_dim, 64, num_layers);
    if (!wgrad_scratch || wgrad_scratch_bytes < need) {
        set_error("%s: wgrad scratch too small (%zu < %zu)", who, wgrad_scratch_bytes, need);
        return LNRF_ERR_SCRATCH_TOO_SMALL;
    }
    LNRF_REQUIRE(bwd_tmem_cols(input_dim, output_dim, num_layers) <= 512, "%s: network too deep for one TMEM allocation", who);
    const uint32_t nparams = (uint32_t)(need / sizeof(float) / kNumSMs);
    cudaError_t e = cudaSuccess;
    uint32_t nslices = 1;  // slices of partial sums the reduction adds up (the atomics path accumulates into one)
    const bool relu2 = bwd_fixed_order(sh);
    LNRF_REQUIRE(!glue || relu2, "%s: the fused colour-net backward needs a ReLU net that fits the two-tile kernel", who);
    if (B > 0 && relu2) {
        const size_t smem = bwd2_smem_bytes(sh);
        auto kern = glue ? k_mlp_bwd2<true> : k_mlp_bwd2<false>;
        static std::atomic<size_t> s_max2[2] = {{0}, {0}};
        std::atomic<size_t>& mx = s_max2[glue ? 1 : 0];
        if (smem > mx.load(std::memory_order_relaxed)) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return cuda_fail(e, who);
            mx.store(smem, std::memory_order_relaxed);
        }
        const uint32_t ntiles = B / kRows;
        const uint32_t want = div_up(ntiles, kBwdGroups);
        const uint32_t grid = want < (uint32_t)kNumSMs ? want : (uint32_t)kNumSMs;
        nslices = grid;  // every CTA writes its whole slice: nothing to clear
        BwdGlue g{};
        if (glue) g = *glue;
        kern<<<grid, 128 * kBwdGroups, smem, st>>>((const __half*)grad_f16, (const __half*)inputs_f16, (const __half*)weights_f16,
                                                   (const __half*)forward_buffer_f16, (__half*)grad_inputs_f16, (float*)wgrad_scratch, B,
                                                   sh, ntiles, glue ? 1 : calc_grad_inputs, g);
        LNRF_LAUNCH_CHECK(who);
    } else {
        e = cudaMemsetAsync(wgrad_scratch, 0, sizeof(float) * nparams, st);
        if (e != cudaSuccess) return cuda_fail(e, who);
    }
    if (B > 0 && !relu2) {
        const uint32_t nbuf = bwd_smem_bytes(sh, 2) <= 227 * 1024 ? 2u : 1u;  // prefetch the next tile when it fits
        const size_t smem = bwd_smem_bytes(sh, nbuf);
        LNRF_REQUIRE(smem <= 227 * 1024, "%s: network needs %zu B of shared memory (> 227 KiB)", who, smem);
        const int variant = sh.act == 0 ? 0 : 1;
        auto kern = variant == 0 ? k_ffmlp_bwd<0, false> : k_ffmlp_bwd<kActRuntime, false>;
        static std::atomic<size_t> s_max_smem[2] = {{0}, {0}};
        std::atomic<size_t>& mx = s_max_smem[variant];
        if (smem > mx.load(std::memory_order_relaxed)) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return cuda_fail(e, who);
            mx.store(smem, std::memory_order_relaxed);
        }
        const uint32_t ntiles = B / kRows;
        const uint32_t per_sm_smem = (uint32_t)((227 * 1024) / (smem + 1024));
        const uint32_t per_sm_tmem = 512u / bwd_tmem_cols(input_dim, output_dim, num_layers);
        uint32_t per_sm = per_sm_smem < per_sm_tmem ? per_sm_smem : per_sm_tmem;
        if (per_sm < 1) per_sm = 1;
        const uint32_t cap = (uint32_t)kNumSMs * per_sm;
        const uint32_t grid = ntiles < cap ? ntiles : cap;
        kern<<<grid, 128, smem, st>>>((const __half*)grad_f16, (const __half*)inputs_f16, (const __half*)weights_f16,
                                      (const __half*)forward_buffer_f16, (__half*)grad_inputs_f16, (float*)wgrad_scratch, B, sh,
                                      ntiles, calc_grad_inputs, nbuf, BwdGlue{});
        LNRF_LAUNCH_CHECK(who);
    }
    if (defer) {  // the caller reduces several networks' partial sums in one launch (wgrad_reduce_pair)
        *defer = WgradPending{(const float*)wgrad_scratch, nslices, (__half*)grad_weights_f16, nparams, accumulate};
        return LNRF_OK;
    }
    k_wgrad_reduce<<<div_up(nparams, 32u), 256, 0, st>>>(WgradPending{(const float*)wgrad_scratch, nslices, (__half*)grad_weights_f16, nparams, accumulate},
                                                         WgradPending{nullptr, 0, nullptr, 0, 0});
    LNRF_LAUNCH_CHECK(who);
    return LNRF_OK;
}

int wgrad_reduce_pair(const char* who, const WgradPending& a, const WgradPending& b, cudaStream_t st) {
    launch_pdl(k_wgrad_reduce, div_up(a.n, 32u) + div_up(b.n, 32u), 256, 0, st, a, b);
    LNRF_LAUNCH_CHECK(who);
    return LNRF_OK;
}

}  // namespace lnrf

extern "C" {

int lnrf_ffmlp_forward(const void* inputs_f16, const void* weights_f16, uint32_t B, uint32_t input_dim, uint32_t output_dim,
                       uint32_t hidden_dim, uint32_t num_layers, uint32_t activation, uint32_t output_activation,
                       void* forward_buffer_f16, void* outputs_f16, lnrf_stream_t stream) {
    MlpShape sh;
    if (int e = check_mlp("ffmlp_forward", B, input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, &sh)) return e;
    return ffmlp_fwd_launch<true>("ffmlp_forward", inputs_f16, weights_f16, B, sh, forward_buffer_f16, outputs_f16,
                                  reinterpret_cast<cudaStream_t>(stream));
}

int lnrf_ffmlp_inference(const void* inputs_f16, const void* weights_f16, uint32_t B, uint32_t input_dim, uint32_t output_dim,
                         uint32_t hidden_dim, uint32_t num_layers, uint32_t activation, uint32_t output_activation,
                         void* inference_buffer_f16, void* outputs_f16, lnrf_stream_t stream) {
    (void)inference_buffer_f16;
    MlpShape sh;
    if (int e = check_mlp("ffmlp_inference", B, input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, &sh)) return e;
    return ffmlp_fwd_launch<false>("ffmlp_inference", inputs_f16, weights_f16, B, sh, nullptr, outputs_f16,
                                   reinterpret_cast<cudaStream_t>(stream));
}

// one fp32 slice of partial weight-gradient sums per CTA of the persistent backward kernel (<= one CTA per SM)
size_t lnrf_ffmlp_wgrad_scratch_bytes(uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers) {
    return sizeof(float) * (size_t)hidden_dim * (input_dim + (size_t)hidden_dim * (num_layers - 1) + output_dim) * (size_t)kNumSMs;
}

int lnrf_ffmlp_backward(const void* grad_f16, const void* inputs_f16, const void* weights_f16, const void* forward_buffer_f16,
                        uint32_t B, uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers,
                        uint32_t activation, uint32_t output_activation, int calc_grad_inputs, void* backward_buffer_f16,
                        void* grad_inputs_f16, void* grad_weights_f16, void* wgrad_scratch, size_t wgrad_scratch_bytes,
                        lnrf_stream_t stream) {
    (void)backward_buffer_f16;  // dL/dhidden never leaves the chip
    MlpShape sh;
    if (int e = check_mlp("ffmlp_backward", B, input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, &sh)) return e;
    LNRF_REQUIRE(grad_f16, "ffmlp_backward: null pointer");
    return lnrf::ffmlp_bwd_run("ffmlp_backward", grad_f16, inputs_f16, weights_f16, forward_buffer_f16, B, sh, calc_grad_inputs,
                               grad_inputs_f16, grad_weights_f16, wgrad_scratch, wgrad_scratch_bytes, nullptr, 0,
                               reinterpret_cast<cudaStream_t>(stream));
}

int lnrf_ffmlp_backward_deterministic(uint32_t input_dim, uint32_t output_dim, uint32_t hidden_dim, uint32_t num_layers, uint32_t activation,
                                      uint32_t output_activation) {
    MlpShape sh;
    if (int e = check_mlp("ffmlp_backward_deterministic", 128, input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, &sh))
        return e;
    return lnrf::bwd_fixed_order(sh) ? 1 : 0;
}

int lnrf_allocate_splitk(size_t size) { (void)size; return LNRF_OK; }
int lnrf_free_splitk(void) { return LNRF_OK; }

}  // extern "C"
