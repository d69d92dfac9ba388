// Memory-bound companions of the tcgen05 convolution on the U-Net path (sm_100a):
//   * per-(sample, channel) moment reduction        (LayerNorm[D,H,W] / GroupNorm statistics)
//   * normalise + affine + activation + fp16 cast   (the A operand of the next convolution)
//   * nearest x2 upsample + fp16 cast               (diffusion_network.py:69, F.interpolate)
//   * single-head attention over the bottleneck     (diffusion_network.py:213-242)
// All activations are channels-last: x[nb][voxel][channel], fp32 in, fp16 out.
#include "unet_kernels.cuh"

#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cstdint>
#include <cstdlib>

#include "conv3d_igemm.cuh"   // kF8Shift

namespace pixie {

namespace {

__device__ __forceinline__ float act_apply(float v, int act) {
    if (act == kActLeaky) return v > 0.f ? v : 0.02f * v;            // nn.LeakyReLU(0.02), training_discrete.py:80
    // nn.SiLU. __fdividef: 2 ulp, two instructions instead of the ~12 of an IEEE division; the value is rounded to 11 + 3 bits next
    if (act == kActSiLU) return __fdividef(v, 1.f + __expf(-v));
    return v;
}

__device__ __forceinline__ uint32_t pack_e5m2x4(float a, float b, float c, float d) {
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E5M2);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E5M2);
    return lo | (hi << 16);
}

// Packs 4 floats (consecutive channels, idx % 4 == 0) to fp16 (hi) and, when lo != nullptr, what the split-precision
// convolution needs next to it:
//   lo_mode 0: the rounding residual f - float(hi) as fp16, same layout as hi;
//   lo_mode 1: the E5M2 correction operands. `lo` is then a byte tensor with 2*ld bytes per voxel row; the 64-channel
//              chunk k occupies bytes [128k, 128k+128): 64 x e5m2((f - float(hi)) * 2^kF8Shift) then 64 x e5m2(f * 2^-kF8Shift)
//              (row strides and channel offsets are multiples of 64, so idx & 63 is the channel inside its chunk).
template <int LOM>   // -1: run-time (lo may be null, lo_mode as passed); 0 / 1: lo present with that mode; 2: no lo tensor
__device__ __forceinline__ void store_hi_lo_t(const float (&f)[4], __half* hi, __half* lo, size_t idx, int lo_mode) {
    if (LOM == 2) lo = nullptr;
    if (LOM == 0 || LOM == 1) lo_mode = LOM;
    __half2 r0 = __floats2half2_rn(f[0], f[1]), r1 = __floats2half2_rn(f[2], f[3]);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&r0); pk.y = *reinterpret_cast<uint32_t*>(&r1);
    *reinterpret_cast<uint2*>(hi + idx) = pk;
    if (lo && lo_mode == 1) {
        const float2 b0 = __half22float2(r0), b1 = __half22float2(r1);
        constexpr float up = (float)(1 << kF8Shift), down = 1.0f / (float)(1 << kF8Shift);
        uint8_t* row = reinterpret_cast<uint8_t*>(lo) + 2 * (idx & ~(size_t)63) + (idx & 63);
        *reinterpret_cast<uint32_t*>(row) = pack_e5m2x4((f[0] - b0.x) * up, (f[1] - b0.y) * up, (f[2] - b1.x) * up, (f[3] - b1.y) * up);
        *reinterpret_cast<uint32_t*>(row + 64) = pack_e5m2x4(f[0] * down, f[1] * down, f[2] * down, f[3] * down);
    } else if (lo) {
        const float2 b0 = __half22float2(r0), b1 = __half22float2(r1);
        __half2 l0 = __floats2half2_rn(f[0] - b0.x, f[1] - b0.y), l1 = __floats2half2_rn(f[2] - b1.x, f[3] - b1.y);
        uint2 pl; pl.x = *reinterpret_cast<uint32_t*>(&l0); pl.y = *reinterpret_cast<uint32_t*>(&l1);
        *reinterpret_cast<uint2*>(lo + idx) = pl;
    }
}
__device__ __forceinline__ void store_hi_lo(const float (&f)[4], __half* hi, __half* lo, size_t idx, int lo_mode) {
    store_hi_lo_t<-1>(f, hi, lo, idx, lo_mode);
}

}  // namespace

// ------------------------------------------------------------------------------------ moments
// grid = (ceil(V / vox_per_block), NB), block = 256.  C % 4 == 0, C/4 <= 256.
__global__ void __launch_bounds__(256)
moments_kernel(const float* __restrict__ x, int V, int C, int vox_per_block, double* __restrict__ stats) {
    const int cols4 = C >> 2;
    const int rows_par = 256 / cols4;
    const int col = threadIdx.x % cols4;
    const int row = threadIdx.x / cols4;
    const int nb = blockIdx.y;
    const int v0 = blockIdx.x * vox_per_block;
    const int v1 = min(V, v0 + vox_per_block);
    float s[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
    if (row < rows_par) {
        const float4* xp = reinterpret_cast<const float4*>(x + ((size_t)nb * V) * C) + col;
#pragma unroll 4
        for (int v = v0 + row; v < v1; v += rows_par) {
            const float4 a = __ldg(xp + (size_t)v * cols4);
            s[0] += a.x; s[1] += a.y; s[2] += a.z; s[3] += a.w;
            q[0] += a.x * a.x; q[1] += a.y * a.y; q[2] += a.z * a.z; q[3] += a.w * a.w;
        }
    }
    __shared__ float sh[256 * 8];
    float* mine = sh + threadIdx.x * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) { mine[j] = s[j]; mine[4 + j] = q[j]; }
    __syncthreads();
    if (threadIdx.x < cols4) {
        double ds[4] = {0, 0, 0, 0}, dq[4] = {0, 0, 0, 0};
        for (int r = 0; r < rows_par; ++r) {
            const float* o = sh + (r * cols4 + threadIdx.x) * 8;
#pragma unroll
            for (int j = 0; j < 4; ++j) { ds[j] += o[j]; dq[j] += o[4 + j]; }
        }
        double* st = stats + ((size_t)nb * C + threadIdx.x * 4) * 2;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(st + 2 * j, ds[j]);
            atomicAdd(st + 2 * j + 1, dq[j]);
        }
    }
}

// ------------------------------------------------------------------------------------ normalise
// y = act((x - mean) * rstd * gamma + beta) -> fp16; optional raw fp16 copy of x.
// mode LN : statistics per (nb, c) over V; gamma/beta indexed by voxel   (nn.LayerNorm([sp,sp,sp]))
// mode GN : statistics per (nb, group) over V x cg channels; gamma/beta indexed by channel
// mode NONE: cast only (raw copy).
// MODE / ACT / LOM (the presence and kind of the `lo` tensors) are compile-time: with run-time switches the pass spent ~46
// thread-instructions per element and was issue-bound at 45 % of HBM (r02 ncu: IPC 2.7, sm throughput 58 %, dram 45 %).
template <int MODE, int ACT, int LOM>
__global__ void __launch_bounds__(256)
norm_act_kernel(NormArgs a) {
    // per-channel (mean, rstd, gamma, beta) once per block, in shared memory (C <= 1024)
    __shared__ float s_mean[1024], s_rstd[1024], s_g[1024], s_b[1024];
    const int nb = blockIdx.y;
    if (MODE != kNormNone) {
        const int cg = (MODE == kNormGN) ? a.C / a.groups : 1;
        for (int ch = threadIdx.x; ch < a.C; ch += blockDim.x) {
            const int grp0 = (ch / cg) * cg;
            double s = 0, q = 0;
            for (int k = 0; k < cg; ++k) {
                s += a.stats[((size_t)nb * a.C + grp0 + k) * 2];
                q += a.stats[((size_t)nb * a.C + grp0 + k) * 2 + 1];
            }
            const double n = (double)a.V * cg;
            const double m = s / n;
            double var = q / n - m * m;
            if (var < 0) var = 0;
            s_mean[ch] = (float)m;
            s_rstd[ch] = (float)(1.0 / sqrt(var + (double)a.eps));
            s_g[ch] = (MODE == kNormGN) ? a.gamma[ch] : 1.f;
            s_b[ch] = (MODE == kNormGN) ? a.beta[ch] : 0.f;
        }
        __syncthreads();
    }
    const int cols4 = a.C >> 2;
    const int rows_par = 256 / cols4;
    const int col = threadIdx.x % cols4;
    const int row = threadIdx.x / cols4;
    if (row >= rows_par) return;
    const int c = col * 4;
    float mean[4] = {0, 0, 0, 0}, rstd[4] = {1, 1, 1, 1}, g[4] = {1, 1, 1, 1}, b[4] = {0, 0, 0, 0};
    if (MODE != kNormNone) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { mean[j] = s_mean[c + j]; rstd[j] = s_rstd[c + j]; g[j] = s_g[c + j]; b[j] = s_b[c + j]; }
    }
    const int v0 = blockIdx.x * a.vox_per_block;
    const int v1 = min(a.V, v0 + a.vox_per_block);
    const float4* xp = reinterpret_cast<const float4*>(a.x + ((size_t)nb * a.V) * a.C) + col;
    // 4 voxel rows per trip with all loads issued first: one 16-byte load in flight per thread is latency-bound
    // (ncu/bench: 25 us per 100 MB pass = 25 % of HBM)
    constexpr int U = 4;
    for (int vb = v0 + row; vb < v1; vb += rows_par * U) {
        float4 xv[U];
        float gv[U], bv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int v = vb + u * rows_par;
            const bool in = v < v1;
            xv[u] = in ? __ldg(xp + (size_t)v * cols4) : make_float4(0.f, 0.f, 0.f, 0.f);
            gv[u] = 1.f; bv[u] = 0.f;
            if (in && MODE == kNormLN && a.dst) { gv[u] = __ldg(a.gamma + v); bv[u] = __ldg(a.beta + v); }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int v = vb + u * rows_par;
            if (v >= v1) break;
            float f[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
            if (a.raw_dst) store_hi_lo_t<-1>(f, a.raw_dst, a.raw_lo, ((size_t)nb * a.V + v) * a.raw_ld + a.raw_c0 + c, a.lo_mode);
            if (a.dst) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float y = f[j];
                    if (MODE == kNormLN) y = (y - mean[j]) * rstd[j] * gv[u] + bv[u];
                    else if (MODE == kNormGN) y = (y - mean[j]) * rstd[j] * g[j] + b[j];
                    f[j] = act_apply(y, ACT);
                }
                store_hi_lo_t<LOM>(f, a.dst, a.dst_lo, ((size_t)nb * a.V + v) * a.dst_ld + a.dst_c0 + c, a.lo_mode);
            }
        }
    }
}

// ------------------------------------------------------------------------------------ upsample x2
// in: fp32 [NB][sp^3][C]; out: fp16 [NB][(2sp)^3][C], nearest neighbour.
__global__ void __launch_bounds__(256)
upsample2_kernel(const float* __restrict__ x, __half* __restrict__ y, __half* __restrict__ ylo, int lo_mode, int sp, int C, long long total4) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int cols4 = C >> 2;
    const int col = (int)(i % cols4);
    long long v = i / cols4;
    const int S = 2 * sp;
    const int w = (int)(v % S); v /= S;
    const int h = (int)(v % S); v /= S;
    const int d = (int)(v % S); v /= S;
    const long long nb = v;
    const long long src = ((nb * sp + (d >> 1)) * sp + (h >> 1)) * sp + (w >> 1);
    const float4 a = __ldg(reinterpret_cast<const float4*>(x + src * C) + col);
    const float f[4] = {a.x, a.y, a.z, a.w};
    store_hi_lo(f, y, ylo, (size_t)i * 4, lo_mode);
}

// ------------------------------------------------------------------------------------ attention
// qkv: fp32 [NB][T][3C] (q | k | v along channels, Conv1d output order, diffusion_network.py:233)
// out: fp16 [NB][T][C] = softmax_s((q_t . k_s) / sqrt(C)) v_s.   One block per kAttnQ query tokens: every key / value row is
// loaded once per block and used for all of them (one query per block re-read K and V 512 times from L2: 230 us per launch,
// r02 launch list); a warp reads a key row as one coalesced line per 128 channels and reduces the kAttnQ dot products by shuffles.
constexpr int kAttnQ = 4;
__global__ void __launch_bounds__(256)
attention_kernel(const float* __restrict__ qkv, __half* __restrict__ out, __half* __restrict__ out_lo, int lo_mode, int T, int C) {
    extern __shared__ __align__(16) float sm[];
    float* qs = sm;                    // [kAttnQ][C]
    float* sc = sm + kAttnQ * C;       // [kAttnQ][T]
    __shared__ float inv_s[kAttnQ];
    const int t0 = blockIdx.x * kAttnQ, nb = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    const float* base = qkv + (size_t)nb * T * 3 * C;
    const float scale = rsqrtf(sqrtf((float)C));     // applied to q and to k (diffusion_network.py:235-238)
    for (int i = threadIdx.x; i < kAttnQ * C; i += blockDim.x) {
        const int q = i / C, c = i - q * C;
        qs[i] = (t0 + q < T) ? base[(size_t)(t0 + q) * 3 * C + c] * scale : 0.f;
    }
    __syncthreads();
    // ---- scores: warp w takes keys w, w + nwarp, ...
    for (int s = warp; s < T; s += nwarp) {
        const float4* kp = reinterpret_cast<const float4*>(base + (size_t)s * 3 * C + C);
        float part[kAttnQ];
#pragma unroll
        for (int q = 0; q < kAttnQ; ++q) part[q] = 0.f;
        for (int c4 = lane; c4 < C / 4; c4 += 32) {
            float4 kv = __ldg(kp + c4);
            kv.x *= scale; kv.y *= scale; kv.z *= scale; kv.w *= scale;
#pragma unroll
            for (int q = 0; q < kAttnQ; ++q) {
                const float4 qv = *reinterpret_cast<const float4*>(qs + q * C + 4 * c4);
                part[q] += qv.x * kv.x + qv.y * kv.y + qv.z * kv.z + qv.w * kv.w;
            }
        }
#pragma unroll
        for (int q = 0; q < kAttnQ; ++q) {
            float v = part[q];
            for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) sc[q * T + s] = v;
        }
    }
    __syncthreads();
    // ---- softmax: warp q normalises query q
    if (warp < kAttnQ) {
        float* row = sc + warp * T;
        float mx = -INFINITY;
        for (int s = lane; s < T; s += 32) mx = fmaxf(mx, row[s]);
        for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float sum = 0.f;
        for (int s = lane; s < T; s += 32) { const float e = __expf(row[s] - mx); row[s] = e; sum += e; }
        for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) inv_s[warp] = 1.f / sum;
    }
    __syncthreads();
    // ---- weighted values: one channel per thread, every value row read once for the kAttnQ queries
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float acc[kAttnQ];
#pragma unroll
        for (int q = 0; q < kAttnQ; ++q) acc[q] = 0.f;
        const float* vp = base + 2 * C + c;
#pragma unroll 4
        for (int s = 0; s < T; ++s) {
            const float v = __ldg(vp + (size_t)s * 3 * C);
#pragma unroll
            for (int q = 0; q < kAttnQ; ++q) acc[q] = fmaf(sc[q * T + s], v, acc[q]);
        }
#pragma unroll
        for (int q = 0; q < kAttnQ; ++q) {
            if (t0 + q >= T) break;
            const float val = acc[q] * inv_s[q];
            const __half hv = __float2half_rn(val);
            const size_t idx = ((size_t)nb * T + t0 + q) * C + c;
            out[idx] = hv;
            if (out_lo && lo_mode == 1) {
                constexpr float up = (float)(1 << kF8Shift), down = 1.0f / (float)(1 << kF8Shift);
                uint8_t* row = reinterpret_cast<uint8_t*>(out_lo) + 2 * (idx & ~(size_t)63) + (idx & 63);
                row[0] = (uint8_t)__nv_cvt_float_to_fp8((val - __half2float(hv)) * up, __NV_SATFINITE, __NV_E5M2);
                row[64] = (uint8_t)__nv_cvt_float_to_fp8(val * down, __NV_SATFINITE, __NV_E5M2);
            } else if (out_lo) out_lo[idx] = __float2half_rn(val - __half2float(hv));
        }
    }
}

// NCDHW fp32 -> NDHWC fp16 (channel-padded), for callers that hand over the reference's input layout
// (my_data.py:221 permute(3,0,1,2)) instead of the on-disk one.
__global__ void __launch_bounds__(256)
ncdhw_to_ndhwc_f16_kernel(const float* __restrict__ x, __half* __restrict__ y, int C, int Cpad, long long V) {
    // one thread per (voxel, channel) of the padded output; reads are strided, used off the hot path only
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int nb = blockIdx.y;
    if (i >= V * Cpad) return;
    const int c = (int)(i % Cpad);
    const long long v = i / Cpad;
    const float val = c < C ? x[((size_t)nb * C + c) * V + v] : 0.f;
    y[(size_t)nb * V * Cpad + i] = __float2half_rn(val);
}

// save_predictions packing (inference_combined.py:173-199): out[0:3] = continuous prediction,
// out[3 + c] = (argmax_c seg_logits == c) as float, c in [0, n_classes); all planar (C, D, H, W).
__global__ void __launch_bounds__(256)
pack_predictions_kernel(const float* __restrict__ seg, const float* __restrict__ cont, float* __restrict__ out,
                        long long V, int n_classes) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int nb = blockIdx.y;
    if (v >= V) return;
    const float* sp = seg + (size_t)nb * n_classes * V;
    int best = 0;
    float bv = sp[v];
    for (int c = 1; c < n_classes; ++c) {           // torch.argmax returns the first maximal index
        const float x = sp[(size_t)c * V + v];
        if (x > bv) { bv = x; best = c; }
    }
    float* op = out + (size_t)nb * (3 + n_classes) * V;
    for (int c = 0; c < 3; ++c) op[(size_t)c * V + v] = cont[((size_t)nb * 3 + c) * V + v];
    for (int c = 0; c < n_classes; ++c) op[(size_t)(3 + c) * V + v] = (c == best) ? 1.f : 0.f;
}

// ------------------------------------------------------------------------------------ launchers
int launch_pack_predictions(const float* seg, const float* cont, float* out, int NB, long long V, int n_classes, cudaStream_t st) {
    dim3 grid((unsigned)((V + 255) / 256), NB);
    pack_predictions_kernel<<<grid, 256, 0, st>>>(seg, cont, out, V, n_classes);
    return (int)cudaGetLastError();
}

// The convolution kernel runs with the maximum shared-memory carve-out (222 KB per CTA). A kernel that asks for the default
// split makes the SM re-partition L1 / shared memory at the kernel boundary, which it can only do when idle; the streaming
// kernels here do not need L1, so they ask for the same carve-out and the ~390 launches of a network keep one configuration.
// The attribute is set once per kernel, before its first launch.
template <auto kernel>
static inline void prefer_max_smem_carveout() {
    static const cudaError_t set = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    (void)set;
}

// Voxels per block: one trip of a block covers (256 / (C/4)) * 4 voxel rows; aim at >= 2 blocks per SM so that the
// 16^3 and 8^3 levels are not run by 16 blocks (r01 ncu: 20 us for a 2 MB tensor), capped at 512 voxels for the big levels.
static inline int vox_per_block_for(int V, int C) {
    const int trip = (256 / (C / 4)) * 4;
    int vpb = (V + 295) / 296;
    vpb = (vpb + trip - 1) / trip * trip;
    return vpb < trip ? trip : (vpb > 512 ? 512 : vpb);
}

int launch_moments(const float* x, int NB, int V, int C, double* stats, cudaStream_t st) {
    if (C % 4 || C / 4 > 256) return 1;
    const int vpb = vox_per_block_for(V, C);
    dim3 grid((V + vpb - 1) / vpb, NB);
    prefer_max_smem_carveout<moments_kernel>();
    moments_kernel<<<grid, 256, 0, st>>>(x, V, C, vpb, stats);
    return (int)cudaGetLastError();
}

int launch_norm_act(NormArgs a, int NB, cudaStream_t st) {
    if (a.C % 4 || a.C / 4 > 256) return 1;
    a.vox_per_block = vox_per_block_for(a.V, a.C);
    dim3 grid((a.V + a.vox_per_block - 1) / a.vox_per_block, NB);
    const int lom = !a.dst_lo ? 2 : (a.lo_mode == 1 ? 1 : 0);
#define PIXIE_NORM_L(M, A) \
    do { if (lom == 2) { prefer_max_smem_carveout<norm_act_kernel<M, A, 2>>(); norm_act_kernel<M, A, 2><<<grid, 256, 0, st>>>(a); } \
         else if (lom == 1) { prefer_max_smem_carveout<norm_act_kernel<M, A, 1>>(); norm_act_kernel<M, A, 1><<<grid, 256, 0, st>>>(a); } \
         else { prefer_max_smem_carveout<norm_act_kernel<M, A, 0>>(); norm_act_kernel<M, A, 0><<<grid, 256, 0, st>>>(a); } } while (0)
#define PIXIE_NORM_A(M) \
    do { if (a.act == kActSiLU) PIXIE_NORM_L(M, kActSiLU); else if (a.act == kActLeaky) PIXIE_NORM_L(M, kActLeaky); else PIXIE_NORM_L(M, kActNone); } while (0)
    if (a.mode == kNormLN) PIXIE_NORM_A(kNormLN);
    else if (a.mode == kNormGN) PIXIE_NORM_A(kNormGN);
    else PIXIE_NORM_A(kNormNone);
#undef PIXIE_NORM_A
#undef PIXIE_NORM_L
    return (int)cudaGetLastError();
}

int launch_upsample2(const float* x, __half* y, __half* ylo, int lo_mode, int NB, int sp, int C, cudaStream_t st) {
    const long long total4 = (long long)NB * 8 * sp * sp * sp * (C / 4);
    prefer_max_smem_carveout<upsample2_kernel>();
    upsample2_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, st>>>(x, y, ylo, lo_mode, sp, C, total4);
    return (int)cudaGetLastError();
}

int launch_attention(const float* qkv, __half* out, __half* out_lo, int lo_mode, int NB, int T, int C, cudaStream_t st) {
    const size_t smem = (size_t)kAttnQ * (C + T) * sizeof(float);
    if (smem > 48 * 1024 || C % 4) return 1;
    dim3 grid((T + kAttnQ - 1) / kAttnQ, NB);
    prefer_max_smem_carveout<attention_kernel>();
    attention_kernel<<<grid, 256, smem, st>>>(qkv, out, out_lo, lo_mode, T, C);
    return (int)cudaGetLastError();
}

int launch_ncdhw_to_ndhwc_f16(const float* x, __half* y, int NB, int C, int Cpad, long long V, cudaStream_t st) {
    dim3 grid((unsigned)((V * Cpad + 255) / 256), NB);
    ncdhw_to_ndhwc_f16_kernel<<<grid, 256, 0, st>>>(x, y, C, Cpad, V);
    return (int)cudaGetLastError();
}

}  // namespace pixie
