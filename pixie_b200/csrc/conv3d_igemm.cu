// tcgen05 implicit-GEMM Conv3d for sm_100a: kernel + host planning. See conv3d_igemm.cuh.
#include "conv3d_igemm.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>

#include <cuda_fp8.h>

namespace pixie {

using namespace ptx;

namespace {

constexpr int kMaxWStages = 2;
constexpr int kMaxSStages = 8;

struct SmemCtrl {
    uint64_t wfull[kMaxWStages];
    uint64_t wempty[kMaxWStages];
    uint64_t sfull[kMaxSStages];
    uint64_t sempty[kMaxSStages];
    uint64_t tfull[2];
    uint64_t tempty[2];
    uint32_t tmem_base;
    int abort_flag;
};

constexpr int kCtlBarrierBytes = 512;     // SmemCtrl
constexpr int kStatsMaxC = 256;
// per epilogue warp: [2][stats_ld] floats (sum, sum of squares), private to the warp -> no atomics

// Reduces v[0..15] (16 channels held by every lane = one voxel row each) over the 32 lanes of the warp.
// Returns, in every lane, the column sum of channel stats_channel_of_lane(lane). 16 shuffles.
__device__ __forceinline__ float warp_colsum16(float (&v)[16], int lane) {
#pragma unroll
    for (int half = 8, off = 16; half >= 1; half >>= 1, off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float keep = up ? v[i + half] : v[i];
            const float send = up ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}
// Same for 32 channels: after the five halving steps lane l holds the column sum of channel l. 31 shuffles.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
    for (int half = 16, off = 16; half >= 1; half >>= 1, off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float keep = up ? v[i + half] : v[i];
            const float send = up ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}
__device__ __forceinline__ int stats_channel_of_lane(int lane) {
    return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
}

struct TileCoord {
    int nb, d0, h0, w0, n0, ph_begin, ph_end, split, tde;
};

// Tile coordinates of work item `wi`. On the MMA issuer's critical path once per tile (r01 trace: ~1000 cycles with signed and
// 64-bit divisions), so: unsigned 32-bit divisions only, and none at all for the split-K bookkeeping of unsplit convolutions.
__device__ __forceinline__ TileCoord decode_tile(const ConvKernelParams& p, int wi) {
    TileCoord t;
    unsigned rest = (unsigned)wi;
    if (p.split_k == 1) {
        t.split = 0; t.ph_begin = 0; t.ph_end = p.n_phases;
    } else {
        const unsigned sk = (unsigned)p.split_k;
        t.split = (int)(rest % sk);
        rest /= sk;
        t.ph_begin = (int)(((unsigned)t.split * (unsigned)p.n_phases) / sk);            // n_phases * split_k < 2^31 (checked at plan time)
        t.ph_end = (int)((((unsigned)t.split + 1u) * (unsigned)p.n_phases) / sk);
    }
    const unsigned nt = rest % (unsigned)p.n_tiles;
    unsigned m = rest / (unsigned)p.n_tiles;
    const unsigned tw = m % (unsigned)p.tiles_w;
    m /= (unsigned)p.tiles_w;
    const unsigned th = m % (unsigned)p.tiles_h;
    m /= (unsigned)p.tiles_h;
    const unsigned td = m % (unsigned)p.tiles_d;
    t.nb = (int)(m / (unsigned)p.tiles_d);
    t.d0 = (int)td * p.TD;
    t.h0 = (int)th * p.TH;
    t.w0 = (int)tw * p.TW;
    t.n0 = (int)nt * p.block_n;
    t.tde = min(p.TD, p.D - t.d0);
    return t;
}

}  // namespace

// One input slab of a 3x3x3 stride-1 phase: 12 MMAs (3 kh x 4 K steps of 16) of N = nblk*BN columns into the nblk adjacent
// accumulators starting at acc0. Everything that depends on (kh, k4) is a compile-time immediate so the single issuing
// thread spends ~4 instructions per tcgen05.mma; with run-time strides it spends ~20 and becomes the kernel's bottleneck
// (r01: 240 instructions per slab at ~7 cycles each vs 12 x 96 tensor-pipe cycles).
template <bool F8, bool ACC>
__device__ __forceinline__ void umma_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc) {
    if (F8) umma_f8_lohi<ACC>(d_tmem, a_lo, b_lo, hi, idesc);
    else umma_f16_lohi<ACC>(d_tmem, a_lo, b_lo, hi, idesc);
}
// (F8: the same smem geometry — 128-byte rows, four 32-byte K steps — read as E5M2 with K = 32 per instruction.)
template <int BN, int TWv, bool F8>
__device__ __forceinline__ void issue_slab_3x3(uint32_t acc0, uint32_t a_lo0, uint32_t b_lo0, uint32_t hi, uint32_t idA,
                                               uint32_t id_old, uint32_t id1, int nold, bool fresh) {
    constexpr uint32_t kKh = (uint32_t)(TWv * 128) >> 4, kTap = (uint32_t)(BN * 128) >> 4;
    if (fresh) {
        // the newest plane's accumulator is overwritten by its first MMA, the older planes accumulate
        if (nold > 0) umma_lohi<F8, true>(acc0, a_lo0, b_lo0, hi, id_old);
        umma_lohi<F8, false>(acc0 + (uint32_t)(nold * BN), a_lo0, b_lo0 + (uint32_t)nold * kTap, hi, id1);
    } else {
        umma_lohi<F8, true>(acc0, a_lo0, b_lo0, hi, idA);
    }
#pragma unroll
    for (int i = 1; i < 12; ++i) {
        const uint32_t kh = (uint32_t)(i >> 2), k4 = (uint32_t)(i & 3);
        umma_lohi<F8, true>(acc0, a_lo0 + kh * kKh + 2u * k4, b_lo0 + kh * 3u * kTap + 2u * k4, hi, idA);
    }
}

__global__ void __launch_bounds__(kConvThreads, 1)
conv3d_igemm_kernel(const __grid_constant__ ConvKernelParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // dynamic smem base is only guaranteed 16 B aligned by the ABI: align manually to 1024 B
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* w_smem = smem;
    uint8_t* s_smem = smem + (size_t)p.w_stages * p.w_stage_bytes;
    SmemCtrl* ctl = reinterpret_cast<SmemCtrl*>(s_smem + (size_t)p.s_stages * p.s_stage_bytes);
    float* stats_sm = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ctl) + kCtlBarrierBytes);   // used iff p.stats
    const int stats_ld = p.stats_ld;     // channels per statistics row (Cout rounded up to 32)
    // plans without alignment slack (p.smem_slack == 0) rely on the 1 KB-aligned dynamic smem base that kernels without
    // static shared memory get in practice; verified here, failing loudly through the error flag instead of corrupting smem
    const bool smem_misaligned = (p.smem_slack == 0) && (smem != smem_raw);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_items = p.NB * p.tiles_d * p.tiles_h * p.tiles_w * p.n_tiles * p.split_k;
    const uint32_t tmem_cols_needed = (uint32_t)(p.acc_sets * p.TD * p.block_n);
    uint32_t tmem_cols = 32;
    while (tmem_cols < tmem_cols_needed) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kMaxWStages; ++i) { mbar_init(&ctl->wfull[i], 1); mbar_init(&ctl->wempty[i], 1); }
        for (int i = 0; i < kMaxSStages; ++i) { mbar_init(&ctl->sfull[i], 1); mbar_init(&ctl->sempty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&ctl->tfull[i], 1); mbar_init(&ctl->tempty[i], 4); }
        ctl->abort_flag = smem_misaligned ? 1 : 0;
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc(&ctl->tmem_base, tmem_cols);
        tmem_relinquish();
    }
    if (warp == 0 && lane == 0) {
        for (int i = 0; i < kConvMaxSrc; ++i) prefetch_tmap(&p.tmA[i]);
        prefetch_tmap(&p.tmB);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = ctl->tmem_base;
    volatile int* abort_flag = &ctl->abort_flag;

    if (warp == 0) {
        // ================================================================ TMA producer (warp-uniform, one elected lane issues)
        int ws = 0, wph = 0, ss = 0, sph = 0;
        bool ok = true;
        for (int wi = blockIdx.x; wi < total_items && ok; wi += gridDim.x) {
            const TileCoord t = decode_tile(p, wi);
            for (int ph = t.ph_begin; ph < t.ph_end && ok; ++ph) {
                const ConvPhase P = p.phases[ph];
                const int ntaps = P.n_kh * P.n_kd;
                ok = mbar_wait(&ctl->wempty[ws], wph ^ 1, abort_flag);
                if (!ok) break;
                if (elect_one()) {
                    mbar_expect_tx(&ctl->wfull[ws], (uint32_t)(ntaps * p.block_n * 128));
                    uint8_t* wdst = w_smem + (size_t)ws * p.w_stage_bytes;
                    for (int tap = 0; tap < ntaps; ++tap)
                        tma_load_2d(wdst + (size_t)tap * p.block_n * 128, &p.tmB, &ctl->wfull[ws],
                                    (P.wtile_base + tap) * 64, t.n0);
                }
                if (++ws == p.w_stages) { ws = 0; wph ^= 1; }

                const int nplanes = t.tde + P.n_kd - 1;
                const uint32_t slab_bytes = (uint32_t)p.slab_rows[P.src] * 128u;
                for (int pl = 0; pl < nplanes && ok; ++pl) {
                    ok = mbar_wait(&ctl->sempty[ss], sph ^ 1, abort_flag);
                    if (!ok) break;
                    if (elect_one()) {
                        mbar_expect_tx(&ctl->sfull[ss], slab_bytes);
                        tma_load_5d(s_smem + (size_t)ss * p.s_stage_bytes, &p.tmA[P.src],
                                    &ctl->sfull[ss], (int)P.c0, t.w0 * p.stride + P.dw,
                                    t.h0 * p.stride + P.dh0, (t.d0 + pl) * p.stride + P.dd0, t.nb);
                    }
                    if (++ss == p.s_stages) { ss = 0; sph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================================================ MMA issuer
        // The whole warp runs this loop with warp-uniform control flow (so the compiler keeps descriptors
        // and addresses in uniform registers); only the tcgen05 instructions themselves are issued by one
        // elected lane. A single divergent thread costs ~25 scalar instructions per MMA (ncu: tensor pipe
        // 23 % busy, issue thread never waiting).
        int ws = 0, wph = 0, ss = 0, sph = 0, as = 0, aph = 0;
        const int max_blk = min(3, 256 / p.block_n);                             // accumulator blocks one MMA may span
        const uint32_t idesc1_h = make_idesc_f16(128, (uint32_t)p.block_n), idesc2_h = make_idesc_f16(128, (uint32_t)(2 * p.block_n)),
                       idesc3_h = make_idesc_f16(128, (uint32_t)(3 * p.block_n));
        const uint32_t idesc1_q = make_idesc_e5m2(128, (uint32_t)p.block_n), idesc2_q = make_idesc_e5m2(128, (uint32_t)(2 * p.block_n)),
                       idesc3_q = make_idesc_e5m2(128, (uint32_t)(3 * p.block_n));
        const uint64_t desc_fixed = make_sw128_desc(0, 1024);   // everything but the start address
        const uint32_t desc_lo = (uint32_t)desc_fixed, desc_hi = (uint32_t)(desc_fixed >> 32);
        const bool fast3 = (p.block_n == 64 || p.block_n == 128) && (p.TW == 16 || p.TW == 8);
        const uint32_t w_base0 = smem_u32(w_smem), s_base0 = smem_u32(s_smem);
        const uint32_t kh_stride16 = (uint32_t)(p.TW * 128) >> 4;             // descriptor units of 16 B
        const uint32_t tap_stride16 = (uint32_t)(p.block_n * 128) >> 4;
        bool ok = true;
        for (int wi = blockIdx.x; wi < total_items && ok; wi += gridDim.x) {
            const TileCoord t = decode_tile(p, wi);
            ok = mbar_wait(&ctl->tempty[as], aph ^ 1, abort_flag);
            if (!ok) break;
            tc_fence_after();
            for (int ph = t.ph_begin; ph < t.ph_end && ok; ++ph) {
                const ConvPhase P = p.phases[ph];
                const int n_kd = P.n_kd, n_kh = P.n_kh;
                const bool f8 = P.f8 != 0;                       // warp-uniform
                const uint32_t idesc1 = f8 ? idesc1_q : idesc1_h, idesc2 = f8 ? idesc2_q : idesc2_h, idesc3 = f8 ? idesc3_q : idesc3_h;
                ok = mbar_wait(&ctl->wfull[ws], wph, abort_flag);
                if (!ok) break;
                const uint32_t w16 = (w_base0 + (uint32_t)(ws * p.w_stage_bytes)) >> 4;
                const int nplanes = t.tde + n_kd - 1;
                for (int pl = 0; pl < nplanes && ok; ++pl) {
                    ok = mbar_wait(&ctl->sfull[ss], sph, abort_flag);
                    if (!ok) break;
                    tc_fence_after();
                    const uint32_t s16 = (s_base0 + (uint32_t)(ss * p.s_stage_bytes)) >> 4;
                    // This slab (input plane pl) feeds output planes d = pl - kd: accumulators d_min..d_max are ADJACENT
                    // column blocks of TMEM and the matching weight tiles (kd = kd_hi..kd_lo) are adjacent row blocks of
                    // the B stage, so one MMA of N = nblk*block_n covers them all (tcgen05.mma has a ~56-cycle floor per
                    // 128xNx16 instruction for N <= 112 and runs at N/2 cycles from N = 128 up: mma_bench.cu).
                    const int d_min = max(0, pl - (n_kd - 1)), d_max = min(t.tde - 1, pl);
                    const int nblk = d_max - d_min + 1, kd_hi = pl - d_min;
                    const bool fresh = (ph == t.ph_begin) && (d_max == pl);   // plane pl's accumulator is first touched here
                    if (elect_one()) {
                        const uint32_t acc0 = tmem_base + (uint32_t)((as * p.TD + d_min) * p.block_n);
                        const uint32_t wblk0 = (uint32_t)(n_kd - 1 - kd_hi);
                        const int nold0 = fresh ? nblk - 1 : nblk;
                        if (n_kh == 3 && n_kd == 3 && nblk <= max_blk && fast3) {
                            const uint32_t idA = nblk == 1 ? idesc1 : (nblk == 2 ? idesc2 : idesc3);
                            const int nold = nblk - 1;
                            const uint32_t id_old = nold == 1 ? idesc1 : idesc2;
                            const uint32_t a_lo0 = desc_lo | (s16 & 0x3FFFu);
                            const uint32_t b_lo0 = desc_lo | ((w16 + wblk0 * tap_stride16) & 0x3FFFu);
                            if (f8) {
                                if (p.block_n == 64) {
                                    if (p.TW == 16) issue_slab_3x3<64, 16, true>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                    else issue_slab_3x3<64, 8, true>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                } else {
                                    if (p.TW == 16) issue_slab_3x3<128, 16, true>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                    else issue_slab_3x3<128, 8, true>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                }
                            } else if (p.block_n == 64) {
                                if (p.TW == 16) issue_slab_3x3<64, 16, false>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                else issue_slab_3x3<64, 8, false>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                            } else {
                                if (p.TW == 16) issue_slab_3x3<128, 16, false>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                                else issue_slab_3x3<128, 8, false>(acc0, a_lo0, b_lo0, desc_hi, idA, id_old, idesc1, nold, fresh);
                            }
                        } else
                        for (int kh = 0; kh < n_kh; ++kh) {
                            const uint32_t a16 = s16 + (uint32_t)kh * kh_stride16;
                            const uint32_t b16 = w16 + ((uint32_t)kh * (uint32_t)n_kd + wblk0) * tap_stride16;
#pragma unroll
                            for (int k4 = 0; k4 < 4; ++k4) {
                                const uint64_t da = desc_fixed | (uint64_t)((a16 + 2u * k4) & 0x3FFFu);
                                const bool split_new = fresh && kh == 0 && k4 == 0;
                                const int nold = split_new ? nold0 : nblk;
                                for (int b = 0; b < nold; b += max_blk) {
                                    const int cnt = min(max_blk, nold - b);
                                    const uint32_t idn = (cnt == 1) ? idesc1 : (cnt == 2 ? idesc2 : idesc3);
                                    const uint64_t db = desc_fixed | (uint64_t)((b16 + (uint32_t)b * tap_stride16 + 2u * k4) & 0x3FFFu);
                                    if (f8) umma_f8(acc0 + (uint32_t)(b * p.block_n), da, db, idn, 1u);
                                    else umma_f16(acc0 + (uint32_t)(b * p.block_n), da, db, idn, 1u);
                                }
                                if (split_new) {
                                    const uint64_t db = desc_fixed | (uint64_t)((b16 + (uint32_t)(nblk - 1) * tap_stride16 + 2u * k4) & 0x3FFFu);
                                    if (f8) umma_f8(acc0 + (uint32_t)((nblk - 1) * p.block_n), da, db, idesc1, 0u);
                                    else umma_f16(acc0 + (uint32_t)((nblk - 1) * p.block_n), da, db, idesc1, 0u);
                                }
                            }
                        }
                        umma_commit(&ctl->sempty[ss]);        // slab slot free once these MMAs retire
                    }
                    if (++ss == p.s_stages) { ss = 0; sph ^= 1; }
                }
                if (elect_one()) umma_commit(&ctl->wempty[ws]);
                if (++ws == p.w_stages) { ws = 0; wph ^= 1; }
            }
            if (elect_one()) umma_commit(&ctl->tfull[as]);            // accumulators complete
            __syncwarp();
            if (++as == p.acc_sets) { as = 0; aph ^= 1; }
        }
    } else {
        // ================================================================ epilogue (warps 2..5)
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int r = q * 32 + lane;            // accumulator row = voxel inside the plane tile
        const int th = r / p.TW, tw = r % p.TW;
        int as = 0, aph = 0;
        bool ok = true;
        const long long DHW = (long long)p.D * p.H * p.W;
        const bool do_stats = p.stats != nullptr;
        float* my_stats = stats_sm + (size_t)(warp - 2) * 2 * stats_ld;
        const int et = threadIdx.x - 64;        // 0..127 among the epilogue threads
        int stats_nb = -1;
        if (do_stats) {
            for (int i = lane; i < 2 * stats_ld; i += 32) my_stats[i] = 0.f;
            __syncwarp();
        }
        auto flush_stats = [&](int nb) {
            // all 4 epilogue warps: fold the warp-private partial sums into the global fp64 accumulators
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int ch = et; ch < p.Cout; ch += 128) {
                float s = 0.f, qq = 0.f;
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    s += stats_sm[(size_t)w * 2 * stats_ld + ch];
                    qq += stats_sm[(size_t)w * 2 * stats_ld + stats_ld + ch];
                }
                atomicAdd(p.stats + ((size_t)nb * p.Cout + ch) * 2, (double)s);
                atomicAdd(p.stats + ((size_t)nb * p.Cout + ch) * 2 + 1, (double)qq);
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int i = lane; i < 2 * stats_ld; i += 32) my_stats[i] = 0.f;
            __syncwarp();
        };
        // f[0..15] = final values of 16 channels of this thread's voxel row (zero where invalid)
        auto add_stats16 = [&](float (&f)[16], int ch0) {
            float sq[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) sq[j] = f[j] * f[j];
            const float s1 = warp_colsum16(f, lane);
            const float s2 = warp_colsum16(sq, lane);
            const int chn = ch0 + stats_channel_of_lane(lane);
            if ((lane & 1) == 0 && chn < p.Cout) {
                my_stats[chn] += s1;
                my_stats[stats_ld + chn] += s2;
            }
            __syncwarp();
        };
        const bool wide_ok = !p.out_planar && ((p.out_ld & 3) == 0) && ((p.out_c0 & 3) == 0);
        // 256-bit accesses need 32-byte aligned rows (cudaMalloc'ed bases are 256-byte aligned)
        const bool wide8_ok = wide_ok && ((p.out_ld & 7) == 0) && ((p.out_c0 & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 31) == 0) &&
                              (p.residual == nullptr || (reinterpret_cast<uintptr_t>(p.residual) & 31) == 0);
        for (int wi = blockIdx.x; wi < total_items && ok; wi += gridDim.x) {
            const TileCoord t = decode_tile(p, wi);
            ok = mbar_wait(&ctl->tfull[as], aph, abort_flag);
            if (!ok) break;
            tc_fence_after();
            if (do_stats && stats_nb != t.nb) {
                if (stats_nb >= 0) flush_stats(stats_nb);
                stats_nb = t.nb;
            }
            const int hh = t.h0 + th, ww = t.w0 + tw;
            const bool row_ok = (hh < p.H) && (ww < p.W);
            const bool first_split = (t.split == 0);
            // ---- wide path: 32-channel chunks, chunk-outer / plane-inner, two planes in flight. One warp per scheduler means
            // nothing hides latency but the warp's own ILP, so both TMEM loads and all residual loads are issued before
            // the first use. Per-channel statistics are accumulated per thread over the tile's planes and reduced across
            // the warp ONCE per (tile, chunk): the per-plane shuffle reduction cost 10 % of a 64->64 conv (r01) and its
            // 250 shuffles per plane competed with the MMA issuer for the MIO queue.
            int c_wide = 0;
            if (wide_ok) {
                const bool use_bias = first_split && p.bias != nullptr;
                const bool use_res = row_ok && first_split && p.residual != nullptr;
                const long long plane_ld = (long long)p.H * p.W * p.out_ld;
                for (; c_wide + 32 <= p.block_n && t.n0 + c_wide + 32 <= p.Cout; c_wide += 32) {
                    const int ch0 = t.n0 + c_wide;
                    float cs[32], cq[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) { cs[j] = 0.f; cq[j] = 0.f; }
                    auto finish = [&](uint32_t (&v)[32], float4 (&r)[8], long long base) {
                        float f[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                        if (use_bias) {
                            const float4* bp = reinterpret_cast<const float4*>(p.bias + ch0);
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 b = __ldg(bp + j);
                                f[4 * j + 0] += b.x; f[4 * j + 1] += b.y; f[4 * j + 2] += b.z; f[4 * j + 3] += b.w;
                            }
                        }
                        if (use_res) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                f[4 * j + 0] += r[j].x; f[4 * j + 1] += r[j].y; f[4 * j + 2] += r[j].z; f[4 * j + 3] += r[j].w;
                            }
                        }
                        if (row_ok) {
                            if (p.atomic_out) {
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    red_add_v4(p.out + base + 4 * j, f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                            } else if (wide8_ok) {
#pragma unroll
                                for (int j = 0; j < 4; ++j) st_global_v8(p.out + base + 8 * j, f + 8 * j);    // one full sector per store
                            } else {
                                float4* op = reinterpret_cast<float4*>(p.out + base);
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                            }
                            if (do_stats) {
#pragma unroll
                                for (int j = 0; j < 32; ++j) { cs[j] += f[j]; cq[j] = fmaf(f[j], f[j], cq[j]); }
                            }
                        }
                    };
                    for (int d = 0; d < t.tde; d += 2) {
                        const bool two = d + 1 < t.tde;                 // warp-uniform
                        const uint32_t acc0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((as * p.TD + d) * p.block_n + c_wide);
                        uint32_t v0[32], v1[32];
                        tmem_ld32(acc0, v0);
                        if (two) tmem_ld32(acc0 + (uint32_t)p.block_n, v1);
                        const long long base0 = ((long long)t.nb * DHW + ((long long)(t.d0 + d) * p.H + hh) * p.W + ww) * p.out_ld + p.out_c0 + ch0;
                        float4 r0[8], r1[8];
                        if (use_res) {
                            if (wide8_ok) {
#pragma unroll
                                for (int j = 0; j < 4; ++j) ld_global_nc_v8(p.residual + base0 + 8 * j, reinterpret_cast<float*>(&r0[2 * j]));
                                if (two) {
#pragma unroll
                                    for (int j = 0; j < 4; ++j)
                                        ld_global_nc_v8(p.residual + base0 + plane_ld + 8 * j, reinterpret_cast<float*>(&r1[2 * j]));
                                }
                            } else {
                                const float4* rp = reinterpret_cast<const float4*>(p.residual + base0);
#pragma unroll
                                for (int j = 0; j < 8; ++j) r0[j] = __ldg(rp + j);
                                if (two) {
                                    const float4* rq = reinterpret_cast<const float4*>(p.residual + base0 + plane_ld);
#pragma unroll
                                    for (int j = 0; j < 8; ++j) r1[j] = __ldg(rq + j);
                                }
                            }
                        }
                        tmem_ld_wait();
                        finish(v0, r0, base0);
                        if (two) finish(v1, r1, base0 + plane_ld);
                    }
                    if (do_stats) {
                        const float s1 = warp_colsum32(cs, lane);       // lane l ends up with channel ch0 + l
                        const float s2 = warp_colsum32(cq, lane);
                        my_stats[ch0 + lane] += s1;
                        my_stats[stats_ld + ch0 + lane] += s2;
                        __syncwarp();
                    }
                }
            }
            for (int d = 0; d < t.tde; ++d) {
                const long long vox = ((long long)(t.d0 + d) * p.H + hh) * p.W + ww;   // inside batch item
                const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16) +
                                     (uint32_t)((as * p.TD + d) * p.block_n);
                int c = c_wide;
                // ---- generic path: 16 channels per step (ragged Cout, planar outputs, narrow tiles)
                for (; c < p.block_n; c += 16) {
                    uint32_t v[16];
                    tmem_ld16(acc + (uint32_t)c, v);
                    tmem_ld_wait();
                    const int ch0 = t.n0 + c;
                    if (ch0 >= p.Cout) continue;              // warp-uniform
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
                    if (first_split && p.bias) {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (ch0 + j < p.Cout) f[j] += __ldg(p.bias + ch0 + j);
                    }
                    if (p.out_planar) {
                        if (row_ok) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                if (ch0 + j >= p.Cout) break;
                                const long long idx = ((long long)t.nb * p.Cout + ch0 + j) * DHW + vox;
                                float val = f[j];
                                if (first_split && p.residual) val += p.residual[idx];
                                if (p.atomic_out) atomicAdd(p.out + idx, val);
                                else p.out[idx] = val;
                            }
                        }
                    } else {
                        const long long base = ((long long)t.nb * DHW + vox) * p.out_ld + p.out_c0 + ch0;
                        const bool vec = (ch0 + 16 <= p.Cout) && ((base & 3) == 0);
                        if (row_ok && first_split && p.residual) {
                            if (vec) {
                                const float4* rp = reinterpret_cast<const float4*>(p.residual + base);
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    const float4 rv = __ldg(rp + j);
                                    f[4 * j + 0] += rv.x; f[4 * j + 1] += rv.y;
                                    f[4 * j + 2] += rv.z; f[4 * j + 3] += rv.w;
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < 16; ++j)
                                    if (ch0 + j < p.Cout) f[j] += p.residual[base + j];
                            }
                        }
                        if (row_ok) {
                            if (vec) {
                                if (p.atomic_out) {
#pragma unroll
                                    for (int j = 0; j < 4; ++j)
                                        red_add_v4(p.out + base + 4 * j, f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                                } else {
                                    float4* op = reinterpret_cast<float4*>(p.out + base);
#pragma unroll
                                    for (int j = 0; j < 4; ++j)
                                        op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < 16; ++j) {
                                    if (ch0 + j >= p.Cout) break;
                                    if (p.atomic_out) atomicAdd(p.out + base + j, f[j]);
                                    else p.out[base + j] = f[j];
                                }
                            }
                        }
                        if (do_stats) {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (!row_ok || ch0 + j >= p.Cout) f[j] = 0.f;
                            add_stats16(f, ch0);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ctl->tempty[as]);
            if (++as == p.acc_sets) { as = 0; aph ^= 1; }
        }
        if (do_stats && stats_nb >= 0 && ok) flush_stats(stats_nb);
    }

    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0 && ctl->abort_flag && p.err_flag) atomicExch(p.err_flag, 1 + (int)blockIdx.x);
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// =====================================================================================  host side

int conv_k_total(const ConvDesc& d) {
    int k = 0;
    for (const auto& s : d.segs) k += s.ks * s.ks * s.ks * d.srcs[s.src].C;
    return k;
}

// Source slots: a (source, kernel-size class) pair needs its own tensor map because the TMA box
// height differs (TH+2 rows for in-slab kh taps vs TH rows).  Slot i of the returned table is used
// as ConvPhase::src.
struct SrcSlot { int src; int n_kh; };

static std::vector<SrcSlot> conv_src_slots(const ConvDesc& d) {
    std::vector<SrcSlot> slots;
    for (const auto& s : d.segs) {
        const int n_kh = (s.ks == 3 && d.stride == 1) ? 3 : 1;
        bool found = false;
        for (const auto& sl : slots) found |= (sl.src == s.src && sl.n_kh == n_kh);
        if (!found) slots.push_back({s.src, n_kh});
    }
    return slots;
}

static int conv_slot_of(const std::vector<SrcSlot>& slots, int src, int n_kh) {
    for (size_t i = 0; i < slots.size(); ++i)
        if (slots[i].src == src && slots[i].n_kh == n_kh) return (int)i;
    return -1;
}

std::vector<ConvPhase> conv_build_phases(const ConvDesc& d) {
    std::vector<ConvPhase> ph;
    const auto slots = conv_src_slots(d);
    int wtile = 0;
    for (const auto& s : d.segs) {
        const ConvSrc& src = d.srcs[s.src];
        const int chunks = src.C / 64;
        if (s.ks == 1) {
            for (int c = 0; c < chunks; ++c) {
                ConvPhase P{};
                P.src = (int8_t)conv_slot_of(slots, s.src, 1);
                P.dw = 0; P.dh0 = 0; P.dd0 = 0; P.n_kh = 1; P.n_kd = 1;
                P.c0 = (int16_t)(c * 64); P.wtile_base = wtile; wtile += 1; P.f8 = s.f8;
                ph.push_back(P);
            }
        } else if (d.stride == 1) {
            for (int c = 0; c < chunks; ++c)
                for (int kw = 0; kw < 3; ++kw) {
                    ConvPhase P{};
                    P.src = (int8_t)conv_slot_of(slots, s.src, 3);
                    P.dw = (int8_t)(kw - 1); P.dh0 = -1; P.dd0 = -1; P.n_kh = 3; P.n_kd = 3;
                    P.c0 = (int16_t)(c * 64); P.wtile_base = wtile; wtile += 9; P.f8 = s.f8;
                    ph.push_back(P);
                }
        } else {
            for (int c = 0; c < chunks; ++c)
                for (int kw = 0; kw < 3; ++kw)
                    for (int kh = 0; kh < 3; ++kh)
                        for (int kd = 0; kd < 3; ++kd) {
                            ConvPhase P{};
                            P.src = (int8_t)conv_slot_of(slots, s.src, 1);
                            P.dw = (int8_t)(kw - 1); P.dh0 = (int8_t)(kh - 1); P.dd0 = (int8_t)(kd - 1);
                            P.n_kh = 1; P.n_kd = 1;
                            P.c0 = (int16_t)(c * 64); P.wtile_base = wtile; wtile += 1; P.f8 = s.f8;
                            ph.push_back(P);
                        }
        }
    }
    return ph;
}

void conv_pack_weights(const ConvDesc& d, const std::vector<const float*>& seg_weights,
                       const std::vector<int>& seg_cin_real, std::vector<__half>& packed) {
    const int K = conv_k_total(d);
    packed.assign((size_t)d.Cout_pad * K, __float2half(0.f));
    int wtile = 0;
    for (size_t si = 0; si < d.segs.size(); ++si) {
        const auto& s = d.segs[si];
        const ConvSrc& src = d.srcs[s.src];
        const int chunks = src.C / 64;
        const int cin = seg_cin_real[si];
        const int ks = s.ks, kv = ks * ks * ks;
        const float* w = seg_weights[si];   // [Cout][cin][kd][kh][kw]
        const float up = (float)(1 << kF8Shift), down = 1.0f / up;
        auto e5m2 = [](float v) { return (uint8_t)__nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E5M2); };
        auto put = [&](int tile, int c, int kd, int kh, int kw) {
            for (int co = 0; co < d.Cout; ++co) {
                // an f8 tile is 128 bytes per row: [e5m2(w / 2^s) x 64 | e5m2((w - fp16(w)) * 2^s) x 64]
                uint8_t* row8 = reinterpret_cast<uint8_t*>(&packed[(size_t)co * K + (size_t)tile * 64]);
                for (int cil = 0; cil < 64; ++cil) {
                    const int ci = c * 64 + cil;
                    if (ci >= cin) continue;
                    float v = w[((size_t)co * cin + ci) * kv + (kd * ks + kh) * ks + kw];
                    if (s.f8) {
                        row8[cil] = e5m2(v * down);
                        row8[64 + cil] = e5m2((v - __half2float(__float2half(v))) * up);
                        continue;
                    }
                    if (s.wlo) v = v - __half2float(__float2half(v));
                    packed[(size_t)co * K + (size_t)tile * 64 + cil] = __float2half(v);
                }
            }
        };
        if (ks == 1) {
            for (int c = 0; c < chunks; ++c) put(wtile++, c, 0, 0, 0);
        } else if (d.stride == 1) {
            for (int c = 0; c < chunks; ++c)
                for (int kw = 0; kw < 3; ++kw) {
                    // tile order inside the phase: kh major, then kd = 2,1,0 — the three kd tiles of one kh are
                    // contiguous so that ONE MMA with N = 3*block_n feeds the accumulators of output planes
                    // p-2, p-1, p (which are adjacent TMEM column blocks)
                    for (int kd = 0; kd < 3; ++kd)
                        for (int kh = 0; kh < 3; ++kh) put(wtile + kh * 3 + (2 - kd), c, kd, kh, kw);
                    wtile += 9;
                }
        } else {
            for (int c = 0; c < chunks; ++c)
                for (int kw = 0; kw < 3; ++kw)
                    for (int kh = 0; kh < 3; ++kh)
                        for (int kd = 0; kd < 3; ++kd) put(wtile++, c, kd, kh, kw);
        }
    }
}

// ---- driver entry point for tensor-map encoding (no link-time dependency on libcuda)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}


static int encode_a_maps(const ConvDesc& d, ConvKernelParams& p, PFN_encodeTiled enc, char* err, int errlen) {
    const auto slots = conv_src_slots(d);
    for (size_t i = 0; i < slots.size(); ++i) {
        const ConvSrc& s = d.srcs[slots[i].src];
        cuuint64_t gdim[5] = {(cuuint64_t)s.C, (cuuint64_t)s.Win, (cuuint64_t)s.Hin, (cuuint64_t)s.Din, (cuuint64_t)d.NB};
        cuuint64_t gstr[4] = {(cuuint64_t)s.C * 2, (cuuint64_t)s.Win * s.C * 2,
                              (cuuint64_t)s.Hin * s.Win * s.C * 2, (cuuint64_t)s.Din * s.Hin * s.Win * s.C * 2};
        cuuint32_t box[5] = {64, (cuuint32_t)(p.TW * d.stride), (cuuint32_t)((p.TH + slots[i].n_kh - 1) * d.stride), 1, 1};
        cuuint32_t estr[5] = {1, (cuuint32_t)d.stride, (cuuint32_t)d.stride, 1, 1};
        CUresult r = enc(&p.tmA[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)s.ptr, gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { snprintf(err, errlen, "cuTensorMapEncodeTiled(A%zu) failed: %d", i, (int)r); return 1; }
    }
    for (size_t i = slots.size(); i < (size_t)kConvMaxSrc; ++i) p.tmA[i] = p.tmA[0];
    return 0;
}

int conv_plan_retarget(const ConvDesc& d, ConvPlan& plan, char* err, int errlen) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) { snprintf(err, errlen, "cuTensorMapEncodeTiled unavailable"); return 1; }
    return encode_a_maps(d, plan.p, enc, err, errlen);
}

int conv_plan_create(const ConvDesc& d, int* d_err_flag, ConvPlan& plan, char* err, int errlen) {
    auto fail = [&](const char* m) { snprintf(err, errlen, "conv_plan_create: %s", m); return 1; };
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return fail("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    if (d.srcs.empty() || d.segs.empty()) return fail("no sources/segments");
    for (const auto& s : d.srcs)
        if (s.C % 64) return fail("source channels must be a multiple of 64");
    if (d.Cout_pad % 16 || d.Cout_pad < d.Cout) return fail("Cout_pad must be a multiple of 16 >= Cout");

    ConvKernelParams& p = plan.p;
    memset(&p, 0, sizeof(p));
    p.NB = d.NB; p.D = d.D; p.H = d.H; p.W = d.W; p.stride = d.stride;
    p.TW = (d.W >= 16) ? 16 : 8;
    p.TH = 128 / p.TW;
    p.Cout = d.Cout;

    const auto slots = conv_src_slots(d);
    if ((int)slots.size() > kConvMaxSrc) return fail("too many (source, tap-class) slots");
    const std::vector<ConvPhase> phases = conv_build_phases(d);
    p.n_phases = (int)phases.size();
    int max_taps = 1;
    bool any3 = false;
    for (const auto& P : phases) { max_taps = std::max(max_taps, P.n_kh * P.n_kd); any3 |= (P.n_kh == 3); }

    // N tile
    int bn = d.block_n;
    if (bn == 0) bn = any3 ? std::min(64, d.Cout_pad) : std::min(256, d.Cout_pad);
    if (bn % 16 || bn > 256 || bn < 16) return fail("bad block_n");
    p.block_n = bn;
    p.n_tiles = (d.Cout_pad + bn - 1) / bn;

    // TD: accumulators per set
    int td = d.td ? d.td : std::min(4, 512 / (2 * bn));
    td = std::max(1, std::min(td, d.D));
    if (!any3) td = std::min(td, 2);    // no plane re-use without kd taps: smaller tiles, more CTAs
    if (!d.td && td > 1) {
        // wave quantisation: a persistent grid of `sms` CTAs finishes in ceil(tiles/sms) rounds; prefer the
        // plane count with the better last-round fill (64^3: TD=4 -> 512 tiles = 3.46 rounds, TD=2 -> 6.92)
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        auto fill = [&](int t) {
            const long long tiles = (long long)d.NB * ((d.W + p.TW - 1) / p.TW) * ((d.H + p.TH - 1) / p.TH) * ((d.D + t - 1) / t) *
                                    ((d.Cout_pad + bn - 1) / bn);
            const long long rounds = (tiles + sms - 1) / sms;
            return (double)tiles / (double)(rounds * sms) * (t == td ? 1.0 : 0.93);   // halving TD costs ~7 % more slab traffic
        };
        if (fill(td / 2) > fill(td)) td /= 2;
    }
    p.TD = td;
    p.acc_sets = (2 * td * bn <= 512) ? 2 : 1;
    if (td * bn > 512) return fail("TD*block_n exceeds TMEM");
    p.tiles_w = (d.W + p.TW - 1) / p.TW;
    p.tiles_h = (d.H + p.TH - 1) / p.TH;
    p.tiles_d = (d.D + p.TD - 1) / p.TD;

    // split-K
    const int items = d.NB * p.tiles_w * p.tiles_h * p.tiles_d * p.n_tiles;
    int split = d.split_k;
    if (split <= 0) {
        split = 1;
        while (items * split < 120 && split * 2 <= p.n_phases && split < 64) split *= 2;
    }
    split = std::max(1, std::min(split, p.n_phases));
    if ((long long)p.n_phases * (split + 1) >= (1ll << 31)) return fail("too many phases for the split-K bookkeeping");
    p.split_k = split;
    p.atomic_out = split > 1;
    plan.needs_zero = split > 1;

    // shared memory plan
    for (size_t i = 0; i < slots.size(); ++i) p.slab_rows[i] = p.TW * (p.TH + slots[i].n_kh - 1);
    int max_rows = 0;
    for (size_t i = 0; i < slots.size(); ++i) max_rows = std::max(max_rows, p.slab_rows[i]);
    p.w_stage_bytes = max_taps * bn * 128;
    p.s_stage_bytes = max_rows * 128;
    // control block: barriers + per-warp statistics rows; the 1 KB alignment slack is dropped when exactly that buys
    // another slab stage (the kernel then verifies the base alignment itself)
    plan.fused_stats = d.stats != nullptr && split == 1 && d.Cout <= kStatsMaxC && !d.out_planar;
    p.stats_ld = (d.Cout + 31) / 32 * 32;
    const int stats_bytes = plan.fused_stats ? 4 * 2 * p.stats_ld * 4 : 0;
    const int ctl_core = kCtlBarrierBytes + stats_bytes;
    auto plan_stages = [&](int slack, int& ws, int& ss) {
        const int avail = 227 * 1024 - ctl_core - slack;
        ws = (2 * p.w_stage_bytes + 2 * p.s_stage_bytes <= avail) ? 2 : 1;
        if (ws * p.w_stage_bytes + 2 * p.s_stage_bytes > avail) return false;
        ss = std::min(std::min(kMaxSStages, 6), (avail - ws * p.w_stage_bytes) / p.s_stage_bytes);
        return true;
    };
    int ws1 = 0, ss1 = 0, ws0 = 0, ss0 = 0;
    const bool ok1 = plan_stages(1024, ws1, ss1), ok0 = plan_stages(0, ws0, ss0);
    if (!ok0) return fail("tile does not fit in shared memory");
    if (ok1 && ws1 >= ws0 && ss1 >= ss0) { p.smem_slack = 1024; p.w_stages = ws1; p.s_stages = ss1; }
    else { p.smem_slack = 0; p.w_stages = ws0; p.s_stages = ss0; }
    const int ctl_bytes = ctl_core + p.smem_slack;
    plan.smem_bytes = p.w_stages * p.w_stage_bytes + p.s_stages * p.s_stage_bytes + ctl_bytes;

    if (encode_a_maps(d, p, enc, err, errlen)) return 1;
    {
        const int K = conv_k_total(d);
        cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)d.Cout_pad};
        cuuint64_t gstr[1] = {(cuuint64_t)K * 2};
        cuuint32_t box[2] = {64, (cuuint32_t)std::min(bn, d.Cout_pad)};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = enc(&p.tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)d.weights, gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { snprintf(err, errlen, "cuTensorMapEncodeTiled(B) failed: %d", (int)r); return 1; }
    }

    if (cudaMalloc(&plan.d_phases, phases.size() * sizeof(ConvPhase)) != cudaSuccess) return fail("cudaMalloc phases");
    cudaMemcpy(plan.d_phases, phases.data(), phases.size() * sizeof(ConvPhase), cudaMemcpyHostToDevice);
    p.phases = plan.d_phases;

    p.bias = d.bias; p.residual = d.residual; p.out = d.out;
    p.out_ld = d.out_ld ? d.out_ld : d.Cout; p.out_c0 = d.out_c0; p.out_planar = d.out_planar;
    p.err_flag = d_err_flag;
    p.stats = plan.fused_stats ? d.stats : nullptr;
    plan.out_bytes = d.out_planar ? (size_t)d.NB * d.Cout * d.D * d.H * d.W * 4
                                  : (size_t)d.NB * d.D * d.H * d.W * p.out_ld * 4;

    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    plan.grid = std::min(items * split, sms);

    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(conv3d_igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
            return fail("cudaFuncSetAttribute(max dynamic smem)");
        attr_set = true;
    }
    return 0;
}

void conv_plan_destroy(ConvPlan& plan) {
    if (plan.d_phases) cudaFree(plan.d_phases);
    plan.d_phases = nullptr;
}

int conv_plan_launch(const ConvPlan& plan, cudaStream_t stream) {
    if (plan.needs_zero) {
        // split-K accumulates with red.add: only the channel slice written by this conv may be
        // cleared when out_ld > Cout, so callers with sliced outputs must not use split-K.
        cudaMemsetAsync(plan.p.out, 0, plan.out_bytes, stream);
    }
    conv3d_igemm_kernel<<<plan.grid, kConvThreads, plan.smem_bytes, stream>>>(plan.p);
    return (int)cudaGetLastError();
}

}  // namespace pixie
