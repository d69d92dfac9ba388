// Implicit-GEMM 3-D convolution on tcgen05 tensor cores (sm_100a), host-side description.
//
// Replaces, for the U-Net path, every torch.nn.Conv3d / Conv1d call of the reference
// (third_party/Wavelet-Generation/models/module/diffusion_network.py:69-71, 91, 208-209, 571-581,
//  663, 674, 687-694, 776, 872) with one persistent, warp-specialised kernel.
//
// Data layout: activations are NDHWC fp16 (the layout voxelize.py:86,111 already writes to disk),
// weights are packed per "phase" (see below) as fp16 [Cout_pad][K] with K contiguous, accumulation
// is fp32 in TMEM, outputs are fp32 (NDHWC, or NCDHW planar for the network head).
//
// GEMM view: M = output voxels (tile = TD planes x TH x TW, TH*TW = 128 rows per accumulator),
// N = output channels (BLOCK_N <= 256 per CTA tile), K = taps x input channels in chunks of 64.
//
// The K loop is organised in PHASES so that shared memory, not L2, serves the tap re-use:
//   phase = (source tensor, 64-channel chunk, kw)  for 3x3x3 stride-1 convolutions.
// For one phase the CTA keeps the 9 (kd,kh) weight tiles resident and marches over the TD+2 input
// planes of its tile; every plane slab ((TH+2) x TW voxels x 64 ch, loaded once by TMA with
// zero-fill for the padding) feeds up to 9 MMAs: kh shifts are 1024 B-aligned row offsets into the
// slab (TW is a multiple of 8 rows of 128 B), kd shifts select which of the TD accumulators the MMA
// targets. kw needs its own slab copy because a one-voxel shift along w is not a multiple of the
// 8-row swizzle atom.  1x1x1 convolutions (projector, ResBlock skip, attention qkv/proj) and
// stride-2 taps are phases with n_kh = n_kd = 1.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <vector>

namespace pixie {

constexpr int kConvMaxSrc = 8;
constexpr int kF8Shift = 6;        // power-of-two rebalancing between the E5M2 operands (see ConvDesc::Seg)
constexpr int kConvThreads = 192;  // warp0 TMA, warp1 MMA, warps2-5 epilogue

struct ConvPhase {        // 16 bytes, lives in global memory
    int8_t src;           // tensor-map index of the activation source
    int8_t dw;            // w offset of the slab origin relative to w0*stride
    int8_t dh0;           // h offset
    int8_t dd0;           // d offset
    int8_t n_kh;          // 1 or 3: kh taps served by row offsets inside one slab
    int8_t n_kd;          // 1 or 3: kd taps served by plane marching
    int16_t c0;           // first channel of the 64-channel chunk inside the source
    int32_t wtile_base;   // index of this phase's first weight tile (64 K-columns each)
    int32_t f8;           // 1: operands are E5M2 bytes (128 per row instead of 64 halfs), issued as kind::f8f6f4
};
static_assert(sizeof(ConvPhase) == 16, "ConvPhase layout");

struct ConvKernelParams {
    CUtensorMap tmA[kConvMaxSrc];
    CUtensorMap tmB;
    const ConvPhase* phases;
    int n_phases;
    int split_k;          // phases are divided into split_k contiguous ranges
    // output geometry
    int NB, D, H, W;      // batch and OUTPUT spatial size
    int stride;           // 1 or 2
    int TW, TH, TD;       // tile: TH*TW == 128
    int tiles_w, tiles_h, tiles_d;
    int Cout;             // real output channels
    int block_n;          // N tile (multiple of 16, <= 256)
    int n_tiles;          // ceil(Cout / block_n)
    // shared-memory plan
    int w_stage_bytes, w_stages;   // weight stages (all taps of one phase)
    int s_stage_bytes, s_stages;   // slab stages
    int slab_rows[kConvMaxSrc];    // rows per slab for each source (TW * (TH + n_kh - 1))
    int acc_sets;                  // 1 or 2 accumulator sets in TMEM
    // epilogue
    const float* bias;       // [Cout] or nullptr
    const float* residual;   // same layout as out, or nullptr
    float* out;              // fp32
    int out_ld;              // channel stride of an NDHWC row (>= Cout)
    int out_c0;              // channel offset inside the row
    int out_planar;          // 1: write NCDHW (out[(n*Cout+c)*DHW + vox])
    int atomic_out;          // 1: red.add into out (split_k > 1); out must be pre-zeroed
    double* stats;           // optional [NB][Cout][2] = (sum, sum of squares) of the outputs over voxels,
                             // accumulated by the epilogue (fused LayerNorm/GroupNorm statistics); or nullptr
    int stats_ld;            // floats per statistics row in shared memory (Cout rounded up to 32)
    int smem_slack;          // bytes reserved for aligning the dynamic smem base to 1 KB (0: the base must already be aligned)
    int* err_flag;           // device int, set non-zero on pipeline timeout
};

// One activation source of a convolution.
struct ConvSrc {
    const __half* ptr;    // NDHWC fp16, [NB][Din][Hin][Win][C]
    int C;                // channels (multiple of 64)
    int Din, Hin, Win;
};

// Host description of one convolution launch.
struct ConvDesc {
    int NB = 1;
    int D = 0, H = 0, W = 0;   // output size
    int stride = 1;
    int Cout = 0;
    // K segments: each segment is (source, kernel size 1 or 3) over all of the source's channels.
    // wlo = 1 packs the fp16 rounding residual of the weights (w - fp16(w)) for split-precision mode.
    // f8 = 1: an E5M2 correction segment (tensor-core rate 2x fp16). Its source rows hold, per 64-channel chunk, 64 bytes
    // e5m2(a_lo * 2^kF8Shift) followed by 64 bytes e5m2(a * 2^-kF8Shift); its weight rows hold e5m2(w * 2^-kF8Shift) followed by
    // e5m2(w_lo * 2^kF8Shift), so one K = 128-byte chunk accumulates a_lo*w + a*w_lo — the two first-order terms a single
    // fp16 pass loses — into the same fp32 accumulator (`C` of such a source counts 2-byte units like the fp16 ones).
    struct Seg { int src; int ks; int wlo = 0; int f8 = 0; };
    std::vector<ConvSrc> srcs;
    std::vector<Seg> segs;
    const __half* weights = nullptr;   // packed by pack_conv_weights(), [Cout_pad][K_total]
    int Cout_pad = 0;                  // rows in the packed weight matrix (multiple of 16)
    const float* bias = nullptr;
    const float* residual = nullptr;
    float* out = nullptr;
    int out_ld = 0, out_c0 = 0, out_planar = 0;
    double* stats = nullptr;           // request fused output statistics (honoured iff plan.fused_stats)
    int split_k = 1;                   // >1 => atomics into pre-zeroed out
    int block_n = 0;                   // 0 = choose
    int td = 0;                        // 0 = choose
};

// K_total (in elements) of a ConvDesc: sum over segments of ks^3 * C.
int conv_k_total(const ConvDesc& d);

// Builds the phase table for `d` (host vector).
std::vector<ConvPhase> conv_build_phases(const ConvDesc& d);

// Packs torch-layout weights [Cout][Cin_seg][kd][kh][kw] (fp32, one tensor per segment) into the
// phase-ordered fp16 matrix [Cout_pad][K_total] expected by the kernel (host memory).
void conv_pack_weights(const ConvDesc& d, const std::vector<const float*>& seg_weights,
                       const std::vector<int>& seg_cin_real, std::vector<__half>& packed);

// A prepared launch: tensor maps encoded, phase table uploaded.
struct ConvPlan {
    ConvKernelParams p{};
    ConvPhase* d_phases = nullptr;
    int grid = 0;
    int smem_bytes = 0;
    bool needs_zero = false;   // out must be zeroed before launch (atomic_out)
    bool fused_stats = false;  // the epilogue accumulates ConvDesc::stats (needs split_k == 1, Cout <= 256)
    size_t out_bytes = 0;
};

// Returns 0 on success; on failure returns non-zero and fills `err`.
int conv_plan_create(const ConvDesc& d, int* d_err_flag, ConvPlan& plan, char* err, int errlen);
void conv_plan_destroy(ConvPlan& plan);
int conv_plan_launch(const ConvPlan& plan, cudaStream_t stream);
// Re-encode the activation tensor maps after the source pointers in `d` changed (same shapes).
int conv_plan_retarget(const ConvDesc& d, ConvPlan& plan, char* err, int errlen);
}  // namespace pixie
