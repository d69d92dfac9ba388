// Standalone bring-up harness for the tcgen05 implicit-GEMM conv (not part of the product library).
// Runs a list of small convolutions against a CPU reference and a few large ones for timing.
//   usage: conv_test [case-filter-substring]
#include "conv3d_igemm.cuh"

#include <cuda_fp8.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

using namespace pixie;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)

struct Case {
    std::string name;
    int NB, Dout, stride;
    std::vector<int> srcC;                 // channels (padded to 64) per source
    std::vector<int> srcCreal;
    std::vector<std::pair<int, int>> segs; // (src, ks)
    int Cout;
    bool bias, residual, planar;
    int split_k, block_n, td;
    bool timing;
    bool f8corr = false;   // fp16 pass + E5M2 correction segment (a_lo*w + a*w_lo) on non-fp16-representable operands
};

static float frand(std::mt19937& g) { return std::uniform_real_distribution<float>(-1.f, 1.f)(g); }

int main(int argc, char** argv) {
    const char* filter = argc > 1 ? argv[1] : "";

    std::vector<Case> cases = {
        {"gemm1x1_64_64_d16", 1, 16, 1, {64}, {64}, {{0, 1}}, 64, false, false, false, 1, 0, 0, false},
        {"gemm1x1_128_32_d16", 1, 16, 1, {128}, {128}, {{0, 1}}, 32, true, false, false, 1, 0, 0, false},
        {"conv3_64_64_d16", 1, 16, 1, {64}, {64}, {{0, 3}}, 64, false, false, false, 1, 0, 0, false},
        {"conv3_64_64_d16_td1", 1, 16, 1, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 1, false},
        {"conv3_32pad_64_d16", 2, 16, 1, {64}, {32}, {{0, 3}}, 64, true, false, false, 1, 0, 0, false},
        {"conv3_cat_skip_d16", 1, 16, 1, {128, 64, 64}, {128, 64, 64}, {{0, 3}, {1, 1}, {2, 1}}, 64, true, true, false, 1, 0, 0, false},
        {"conv3_128_128_d16", 1, 16, 1, {128}, {128}, {{0, 3}}, 128, true, true, false, 1, 0, 0, false},
        {"conv3_256_256_d8_splitk", 1, 8, 1, {256}, {256}, {{0, 3}}, 256, true, true, false, 0, 0, 0, false},
        {"conv3_s2_64_64_d16to8", 1, 8, 2, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, false},
        {"conv3_s2_64_64_d32to16", 1, 16, 2, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, false},
        {"head_64_3_planar_d16", 1, 16, 1, {64}, {64}, {{0, 3}}, 3, true, false, true, 1, 0, 0, false},
        {"qkv_256_768_d8", 1, 8, 1, {256}, {256}, {{0, 1}}, 768, true, false, false, 1, 0, 0, false},
        {"conv3_256_256_d4", 1, 4, 1, {256}, {256}, {{0, 3}}, 256, true, false, false, 0, 0, 0, false},
        {"x2_gemm1x1_128_64_d16", 1, 16, 1, {128}, {128}, {{0, 1}}, 64, true, false, false, 1, 0, 0, false, true},
        {"x2_conv3_64_64_d16", 1, 16, 1, {64}, {64}, {{0, 3}}, 64, true, true, false, 1, 0, 0, false, true},
        {"x2_conv3_128_128_d16", 2, 16, 1, {128}, {128}, {{0, 3}}, 128, true, false, false, 1, 0, 0, false, true},
        {"x2_conv3_s2_64_64_d16to8", 1, 8, 2, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, false, true},
        {"x2_conv3_256_256_d8_splitk", 1, 8, 1, {256}, {256}, {{0, 3}}, 256, true, false, false, 0, 0, 0, false, true},
        {"T_x2_conv3_64_64_d64", 1, 64, 1, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, true, true},
        {"T_x2_conv3_128_64_d64", 1, 64, 1, {128}, {128}, {{0, 3}}, 64, true, true, false, 1, 0, 0, true, true},
        {"T_conv3_64_64_d64", 1, 64, 1, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, true},
        {"T_conv3_64_64_d64_td2", 1, 64, 1, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 2, true},
        {"T_conv3_128_64_d64", 1, 64, 1, {128}, {128}, {{0, 3}}, 64, true, true, false, 1, 0, 0, true},
        {"T_conv3_128_128_d64", 1, 64, 1, {128}, {128}, {{0, 3}}, 128, true, false, false, 1, 0, 0, true},
        {"T_conv3_128_128_d64_bn128", 1, 64, 1, {128}, {128}, {{0, 3}}, 128, true, false, false, 1, 128, 0, true},
        {"T_gemm1x1_512_128_d64", 1, 64, 1, {512}, {512}, {{0, 1}}, 128, true, false, false, 1, 0, 0, true},
        {"T_conv3_64_64_d32", 1, 32, 1, {64}, {64}, {{0, 3}}, 64, true, false, false, 1, 0, 0, true},
        {"T_conv3_256_256_d8", 1, 8, 1, {256}, {256}, {{0, 3}}, 256, true, false, false, 0, 0, 0, true},
        {"T_conv3_128_128_d16", 1, 16, 1, {128}, {128}, {{0, 3}}, 128, true, false, false, 0, 0, 0, true},
    };

    int* d_err = nullptr;
    CK(cudaMalloc(&d_err, sizeof(int)));
    int n_fail = 0, n_run = 0;

    for (const Case& c : cases) {
        if (filter[0] && c.name.find(filter) == std::string::npos) continue;
        ++n_run;
        std::mt19937 gen(1234);
        const int Do = c.Dout, Di = c.Dout * c.stride;
        const size_t vox_in = (size_t)c.NB * Di * Di * Di, vox_out = (size_t)c.NB * Do * Do * Do;

        ConvDesc d;
        d.NB = c.NB; d.D = d.H = d.W = Do; d.stride = c.stride; d.Cout = c.Cout;
        d.Cout_pad = (c.Cout + 15) / 16 * 16;
        d.split_k = c.split_k; d.block_n = c.block_n; d.td = c.td; d.out_planar = c.planar;

        const float f8up = (float)(1 << kF8Shift), f8down = 1.0f / f8up;
        auto e5m2 = [](float v) { return (uint8_t)__nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E5M2); };
        auto e5m2f = [](uint8_t b) { return __half2float(__half(__nv_cvt_fp8_to_halfraw(b, __NV_E5M2))); };
        std::vector<std::vector<__half>> h_src(c.srcC.size());
        std::vector<std::vector<float>> h_true(c.srcC.size());          // f8corr: the un-rounded activations
        std::vector<std::vector<uint8_t>> h_pair(c.srcC.size());        // f8corr: [e5m2(a_lo * 2^s) x 64 | e5m2(a / 2^s) x 64] per chunk
        std::vector<__half*> d_src(c.srcC.size());
        std::vector<__half*> d_pair(c.srcC.size(), nullptr);
        for (size_t s = 0; s < c.srcC.size(); ++s) {
            const int C = c.srcC[s];
            h_src[s].resize(vox_in * C);
            if (c.f8corr) { h_true[s].resize(vox_in * C); h_pair[s].assign(vox_in * C * 2, 0); }
            for (size_t v = 0; v < vox_in; ++v)
                for (int ch = 0; ch < C; ++ch) {
                    const float a = ch < c.srcCreal[s] ? frand(gen) : 0.f;
                    const __half hi = __float2half(a);
                    h_src[s][v * C + ch] = hi;
                    if (c.f8corr) {
                        h_true[s][v * C + ch] = a;
                        uint8_t* row = &h_pair[s][(v * C + (size_t)(ch & ~63)) * 2];
                        row[ch & 63] = e5m2((a - __half2float(hi)) * f8up);
                        row[64 + (ch & 63)] = e5m2(a * f8down);
                    }
                }
            CK(cudaMalloc(&d_src[s], h_src[s].size() * 2));
            CK(cudaMemcpy(d_src[s], h_src[s].data(), h_src[s].size() * 2, cudaMemcpyHostToDevice));
            d.srcs.push_back({d_src[s], C, Di, Di, Di});
        }
        if (c.f8corr)
            for (size_t s = 0; s < c.srcC.size(); ++s) {
                CK(cudaMalloc(&d_pair[s], h_pair[s].size()));
                CK(cudaMemcpy(d_pair[s], h_pair[s].data(), h_pair[s].size(), cudaMemcpyHostToDevice));
                d.srcs.push_back({d_pair[s], c.srcC[s], Di, Di, Di});          // source index = s + n_src
            }
        std::vector<std::vector<float>> h_w(c.segs.size());
        std::vector<const float*> wptr;
        std::vector<int> cin_real;
        for (size_t g = 0; g < c.segs.size(); ++g) {
            const int src = c.segs[g].first, ks = c.segs[g].second;
            d.segs.push_back({src, ks});
            const int cin = c.srcCreal[src];
            h_w[g].resize((size_t)c.Cout * cin * ks * ks * ks);
            const float sc = 1.0f / std::sqrt((float)cin * ks * ks * ks);
            for (auto& x : h_w[g]) x = c.f8corr ? frand(gen) * sc : __half2float(__float2half(frand(gen) * sc));
            wptr.push_back(h_w[g].data());
            cin_real.push_back(cin);
            if (c.f8corr) {
                ConvDesc::Seg q{src + (int)c.srcC.size(), ks, 0, 1};
                d.segs.push_back(q);
                wptr.push_back(h_w[g].data());
                cin_real.push_back(cin);
            }
        }
        std::vector<__half> packed;
        conv_pack_weights(d, wptr, cin_real, packed);
        __half* d_w;
        CK(cudaMalloc(&d_w, packed.size() * 2));
        CK(cudaMemcpy(d_w, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
        d.weights = d_w;

        std::vector<float> h_bias(c.Cout), h_res;
        float *d_bias = nullptr, *d_res = nullptr, *d_out = nullptr;
        for (auto& x : h_bias) x = frand(gen);
        if (c.bias) {
            CK(cudaMalloc(&d_bias, c.Cout * 4));
            CK(cudaMemcpy(d_bias, h_bias.data(), c.Cout * 4, cudaMemcpyHostToDevice));
            d.bias = d_bias;
        }
        const size_t out_elems = vox_out * c.Cout;
        if (c.residual) {
            h_res.resize(out_elems);
            for (auto& x : h_res) x = frand(gen);
            CK(cudaMalloc(&d_res, out_elems * 4));
            CK(cudaMemcpy(d_res, h_res.data(), out_elems * 4, cudaMemcpyHostToDevice));
            d.residual = d_res;
        }
        CK(cudaMalloc(&d_out, out_elems * 4));
        CK(cudaMemset(d_out, 0xFF, out_elems * 4));   // NaN pattern: unwritten outputs are caught
        d.out = d_out; d.out_ld = c.Cout;

        double* d_stats = nullptr;
        CK(cudaMalloc(&d_stats, (size_t)c.NB * c.Cout * 2 * sizeof(double)));
        CK(cudaMemset(d_stats, 0, (size_t)c.NB * c.Cout * 2 * sizeof(double)));
        d.stats = getenv("CONV_TEST_NO_STATS") ? nullptr : d_stats;

        CK(cudaMemset(d_err, 0, sizeof(int)));
        ConvPlan plan;
        char err[256] = {0};
        if (conv_plan_create(d, d_err, plan, err, sizeof(err))) {
            printf("[%s] PLAN FAILED: %s\n", c.name.c_str(), err);
            ++n_fail;
            continue;
        }
        printf("[%s] grid=%d smem=%d bn=%d TD=%d TW=%d TH=%d acc_sets=%d w_stages=%d s_stages=%d phases=%d split=%d\n",
               c.name.c_str(), plan.grid, plan.smem_bytes, plan.p.block_n, plan.p.TD, plan.p.TW, plan.p.TH,
               plan.p.acc_sets, plan.p.w_stages, plan.p.s_stages, plan.p.n_phases, plan.p.split_k);
        fflush(stdout);

        int lrc = conv_plan_launch(plan, 0);
        cudaError_t se = cudaDeviceSynchronize();
        int h_err = 0;
        cudaMemcpy(&h_err, d_err, sizeof(int), cudaMemcpyDeviceToHost);
        if (lrc || se != cudaSuccess || h_err) {
            printf("[%s] LAUNCH FAILED: launch=%d sync=%s pipeline_timeout_flag=%d\n", c.name.c_str(), lrc,
                   cudaGetErrorString(se), h_err);
            ++n_fail;
            if (se != cudaSuccess) { printf("sticky CUDA error, stopping\n"); return 3; }
            continue;
        }

        if (c.timing) {
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            for (int i = 0; i < 3; ++i) conv_plan_launch(plan, 0);
            const int iters = 20;
            float ms = 0;
            if (getenv("CONV_TEST_COLD")) {
                // cold launches: a 512 MB memset (evicts L2 and the instruction caches' backing lines) before every timed launch
                static void* scrub = nullptr;
                if (!scrub) CK(cudaMalloc(&scrub, 512u << 20));
                for (int i = 0; i < iters; ++i) {
                    CK(cudaMemsetAsync(scrub, i, 512u << 20, 0));
                    cudaEventRecord(e0);
                    conv_plan_launch(plan, 0);
                    cudaEventRecord(e1);
                    CK(cudaEventSynchronize(e1));
                    float t = 0; cudaEventElapsedTime(&t, e0, e1); ms += t;
                }
            } else {
                cudaEventRecord(e0);
                for (int i = 0; i < iters; ++i) conv_plan_launch(plan, 0);
                cudaEventRecord(e1);
                CK(cudaEventSynchronize(e1));
                cudaEventElapsedTime(&ms, e0, e1);
            }
            ms /= iters;
            double flops = 2.0 * vox_out * c.Cout * (double)conv_k_total(d);
            printf("[%s] TIME %.3f ms  %.1f TFLOP/s (padded-K flops)  [bn=%d TW=%d TD=%d w_stages=%d s_stages=%d split=%d smem=%d]\n", c.name.c_str(), ms, flops / ms * 1e-9,
                   plan.p.block_n, plan.p.TW, plan.p.TD, plan.p.w_stages, plan.p.s_stages, plan.p.split_k, plan.smem_bytes);
        }

        // verification (sampled voxels for big cases)
        std::vector<float> h_out(out_elems);
        CK(cudaMemcpy(h_out.data(), d_out, out_elems * 4, cudaMemcpyDeviceToHost));
        const size_t nsample = c.timing ? 600 : vox_out;
        double max_err = 0, max_ref = 0, max_true_err = 0, max_fp16_err = 0;
        size_t bad = 0, nan_cnt = 0;
        std::mt19937 g2(99);
        for (size_t si = 0; si < nsample; ++si) {
            size_t v = c.timing ? (size_t)(std::uniform_int_distribution<size_t>(0, vox_out - 1)(g2)) : si;
            if (c.timing && si < 64) v = si * (vox_out / 64);   // include structured positions (corners/edges)
            size_t t = v;
            const int ow = t % Do; t /= Do;
            const int oh = t % Do; t /= Do;
            const int od = t % Do; t /= Do;
            const int nb = (int)t;
            for (int co = 0; co < c.Cout; ++co) {
                double acc = c.bias ? h_bias[co] : 0.0, acc_true = acc, acc_h = acc;
                for (size_t g = 0; g < c.segs.size(); ++g) {
                    const int src = c.segs[g].first, ks = c.segs[g].second, pad = ks / 2;
                    const int cin = c.srcCreal[src], C = c.srcC[src];
                    for (int kd = 0; kd < ks; ++kd)
                        for (int kh = 0; kh < ks; ++kh)
                            for (int kw = 0; kw < ks; ++kw) {
                                const int id = od * c.stride + kd - pad, ih = oh * c.stride + kh - pad, iw = ow * c.stride + kw - pad;
                                if (ks == 1) { /* 1x1 convs always read the same-resolution voxel */ }
                                if (id < 0 || ih < 0 || iw < 0 || id >= Di || ih >= Di || iw >= Di) continue;
                                const __half* xp = &h_src[src][((((size_t)nb * Di + id) * Di + ih) * Di + iw) * C];
                                const float* wp = &h_w[g][(size_t)co * cin * ks * ks * ks + (kd * ks + kh) * ks + kw];
                                if (!c.f8corr) {
                                    for (int ci = 0; ci < cin; ++ci)
                                        acc += (double)__half2float(xp[ci]) * wp[(size_t)ci * ks * ks * ks];
                                    continue;
                                }
                                // what the kernel is asked to compute: fp16(a) fp16(w) + A1 W1 + A2 W2 on the stored operands
                                const size_t vrow = (((size_t)nb * Di + id) * Di + ih) * Di + iw;
                                for (int ci = 0; ci < cin; ++ci) {
                                    const float w = wp[(size_t)ci * ks * ks * ks], wh = __half2float(__float2half(w));
                                    const uint8_t* row = &h_pair[src][(vrow * C + (size_t)(ci & ~63)) * 2];
                                    const double a1 = e5m2f(row[ci & 63]), a2 = e5m2f(row[64 + (ci & 63)]);
                                    const double w1 = e5m2f(e5m2(w * f8down)), w2 = e5m2f(e5m2((w - wh) * f8up));
                                    const double hh = (double)__half2float(xp[ci]) * wh;
                                    acc += hh + a1 * w1 + a2 * w2;
                                    acc_h += hh;
                                    acc_true += (double)h_true[src][vrow * C + ci] * w;
                                }
                            }
                }
                const size_t oidx_nd = v * c.Cout + co;
                if (c.residual) acc += h_res[oidx_nd];
                const size_t oidx = c.planar ? ((size_t)nb * c.Cout + co) * ((size_t)Do * Do * Do) + (v % ((size_t)Do * Do * Do)) : oidx_nd;
                const float got = h_out[oidx];
                if (std::isnan(got)) { ++nan_cnt; continue; }
                const double e = std::fabs(got - acc);
                if (c.f8corr) {
                    const double rr = c.residual ? h_res[oidx_nd] : 0.0;
                    max_true_err = std::max(max_true_err, std::fabs(got - (acc_true + rr)));
                    max_fp16_err = std::max(max_fp16_err, std::fabs(acc_h - acc_true));
                }
                max_err = std::max(max_err, e);
                max_ref = std::max(max_ref, std::fabs(acc));
                if (e > 2e-3 * std::max(1.0, std::fabs(acc))) ++bad;
            }
        }
        // fused statistics: per-(sample, channel) sum and sum of squares of the outputs
        size_t stats_bad = 0;
        if (plan.fused_stats && !c.timing) {
            std::vector<double> h_stats((size_t)c.NB * c.Cout * 2);
            CK(cudaMemcpy(h_stats.data(), d_stats, h_stats.size() * sizeof(double), cudaMemcpyDeviceToHost));
            const size_t vpb = (size_t)Do * Do * Do;
            for (int nb = 0; nb < c.NB; ++nb) {
                for (int co = 0; co < c.Cout; ++co) {
                    double s = 0, q = 0;
                    for (size_t v = 0; v < vpb; ++v) { const double x = h_out[((size_t)nb * vpb + v) * c.Cout + co]; s += x; q += x * x; }
                    const double gs = h_stats[((size_t)nb * c.Cout + co) * 2], gq = h_stats[((size_t)nb * c.Cout + co) * 2 + 1];
                    if (std::fabs(gs - s) > 1e-3 * (1 + std::fabs(s)) + 1e-4 * std::sqrt(q * vpb) || std::fabs(gq - q) > 1e-4 * (1 + q)) {
                        if (stats_bad < 3) printf("   stats mismatch nb=%d co=%d: sum %g vs %g, sumsq %g vs %g\n", nb, co, gs, s, gq, q);
                        ++stats_bad;
                    }
                }
            }
            printf("[%s] fused stats checked: bad=%zu\n", c.name.c_str(), stats_bad);
        }
        const bool pass = (bad == 0 && nan_cnt == 0 && stats_bad == 0);
        printf("[%s] %s max_err=%.3e max_ref=%.3f bad=%zu nan=%zu\n", c.name.c_str(), pass ? "PASS" : "FAIL", max_err, max_ref, bad, nan_cnt);
        if (c.f8corr) printf("[%s] vs exact a*w: fp16 pass + e5m2 corrections %.3e, single fp16 pass alone %.3e\n", c.name.c_str(), max_true_err, max_fp16_err);
        if (!pass) {
            ++n_fail;
            // print a few values to help diagnose layout errors
            for (int i = 0; i < 8 && i < (int)out_elems; ++i) printf("   out[%d]=%g\n", i, h_out[i]);
        }
        fflush(stdout);

        conv_plan_destroy(plan);
        for (auto p : d_src) cudaFree(p);
        for (auto p : d_pair) cudaFree(p);
        cudaFree(d_w); cudaFree(d_bias); cudaFree(d_res); cudaFree(d_out); cudaFree(d_stats);
    }
    printf("SUMMARY run=%d fail=%d\n", n_run, n_fail);
    return n_fail ? 1 : 0;
}
