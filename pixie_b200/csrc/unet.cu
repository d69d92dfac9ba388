// U-Net executor: builds, from the reference's constructor arguments and state dict, the list of
// kernel launches that computes SegmentationUNet / RegressionUNet.forward on one B200.
//
// Graph restated from third_party/Wavelet-Generation/models/module/diffusion_network.py:
//   FeatureProjector 534-589, MyResBlock 639-710, Downsample 75-97, Upsample 51-72,
//   AttentionBlock 192-221, MyUNetModel.__init__ 734-873 / forward 899-935.
// Data flow: every convolution output is an fp32 channels-last tensor (the residual stream never
// leaves fp32); every convolution input is an fp16 channels-last tensor produced by the
// normalise/activate kernel (or the cast / upsample kernels).  torch.cat([h, skip]) (:932) is never
// materialised in fp32: the two sources are normalised into channel slices of one fp16 buffer.
// The ResBlock's 1x1 skip convolution (:687-694) is folded into its second 3x3x3 convolution as
// extra K phases over the raw (un-normalised) fp16 input.
#include "unet.cuh"
#include "conv3d_igemm.cuh"
#include "unet_kernels.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

namespace pixie {

namespace {

struct HostTensor {
    std::vector<float> data;
    std::vector<int64_t> shape;
};

struct ConvOp {
    ConvDesc desc;
    ConvPlan plan;
};

struct DevT {          // fp32 activation [NB][sp^3][C]
    float* p = nullptr;
    int C = 0, sp = 0;
    double* stats = nullptr;   // [NB][C][2] (sum, sumsq over voxels), filled by the producer when requested
};

}  // namespace

struct UNet {
    pixie_unet_config cfg{};
    std::map<std::string, HostTensor> params;
    bool finalized = false;
    int NBmax = 1;

    std::vector<void*> allocs;
    std::vector<std::function<int(cudaStream_t)>> ops;   // bound to the batch size in `cur_nb`
    std::vector<int> op_kinds;                            // PIXIE_OP_* per op
    std::vector<double> op_flops;                         // algorithmic FLOPs per op (convs only)
    std::vector<std::unique_ptr<ConvOp>> convs;
    std::map<std::string, DevT> named;
    int* d_err = nullptr;              // device view of h_err
    volatile int* h_err = nullptr;     // mapped pinned host flag: a convolution that gave up waiting on its pipeline sets it
    double* d_stats = nullptr;
    size_t stats_doubles = 0, stats_cap = 0;
    int cur_nb = 1;
    double flops = 0;
    int n_launch = 0;
    // I/O plumbing
    ConvOp* first_conv = nullptr;      // consumes the user's feature grid
    ConvOp* head_conv = nullptr;       // writes the user's output
    int feat_cpad = 0;
    __half* feat_staging = nullptr;    // for forward_ncdhw / forward_host
    float* out_staging = nullptr;
    std::string error;
    // whole-forward CUDA graphs, keyed by (batch, input pointer, output pointer); a few entries so that callers that
    // alternate between buffers (double-buffered host pipeline) replay instead of re-capturing
    struct GraphEntry { cudaGraphExec_t exec = nullptr; const void* feat = nullptr; float* out = nullptr; int nb = 0; };
    static constexpr int kGraphSlots = 4;
    GraphEntry graphs[kGraphSlots];
    int graph_next = 0;
    bool use_graph = true;          // cleared when a capture or instantiation fails: launch directly from then on

    ~UNet() {
        for (auto& g : graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
        for (auto& c : convs) conv_plan_destroy(c->plan);
        for (void* p : allocs) cudaFree(p);
        if (h_err) cudaFreeHost(const_cast<int*>(h_err));
    }
};

namespace {

struct Builder {
    UNet& u;
    int NB;
    bool precise;          // split-precision: every activation tensor carries a second tensor (`lo`)
    bool f8corr;           // ... holding E5M2 correction operands (precision 2) instead of the fp16 residual (precision 1)
    std::string err;

    explicit Builder(UNet& un) : u(un), NB(un.NBmax), precise(un.cfg.precision >= 1), f8corr(un.cfg.precision == 2) {}

    bool fail(const std::string& m) { if (err.empty()) err = m; return false; }

    template <typename T>
    T* dalloc(size_t n) {
        void* p = nullptr;
        if (cudaMalloc(&p, n * sizeof(T)) != cudaSuccess) { fail("cudaMalloc failed"); return nullptr; }
        cudaMemset(p, 0, n * sizeof(T));
        u.allocs.push_back(p);
        return reinterpret_cast<T*>(p);
    }
    float* upload(const std::vector<float>& v) {
        float* d = dalloc<float>(v.size());
        if (d) cudaMemcpy(d, v.data(), v.size() * 4, cudaMemcpyHostToDevice);
        return d;
    }
    const HostTensor* param(const std::string& name, size_t expect_numel) {
        auto it = u.params.find(name);
        if (it == u.params.end()) { fail("missing state-dict entry: " + name); return nullptr; }
        if (it->second.data.size() != expect_numel) {
            fail("state-dict entry " + name + " has wrong size");
            return nullptr;
        }
        return &it->second;
    }
    size_t vox(int sp) const { return (size_t)sp * sp * sp; }

    double* stats_slot(int C) {
        double* s = u.d_stats + u.stats_doubles;
        u.stats_doubles += (size_t)NB * C * 2;
        return s;
    }

    // -------------------------------------------------------------------------------- op emitters
    struct F16 { __half* hi = nullptr; __half* lo = nullptr; int C = 0; int sp = 0; };

    F16 alloc_f16(int C, int sp) {
        F16 t; t.C = C; t.sp = sp;
        t.hi = dalloc<__half>((size_t)NB * vox(sp) * C);
        if (precise) t.lo = dalloc<__half>((size_t)NB * vox(sp) * C);
        return t;
    }

    void emit_moments(const DevT& x, double* stats) {
        UNet* up = &u;
        const int V = (int)vox(x.sp), C = x.C;
        const float* xp = x.p;
        u.ops.push_back([=](cudaStream_t st) { return launch_moments(xp, up->cur_nb, V, C, stats, st); });
        u.op_kinds.push_back(PIXIE_OP_MOMENTS); u.op_flops.push_back(0);
    }

    // normalise x (LN with per-voxel affine, or GN) into channel slice [c0, c0+x.C) of dst;
    // optionally also an un-normalised fp16 copy into raw.
    void emit_norm(const DevT& x, const double* stats, int mode, int groups, const float* gamma, const float* beta,
                   int act, const F16* dst, int c0, const F16* raw, int raw_c0) {
        NormArgs a;
        a.x = x.p; a.V = (int)vox(x.sp); a.C = x.C; a.stats = stats; a.mode = mode; a.groups = groups;

        a.gamma = gamma; a.beta = beta; a.eps = 1e-5f; a.act = act;
        a.lo_mode = f8corr ? 1 : 0;
        if (dst) { a.dst = dst->hi; a.dst_lo = dst->lo; a.dst_ld = dst->C; a.dst_c0 = c0; }
        if (raw) { a.raw_dst = raw->hi; a.raw_lo = raw->lo; a.raw_ld = raw->C; a.raw_c0 = raw_c0; }
        UNet* up = &u;
        u.ops.push_back([=](cudaStream_t st) { return launch_norm_act(a, up->cur_nb, st); });
        u.op_kinds.push_back(PIXIE_OP_NORM); u.op_flops.push_back(0);
    }

    struct ConvIn { F16 t; int ks; int cin_real; std::string wname; };

    // out[C_out] = sum_i conv_ks_i(in_i) + sum of biases (+ residual)
    // want_stats: the output feeds a LayerNorm / GroupNorm -> per-(n,c) moments are produced too, by the conv
    // epilogue when possible (no split-K), else by a moments launch right after the conv.
    ConvOp* emit_conv(const std::vector<ConvIn>& ins, int sp_out, int stride, int Cout, const float* residual,
                      float* out, bool planar, const std::vector<std::string>& bias_names, DevT* want_stats = nullptr) {
        auto op = std::make_unique<ConvOp>();
        const double flops_before = u.flops;
        ConvDesc& d = op->desc;
        d.NB = NB; d.D = d.H = d.W = sp_out; d.stride = stride; d.Cout = Cout;
        d.Cout_pad = (Cout + 15) / 16 * 16;
        d.split_k = 0;   // auto
        if (Cout % 128 == 0 && sp_out >= 32 && !planar) d.block_n = 128;   // halves the A-slab traffic per output channel
        std::vector<const float*> wptr;
        std::vector<int> cin_real;
        std::vector<std::vector<float>> keep;
        for (const auto& in : ins) {
            const int ks = in.ks, kv = ks * ks * ks;
            const HostTensor* w = param(in.wname, (size_t)Cout * in.cin_real * kv);
            if (!w) return nullptr;
            const int si = (int)d.srcs.size();
            d.srcs.push_back({in.t.hi, in.t.C, in.t.sp, in.t.sp, in.t.sp});
            d.segs.push_back({si, ks, 0});
            wptr.push_back(w->data.data()); cin_real.push_back(in.cin_real);
            u.flops += 2.0 * (double)vox(sp_out) * Cout * in.cin_real * kv;
            if (f8corr && in.t.lo) {
                // a_lo * w + a * w_lo in ONE segment of E5M2 operands at twice the fp16 MMA rate (2 pass-equivalents per
                // algorithmic FLOP instead of 3; error 2^-3 of a single fp16 pass, measured 3e-4 max-abs end to end)
                const int sl = (int)d.srcs.size();
                d.srcs.push_back({in.t.lo, in.t.C, in.t.sp, in.t.sp, in.t.sp});
                ConvDesc::Seg q{sl, ks, 0, 1};
                d.segs.push_back(q);
                wptr.push_back(w->data.data()); cin_real.push_back(in.cin_real);
            } else if (precise && in.t.lo) {
                // a_lo * w_hi  and  a_hi * w_lo
                const int sl = (int)d.srcs.size();
                d.srcs.push_back({in.t.lo, in.t.C, in.t.sp, in.t.sp, in.t.sp});
                d.segs.push_back({sl, ks, 0});
                wptr.push_back(w->data.data()); cin_real.push_back(in.cin_real);
                d.segs.push_back({si, ks, 1});
                wptr.push_back(w->data.data()); cin_real.push_back(in.cin_real);
            } else if (precise) {
                d.segs.push_back({si, ks, 1});
                wptr.push_back(w->data.data()); cin_real.push_back(in.cin_real);
            }
        }
        std::vector<__half> packed;
        conv_pack_weights(d, wptr, cin_real, packed);
        __half* dw = dalloc<__half>(packed.size());
        if (!dw) return nullptr;
        cudaMemcpy(dw, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice);
        d.weights = dw;
        std::vector<float> bias(Cout, 0.f);
        for (const auto& bn : bias_names) {
            const HostTensor* b = param(bn, (size_t)Cout);
            if (!b) return nullptr;
            for (int i = 0; i < Cout; ++i) bias[i] += b->data[i];
        }
        d.bias = upload(bias);
        d.residual = residual;
        d.out = out; d.out_ld = Cout; d.out_c0 = 0; d.out_planar = planar ? 1 : 0;
        if (want_stats) { want_stats->stats = stats_slot(Cout); d.stats = want_stats->stats; }
        char e[256] = {0};
        if (conv_plan_create(d, u.d_err, op->plan, e, sizeof(e))) { fail(e); return nullptr; }
        ConvOp* raw = op.get();
        UNet* up = &u;
        u.ops.push_back([=](cudaStream_t st) {
            // the plan was built for NBmax; smaller batches only shrink the tile count
            ConvPlan pl = raw->plan;
            pl.p.NB = up->cur_nb;
            const int items = pl.p.NB * pl.p.tiles_d * pl.p.tiles_h * pl.p.tiles_w * pl.p.n_tiles * pl.p.split_k;
            pl.grid = items < pl.grid ? items : pl.grid;
            return conv_plan_launch(pl, st);
        });
        u.op_kinds.push_back(PIXIE_OP_CONV); u.op_flops.push_back(u.flops - flops_before);
        const bool fused = raw->plan.fused_stats;
        u.convs.push_back(std::move(op));
        if (want_stats && !fused) emit_moments(*want_stats, want_stats->stats);
        return raw;
    }

    DevT alloc_f32(int C, int sp, const std::string& name) {
        DevT t; t.C = C; t.sp = sp;
        t.p = dalloc<float>((size_t)NB * vox(sp) * C);
        if (!name.empty()) u.named[name] = t;
        return t;
    }

    // MyResBlock (:639-710) over the channel concatenation of `xs`.
    DevT resblock(const std::vector<DevT>& xs, int Cout, const std::string& path) {
        const int sp = xs[0].sp;
        int Cin = 0;
        for (auto& x : xs) Cin += x.C;
        const bool has_skip = (Cin != Cout);
        const size_t V = vox(sp);
        const HostTensor* g1 = param(path + ".in_layers.0.weight", V);
        const HostTensor* b1 = param(path + ".in_layers.0.bias", V);
        const HostTensor* g2 = param(path + ".out_layers.0.weight", V);
        const HostTensor* b2 = param(path + ".out_layers.0.bias", V);
        if (!g1 || !b1 || !g2 || !b2) return {};
        const float *dg1 = upload(g1->data), *db1 = upload(b1->data), *dg2 = upload(g2->data), *db2 = upload(b2->data);

        F16 a = alloc_f16(Cin, sp);
        F16 raw;
        if (has_skip) raw = alloc_f16(Cin, sp);
        int c0 = 0;
        for (auto& x : xs) {
            if (!x.stats) { fail("internal: input of " + path + " has no statistics"); return {}; }
            emit_norm(x, x.stats, kNormLN, 1, dg1, db1, kActLeaky, &a, c0, has_skip ? &raw : nullptr, c0);
            c0 += x.C;
        }
        DevT t = alloc_f32(Cout, sp, "");
        if (!emit_conv({{a, 3, Cin, path + ".in_layers.2.weight"}}, sp, 1, Cout, nullptr, t.p, false,
                       {path + ".in_layers.2.bias"}, &t)) return {};
        F16 b = alloc_f16(Cout, sp);
        emit_norm(t, t.stats, kNormLN, 1, dg2, db2, kActLeaky, &b, 0, nullptr, 0);
        DevT out = alloc_f32(Cout, sp, path);
        std::vector<ConvIn> ins = {{b, 3, Cout, path + ".out_layers.3.weight"}};
        std::vector<std::string> biases = {path + ".out_layers.3.bias"};
        if (has_skip) {
            ins.push_back({raw, 1, Cin, path + ".skip_connection.weight"});
            biases.push_back(path + ".skip_connection.bias");
        }
        if (!emit_conv(ins, sp, 1, Cout, has_skip ? nullptr : xs[0].p, out.p, false, biases, &out)) return {};
        u.named[path] = out;
        return out;
    }

    DevT downsample(const DevT& x, const std::string& path) {
        F16 raw = alloc_f16(x.C, x.sp);
        emit_norm(x, nullptr, kNormNone, 1, nullptr, nullptr, kActNone, nullptr, 0, &raw, 0);
        const int sp_out = (x.sp + 1) / 2;
        DevT out = alloc_f32(x.C, sp_out, path);
        if (!emit_conv({{raw, 3, x.C, path + ".op.weight"}}, sp_out, 2, x.C, nullptr, out.p, false, {path + ".op.bias"}, &out)) return {};
        return out;
    }

    DevT upsample(const DevT& x, const std::string& path) {
        F16 up = alloc_f16(x.C, 2 * x.sp);
        {
            UNet* upn = &u;
            const float* xp = x.p; __half* hi = up.hi; __half* lo = up.lo; const int sp = x.sp, C = x.C;
            const int lom = f8corr ? 1 : 0;
            u.ops.push_back([=](cudaStream_t st) { return launch_upsample2(xp, hi, lo, lom, upn->cur_nb, sp, C, st); });
            u.op_kinds.push_back(PIXIE_OP_UPSAMPLE); u.op_flops.push_back(0);
        }
        DevT out = alloc_f32(x.C, 2 * x.sp, path);
        if (!emit_conv({{up, 3, x.C, path + ".conv.weight"}}, 2 * x.sp, 1, x.C, nullptr, out.p, false, {path + ".conv.bias"}, &out)) return {};
        return out;
    }

    DevT attention(const DevT& x, const std::string& path) {
        const int C = x.C, T = (int)vox(x.sp);
        const HostTensor* g = param(path + ".norm.weight", (size_t)C);
        const HostTensor* b = param(path + ".norm.bias", (size_t)C);
        if (!g || !b) return {};
        F16 n = alloc_f16(C, x.sp);
        if (!x.stats) { fail("internal: attention input has no statistics"); return {}; }
        emit_norm(x, x.stats, kNormGN, 32, upload(g->data), upload(b->data), kActNone, &n, 0, nullptr, 0);
        DevT qkv = alloc_f32(3 * C, x.sp, "");
        if (!emit_conv({{n, 1, C, path + ".qkv.weight"}}, x.sp, 1, 3 * C, nullptr, qkv.p, false, {path + ".qkv.bias"})) return {};
        F16 at = alloc_f16(C, x.sp);
        {
            UNet* upn = &u;
            const float* qp = qkv.p; __half* hi = at.hi; __half* lo = at.lo;
            const int lom = f8corr ? 1 : 0;
            u.ops.push_back([=](cudaStream_t s) { return launch_attention(qp, hi, lo, lom, upn->cur_nb, T, C, s); });
            u.op_kinds.push_back(PIXIE_OP_ATTENTION); u.op_flops.push_back(0);
        }
        DevT out = alloc_f32(C, x.sp, path);
        if (!emit_conv({{at, 1, C, path + ".proj_out.weight"}}, x.sp, 1, C, x.p, out.p, false, {path + ".proj_out.bias"}, &out)) return {};
        return out;
    }

    bool build() {
        const pixie_unet_config& c = u.cfg;
        const int G = c.grid_size;
        {   // mapped pinned flag: the host can poll it without synchronising (checked at the start of every forward
            // and after every synchronising call), the kernels write it through the device alias
            int* h = nullptr;
            if (cudaHostAlloc(&h, sizeof(int), cudaHostAllocMapped) != cudaSuccess) return fail("cudaHostAlloc");
            *h = 0;
            u.h_err = h;
            if (cudaHostGetDevicePointer(&u.d_err, h, 0) != cudaSuccess) return fail("cudaHostGetDevicePointer");
        }
        u.stats_cap = (size_t)NB * 2 * 64 * 1024;   // doubles; far above the ~70 norms x <=512 channels
        u.d_stats = dalloc<double>(u.stats_cap);

        // ---- input: fp16 NDHWC feature grid, channels padded to a multiple of 64
        u.feat_cpad = (c.feature_channels + 63) / 64 * 64;
        u.feat_staging = dalloc<__half>((size_t)NB * vox(G) * u.feat_cpad);
        F16 feat; feat.hi = u.feat_staging; feat.lo = nullptr; feat.C = u.feat_cpad; feat.sp = G;

        // ---- projector (FeatureProjector :534-589)
        F16 unet_in;
        size_t first_conv_idx = u.convs.size();
        if (c.feature_channels == c.cond_dim) {
            unet_in = feat;                                   // projector is None (training_discrete.py:63-68)
        } else if (c.feature_channels > c.cond_dim) {
            const int Hc = 128;
            DevT c0 = alloc_f32(Hc, G, "projector.net.0");
            if (!emit_conv({{feat, 1, c.feature_channels, "projector.net.0.weight"}}, G, 1, Hc, nullptr, c0.p, false, {"projector.net.0.bias"}, &c0)) return false;
            const HostTensor *g1 = param("projector.net.1.weight", Hc), *b1 = param("projector.net.1.bias", Hc);
            if (!g1 || !b1) return false;
            F16 a1 = alloc_f16(Hc, G);
            emit_norm(c0, c0.stats, kNormGN, 32, upload(g1->data), upload(b1->data), kActSiLU, &a1, 0, nullptr, 0);
            DevT c1 = alloc_f32(Hc, G, "projector.net.3");
            if (!emit_conv({{a1, 3, Hc, "projector.net.3.weight"}}, G, 1, Hc, nullptr, c1.p, false, {"projector.net.3.bias"}, &c1)) return false;
            const HostTensor *g2 = param("projector.net.4.weight", Hc), *b2 = param("projector.net.4.bias", Hc);
            if (!g2 || !b2) return false;
            F16 a2 = alloc_f16(Hc, G);
            emit_norm(c1, c1.stats, kNormGN, 32, upload(g2->data), upload(b2->data), kActSiLU, &a2, 0, nullptr, 0);
            DevT c2 = alloc_f32(c.cond_dim, G, "projector.net.6");
            if (!emit_conv({{a2, 1, Hc, "projector.net.6.weight"}}, G, 1, c.cond_dim, nullptr, c2.p, false, {"projector.net.6.bias"}, &c2)) return false;
            const HostTensor *g3 = param("projector.net.7.weight", c.cond_dim), *b3 = param("projector.net.7.bias", c.cond_dim);
            if (!g3 || !b3) return false;
            unet_in = alloc_f16((c.cond_dim + 63) / 64 * 64, G);     // zero-padded channels stay zero
            emit_norm(c2, c2.stats, kNormGN, 32, upload(g3->data), upload(b3->data), kActNone, &unet_in, 0, nullptr, 0);
        } else {
            // light projector: Conv3d 1x1 -> GroupNorm(max(out/2,1)) -> SiLU
            DevT c0 = alloc_f32(c.cond_dim, G, "projector.net.0");
            if (!emit_conv({{feat, 1, c.feature_channels, "projector.net.0.weight"}}, G, 1, c.cond_dim, nullptr, c0.p, false, {"projector.net.0.bias"}, &c0)) return false;
            const HostTensor *g1 = param("projector.net.1.weight", c.cond_dim), *b1 = param("projector.net.1.bias", c.cond_dim);
            if (!g1 || !b1) return false;
            unet_in = alloc_f16((c.cond_dim + 63) / 64 * 64, G);
            const int groups = c.cond_dim / 2 > 1 ? c.cond_dim / 2 : 1;
            emit_norm(c0, c0.stats, kNormGN, groups, upload(g1->data), upload(b1->data), kActSiLU, &unet_in, 0, nullptr, 0);
        }

        // ---- MyUNetModel (:734-873); same construction order so module paths match the state dict
        const int mc = c.model_channels;
        std::vector<DevT> hs;
        DevT h = alloc_f32(mc, G, "unet.input_blocks.0");
        if (!emit_conv({{unet_in, 3, c.cond_dim, "unet.input_blocks.0.0.weight"}}, G, 1, mc, nullptr, h.p, false, {"unet.input_blocks.0.0.bias"}, &h)) return false;
        u.first_conv = u.convs[first_conv_idx].get();
        hs.push_back(h);
        int ch = mc, sp = G, blk = 1;
        for (int level = 0; level < c.n_levels; ++level) {
            const int mult = c.channel_mult[level];
            for (int r = 0; r < c.num_res_blocks; ++r) {
                h = resblock({h}, mult * mc, "unet.input_blocks." + std::to_string(blk) + ".0");
                if (!h.p) return false;
                ch = mult * mc;
                hs.push_back(h);
                ++blk;
            }
            if (level != c.n_levels - 1) {
                h = downsample(h, "unet.input_blocks." + std::to_string(blk) + ".0");
                if (!h.p) return false;
                hs.push_back(h);
                ++blk;
                sp = (sp + 1) / 2;
            }
        }
        h = resblock({h}, ch, "unet.middle_block.0");
        if (!h.p) return false;
        h = attention(h, "unet.middle_block.1");
        if (!h.p) return false;
        h = resblock({h}, ch, "unet.middle_block.2");
        if (!h.p) return false;
        int ob = 0;
        for (int level = c.n_levels - 1; level >= 0; --level) {
            const int mult = c.channel_mult[level];
            for (int i = 0; i < c.num_res_blocks + 1; ++i) {
                DevT skip = hs.back();
                hs.pop_back();
                if (skip.sp != h.sp) return fail("odd grid sizes are not supported (crop path :925-930)");
                h = resblock({h, skip}, mc * mult, "unet.output_blocks." + std::to_string(ob) + ".0");
                if (!h.p) return false;
                if (level && i == c.num_res_blocks) {
                    h = upsample(h, "unet.output_blocks." + std::to_string(ob) + ".1");
                    if (!h.p) return false;
                }
                ++ob;
            }
        }
        // ---- head (:869-873)
        {
            const size_t V = vox(G);
            const HostTensor *g = param("unet.out.0.weight", V), *b = param("unet.out.0.bias", V);
            if (!g || !b) return false;
            F16 a = alloc_f16(mc, G);
            if (!h.stats) return fail("internal: head input has no statistics");
            emit_norm(h, h.stats, kNormLN, 1, upload(g->data), upload(b->data), kActLeaky, &a, 0, nullptr, 0);
            u.out_staging = dalloc<float>((size_t)NB * c.out_channels * V);
            u.head_conv = emit_conv({{a, 3, mc, "unet.out.2.weight"}}, G, 1, c.out_channels, nullptr, u.out_staging, true, {"unet.out.2.bias"});
            if (!u.head_conv) return false;
        }
        if (u.stats_doubles > u.stats_cap) return fail("stats arena overflow");
        if (!err.empty()) return false;
        return cudaDeviceSynchronize() == cudaSuccess || fail("CUDA error during finalize");
    }
};

}  // namespace

// ----------------------------------------------------------------------------------------- API
UNet* unet_create(const pixie_unet_config& cfg, std::string& err) {
    if (cfg.n_levels < 1 || cfg.n_levels > 8) { err = "n_levels out of range"; return nullptr; }
    if (cfg.grid_size % (1 << (cfg.n_levels - 1))) { err = "grid_size must be divisible by 2^(levels-1)"; return nullptr; }
    if (cfg.model_channels % 64) { err = "model_channels must be a multiple of 64"; return nullptr; }
    if (cfg.precision < 0 || cfg.precision > 2) { err = "precision must be 0 (fp16), 1 (fp16x3) or 2 (fp16 + e5m2 corrections)"; return nullptr; }
    auto* u = new UNet();
    u->cfg = cfg;
    u->NBmax = cfg.max_batch > 0 ? cfg.max_batch : 1;
    return u;
}

int unet_set_tensor(UNet* u, const char* name, const float* data, const int64_t* shape, int ndim) {
    if (u->finalized) { u->error = "set_tensor after finalize"; return 1; }
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(data, data + n);
    u->params[name] = std::move(t);
    return 0;
}

int unet_finalize(UNet* u) {
    if (u->finalized) return 0;
    Builder b(*u);
    if (!b.build()) { u->error = b.err.empty() ? "finalize failed" : b.err; return 1; }
    u->params.clear();
    u->finalized = true;
    u->n_launch = (int)u->ops.size() + 1;   // + stats memset
    return 0;
}

static int enqueue_ops(UNet* u, cudaStream_t st) {
    cudaMemsetAsync(u->d_stats, 0, u->stats_doubles * sizeof(double), st);
    for (auto& op : u->ops) {
        const int rc = op(st);
        if (rc) { u->error = "kernel launch failed, cuda error " + std::to_string(rc); return 1; }
    }
    return 0;
}

static int run_ops(UNet* u, int batch, const void* feat, float* out, cudaStream_t st) {
    u->cur_nb = batch;
    if (u->use_graph) {
        UNet::GraphEntry* hit = nullptr;
        for (auto& g : u->graphs) if (g.exec && g.nb == batch && g.feat == feat && g.out == out) hit = &g;
        if (!hit) {
            UNet::GraphEntry& slot = u->graphs[u->graph_next];
            u->graph_next = (u->graph_next + 1) % UNet::kGraphSlots;
            if (slot.exec) { cudaGraphExecDestroy(slot.exec); slot.exec = nullptr; }
            cudaStream_t cs;                      // the caller's stream may be the legacy default stream, which cannot capture
            cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
            cudaGraph_t g = nullptr;
            bool ok = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int rc = enqueue_ops(u, cs);
                ok = (cudaStreamEndCapture(cs, &g) == cudaSuccess) && g && rc == 0;
            }
            if (ok) ok = cudaGraphInstantiate(&slot.exec, g, 0) == cudaSuccess;
            if (g) cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            if (!ok) { cudaGetLastError(); slot.exec = nullptr; u->use_graph = false; }
            else { slot.nb = batch; slot.feat = feat; slot.out = out; hit = &slot; }
        }
        if (hit && hit->exec) {
            if (cudaGraphLaunch(hit->exec, st) != cudaSuccess) { u->error = "cudaGraphLaunch failed"; return 1; }
            return 0;
        }
    }
    return enqueue_ops(u, st);
}

// Non-blocking: reports (and re-arms) a pipeline timeout raised by any forward enqueued so far that has already run.
static int check_err_flag(UNet* u) {
    const int h = u->h_err ? *u->h_err : 0;
    if (h) {
        *u->h_err = 0;
        u->error = "conv pipeline timeout (device flag " + std::to_string(h) + "): the outputs of the affected forward are invalid";
        return 1;
    }
    return 0;
}

int unet_forward(UNet* u, const void* feat_f16, int batch, float* out, cudaStream_t st) {
    if (!u->finalized) { u->error = "forward before finalize"; return 1; }
    if (check_err_flag(u)) return 1;          // an earlier (asynchronous) forward timed out: do not hand out more garbage
    if (batch < 1 || batch > u->NBmax) { u->error = "batch exceeds max_batch"; return 1; }
    // point the first convolution at the caller's grid and the head at the caller's output
    ConvOp* fc = u->first_conv;
    const __half* fp = reinterpret_cast<const __half*>(feat_f16);
    char e[256] = {0};
    if (fc->desc.srcs[0].ptr != fp) {
        fc->desc.srcs[0].ptr = fp;
        if (conv_plan_retarget(fc->desc, fc->plan, e, sizeof(e))) { u->error = e; return 1; }
    }
    u->head_conv->plan.p.out = out;
    return run_ops(u, batch, feat_f16, out, st);
}

int unet_profile(UNet* u, const void* feat_f16, int batch, float* out, cudaStream_t st, float* ms, int* kinds, double* flops, int cap) {
    if (!u->finalized) { u->error = "profile before finalize"; return -1; }
    const int n = (int)u->ops.size();
    if (cap < n) { u->error = "profile: buffers too small"; return -1; }
    if (unet_forward(u, feat_f16, batch, out, st)) return -1;      // warm + retarget
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) cudaEventCreate(&e);
    u->cur_nb = batch;
    cudaMemsetAsync(u->d_stats, 0, u->stats_doubles * sizeof(double), st);
    cudaEventRecord(ev[0], st);
    for (int i = 0; i < n; ++i) {
        if (u->ops[i](st)) { u->error = "kernel launch failed"; return -1; }
        cudaEventRecord(ev[i + 1], st);
    }
    cudaStreamSynchronize(st);
    for (int i = 0; i < n; ++i) {
        cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
        kinds[i] = u->op_kinds[i];
        flops[i] = u->op_flops[i];
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return n;
}

int unet_forward_ncdhw(UNet* u, const float* feat_f32, int batch, float* out, cudaStream_t st) {
    if (!u->finalized) { u->error = "forward before finalize"; return 1; }
    if (batch < 1 || batch > u->NBmax) { u->error = "batch exceeds max_batch"; return 1; }
    const long long V = (long long)u->cfg.grid_size * u->cfg.grid_size * u->cfg.grid_size;
    if (launch_ncdhw_to_ndhwc_f16(feat_f32, u->feat_staging, batch, u->cfg.feature_channels, u->feat_cpad, V, st)) {
        u->error = "layout conversion launch failed";
        return 1;
    }
    return unet_forward(u, u->feat_staging, batch, out, st);
}

int unet_forward_host(UNet* u, const void* feat_host, int batch, float* out_host, cudaStream_t st) {
    if (!u->finalized) { u->error = "forward before finalize"; return 1; }
    if (batch < 1 || batch > u->NBmax) { u->error = "batch exceeds max_batch"; return 1; }
    if (u->feat_cpad != u->cfg.feature_channels) { u->error = "forward_host needs feature_channels % 64 == 0"; return 1; }
    const size_t V = (size_t)u->cfg.grid_size * u->cfg.grid_size * u->cfg.grid_size;
    if (cudaMemcpyAsync(u->feat_staging, feat_host, (size_t)batch * V * u->feat_cpad * 2, cudaMemcpyHostToDevice, st) != cudaSuccess) {
        u->error = "H2D copy failed"; return 1;
    }
    if (unet_forward(u, u->feat_staging, batch, u->out_staging, st)) return 1;
    if (cudaMemcpyAsync(out_host, u->out_staging, (size_t)batch * u->cfg.out_channels * V * 4, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
        u->error = "D2H copy failed"; return 1;
    }
    if (cudaStreamSynchronize(st) != cudaSuccess) { u->error = "stream sync failed"; return 1; }
    return check_err_flag(u);
}

int64_t unet_debug_fetch(UNet* u, const char* name, float* host_out, int64_t capacity) {
    auto it = u->named.find(name);
    if (it == u->named.end()) { u->error = std::string("no such activation: ") + name; return -1; }
    const DevT& t = it->second;
    const int64_t n = (int64_t)u->cur_nb * t.sp * t.sp * t.sp * t.C;
    if (n > capacity) { u->error = "debug_fetch: buffer too small"; return -2; }
    if (cudaDeviceSynchronize() != cudaSuccess) { u->error = "sync failed"; return -3; }
    if (check_err_flag(u)) return -4;
    cudaMemcpy(host_out, t.p, (size_t)n * 4, cudaMemcpyDeviceToHost);
    return n;
}

const std::string& unet_error(UNet* u) { return u->error; }
int unet_launch_count(UNet* u) {
    int n = 1;
    for (auto& c : u->convs) n += c->plan.needs_zero ? 1 : 0;
    return n + (int)u->ops.size();
}
double unet_flops(UNet* u) { return u->flops; }
int unet_check(UNet* u) {
    if (cudaDeviceSynchronize() != cudaSuccess) { u->error = "CUDA error"; return 1; }
    return check_err_flag(u);
}
void unet_destroy(UNet* u) { delete u; }

}  // namespace pixie
