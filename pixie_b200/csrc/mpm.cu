// MLS-MPM / APIC substep for sm_100a.  Replaces MPM_Simulator_WARP.p2g2p
// (third_party/PhysGaussian/mpm_solver_warp/mpm_solver_warp.py:514-637) and the Warp kernels it
// launches (mpm_utils.py:295-588, BC closures mpm_solver_warp.py:785-1179).
//
// One substep = two launches (mpm_fused.cuh), replayed from CUDA graphs with the simulation clock on the device:
//   mpm_fused_kernel   : g2p(i) -> particle BCs / return map / stress(i+1) -> warp-aggregated p2g(i+1), on a private
//                        cell-sorted SoA copy of the particle state (grid node = float4 {mv.xyz, m})
//   mpm_gridbox_kernel : normalise + gravity + damping + every grid BC (device BC table, registration order) -> grid_v over
//                        the particles' node box; clears the {mv, m} nodes it consumed (zero_grid fused away); advances the
//                        clock and the moving cuboids (the reference's host-side `modify`, mpm_solver_warp.py:899-905,
//                        and `self.time += dt`, :637)
// In slab-decomposed runs the grid sweep also adds the neighbours' partial sums on the shared planes (device-side exchange).  This file holds the small setup /
// export kernels (on the caller's arrays) and the host side.
#include "mpm.cuh"
#include "mpm_math.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cub/cub.cuh>

namespace pixie {

using namespace mpm;

namespace {

constexpr int kMaxBC = 256;    // release_particles_sequentially registers 50 modifiers per call (two calls + a scene's own BCs fit)

struct DevBC {
    int kind;
    float point[3], normal[3], size[3], velocity[3];
    float start_time, end_time, friction;
    int surface_type, reset;
    float h1[3], h2[3], hhr[2];
    float rotation_scale, translation_scale;
    const int* mask;
};

struct DevState {
    // particles
    float *x, *v, *F, *F_trial, *C, *stress, *R, *cov, *init_cov;
    float *vol, *mass, *density, *E, *nu, *mu, *lam, *bulk, *yield_stress;
    int *material, *selection;
    // grid
    float4* grid_mv;    // {momentum.xyz, mass}
    float4* grid_v;     // {velocity.xyz, 0}
    // clock + BCs
    double* time;
    DevBC* bcs;
    int n_bc;
    // scalars
    int n, n_grid;
    float dx, inv_dx;
    float gx, gy, gz;
    float rpic_damping, grid_v_damping_scale, alpha, hardening, xi, plastic_viscosity, softening;
    int update_cov_with_F;
};

__device__ __forceinline__ M3 load_m3(const float* p, int i) {
    M3 a;
#pragma unroll
    for (int k = 0; k < 9; ++k) a.m[k] = p[(size_t)i * 9 + k];
    return a;
}
__device__ __forceinline__ void store_m3(float* p, int i, const M3& a) {
#pragma unroll
    for (int k = 0; k < 9; ++k) p[(size_t)i * 9 + k] = a.m[k];
}

// ------------------------------------------------------------------------------------------ setup kernels
__global__ void mpm_mu_lam_kernel(const DevState s) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    const float E = s.E[p], nu = s.nu[p];
    s.mu[p] = E / (2.0f * (1.0f + nu));
    s.lam[p] = E * nu / ((1.0f + nu) * (1.0f - 2.0f * nu));
}
__global__ void mpm_bulk_kernel(const DevState s) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    s.bulk[p] = s.lam[p] + 2.f / 3.f * s.mu[p];
}
__global__ void mpm_mass_kernel(const DevState s) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    s.mass[p] = s.density[p] * s.vol[p];
}
__global__ void mpm_cov_from_F_kernel(const DevState s) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    const M3 F = load_m3(s.F_trial, p);
    const float* ic = s.init_cov + (size_t)p * 6;
    M3 c0;
    c0.m[0] = ic[0]; c0.m[1] = ic[1]; c0.m[2] = ic[2]; c0.m[3] = ic[1]; c0.m[4] = ic[3]; c0.m[5] = ic[4];
    c0.m[6] = ic[2]; c0.m[7] = ic[4]; c0.m[8] = ic[5];
    const M3 c = m3_mul_t(m3_mul(F, c0), F);
    float* o = s.cov + (size_t)p * 6;
    o[0] = c.m[0]; o[1] = c.m[1]; o[2] = c.m[2]; o[3] = c.m[4]; o[4] = c.m[5]; o[5] = c.m[8];
}
__global__ void mpm_R_from_F_kernel(const DevState s) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    const M3 F = load_m3(s.F_trial, p);
    M3 U, V; V3 sig;
    svd3(F, U, sig, V);
    // svd3 already returns proper rotations, so the det < 0 fix-ups of compute_R_from_F (:568-576) are no-ops
    const M3 R = m3_mul_t(U, V);
    store_m3(s.R, p, m3_t(R));
}
__global__ void mpm_additional_params_kernel(const DevState s, const float* __restrict__ boxes, int n_boxes) {
    __shared__ float sb[128 * 10];
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    float px = 0, py = 0, pz = 0;
    if (p < s.n) { px = s.x[3 * p]; py = s.x[3 * p + 1]; pz = s.x[3 * p + 2]; }
    int hit = -1;
    float hv[4] = {0, 0, 0, 0};
    for (int b0 = 0; b0 < n_boxes; b0 += 128) {
        const int nb = min(128, n_boxes - b0);
        __syncthreads();
        for (int i = threadIdx.x; i < nb * 10; i += blockDim.x) sb[i] = boxes[(size_t)b0 * 10 + i];
        __syncthreads();
        for (int b = 0; b < nb; ++b) {
            const float* B = sb + b * 10;
            if (px > B[0] - B[3] && px < B[0] + B[3] && py > B[1] - B[4] && py < B[1] + B[4] &&
                pz > B[2] - B[5] && pz < B[2] + B[5]) {
                hit = b0 + b; hv[0] = B[6]; hv[1] = B[7]; hv[2] = B[8]; hv[3] = B[9];   // later boxes override
            }
        }
    }
    if (p < s.n && hit >= 0) {
        s.E[p] = hv[0]; s.nu[p] = hv[1]; s.density[p] = hv[2]; s.material[p] = (int)hv[3];
    }
}
__global__ void mpm_select_box_kernel(const DevState s, float3 point, float3 size, int* mask) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    const float ox = s.x[3 * p] - point.x, oy = s.x[3 * p + 1] - point.y, oz = s.x[3 * p + 2] - point.z;
    mask[p] = (fabsf(ox) < size.x && fabsf(oy) < size.y && fabsf(oz) < size.z) ? 1 : 0;
}
__global__ void mpm_select_cyl_kernel(const DevState s, float3 point, float3 normal, float half_height, float radius, int* mask) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= s.n) return;
    const float ox = s.x[3 * p] - point.x, oy = s.x[3 * p + 1] - point.y, oz = s.x[3 * p + 2] - point.z;
    const float on = ox * normal.x + oy * normal.y + oz * normal.z;
    const float vd = fabsf(on);
    const float hx = ox - on * normal.x, hy = oy - on * normal.y, hz = oz - on * normal.z;
    const float hd = sqrtf(hx * hx + hy * hy + hz * hz);
    mask[p] = (vd < half_height && hd < radius) ? 1 : 0;
}

#include "mpm_fused.cuh"

}  // namespace

// ============================================================================================ host
struct Mpm {
    int n = 0, n_grid = 0;
    int n_active = 0;                  // particles [0, n_active) are live (slab mode migrates particles between ranks)
    int x_begin = 0, x_end = 0;        // grid planes this instance updates ([0, n_grid) unless slab-decomposed)
    float grid_lim = 1.f;
    void* fields[PIXIE_MPM_FIELD_COUNT] = {nullptr};
    pixie_mpm_params params{};
    std::vector<DevBC> bcs;
    float4* grid_mv = nullptr;
    float4* grid_v = nullptr;
    DevBC* d_bcs = nullptr;
    bool graph_valid = false;          // false: parameters / BCs changed, captured launches are stale
    // a few cached CUDA graphs keyed by (substep count, clock parity + grid parity, dt)
    static constexpr int kGraphSlots = 4;
    struct GraphSlot { cudaGraphExec_t exec = nullptr; int count = 0, parity = 0, launches = 0; double dt = 0; } graphs[kGraphSlots];
    int graph_next = 0;
    std::string error;

    // ---- cell order (radix sort of base-cell keys) = physical order of the private particle copy
    int *cell_order = nullptr, *cell_keys = nullptr, *cell_keys_sorted = nullptr, *cell_idx = nullptr;
    void* cub_tmp = nullptr;
    size_t cub_bytes = 0;

    // ---- fused path (mpm_fused.cuh): private cell-sorted SoA copy of the particle state
    struct FsBuf { float* f = nullptr; int *material = nullptr, *selection = nullptr, *perm = nullptr; } fs[2];
    int cap = 0;
    int* d_box = nullptr;              // [6] node box swept by the grid kernel
    double* tslots = nullptr;          // [2] clock, by substep parity
    float* pts = nullptr;              // [2][kMaxBC][3] collider points (the cuboid ones move), by substep parity
    int tpar = 0;
    bool internal_valid = false;       // sorted state mirrors the caller's arrays (+ steps taken since)
    bool user_stale = false;           // sorted state is ahead of the caller's arrays
    int steps_since_sort = 0;
    // ---- slab-decomposed runs on the fused path: exchange buffer = [SlabFlags][grid_mv], neighbours' buffers, overlap totals
    uint8_t* xbuf = nullptr;           // owns grid_mv (+ the flags block in front of it): one allocation, one IPC handle
    bool slab = false;
    int slab_x0 = 0, slab_x1 = 0, slab_slack = 1;
    const uint8_t* peer_xbuf[2] = {nullptr, nullptr};
    float4* grid_mv_alt = nullptr;     // second {mv, m} grid (slab mode alternates between the two by substep parity)
    int gpar = 0;                      // which of the two grids the next scatter targets (0 outside slab mode)
    int ov_lo[2] = {0, 0}, ov_hi[2] = {0, 0};
    bool g2p_pending = false;          // slab phases: the gather of the last finished substep has not run yet
    float slab_dt = 0.f;               // ... and the dt it has to use
    long long launches = 0;            // kernels of this library launched for this handle (bench.py's gpu_launches)
};

static constexpr int kFusedGraphSteps = 50;    // substeps per graph replay
static constexpr int kMinGraphSteps = 4;       // shorter batches are launched directly
static constexpr int kResortEvery = 100;       // substeps between re-sorts; CFL keeps a particle within ~a cell of its slot far longer
static constexpr int kBoxMargin = 2;           // nodes added around the particles' node box at every sort

static DevState make_state(Mpm* m) {
    DevState s{};
    auto f = [&](int id) { return reinterpret_cast<float*>(m->fields[id]); };
    s.x = f(PIXIE_MPM_X); s.v = f(PIXIE_MPM_V); s.F = f(PIXIE_MPM_F); s.F_trial = f(PIXIE_MPM_F_TRIAL);
    s.C = f(PIXIE_MPM_C); s.stress = f(PIXIE_MPM_STRESS); s.R = f(PIXIE_MPM_R); s.cov = f(PIXIE_MPM_COV);
    s.init_cov = f(PIXIE_MPM_INIT_COV); s.vol = f(PIXIE_MPM_VOL); s.mass = f(PIXIE_MPM_MASS);
    s.density = f(PIXIE_MPM_DENSITY); s.E = f(PIXIE_MPM_E); s.nu = f(PIXIE_MPM_NU); s.mu = f(PIXIE_MPM_MU);
    s.lam = f(PIXIE_MPM_LAM); s.bulk = f(PIXIE_MPM_BULK); s.yield_stress = f(PIXIE_MPM_YIELD);
    s.material = reinterpret_cast<int*>(m->fields[PIXIE_MPM_MATERIAL]);
    s.selection = reinterpret_cast<int*>(m->fields[PIXIE_MPM_SELECTION]);
    s.grid_mv = m->grid_mv; s.grid_v = m->grid_v; s.time = m->tslots; s.bcs = m->d_bcs; s.n_bc = (int)m->bcs.size();
    s.n = m->n_active; s.n_grid = m->n_grid;
    // dx, inv_dx exactly as mpm_solver_warp.py:61-66 (Python doubles rounded to fp32 members)
    s.dx = (float)((double)m->grid_lim / (double)m->n_grid);
    s.inv_dx = (float)((double)m->n_grid / (double)m->grid_lim);
    const pixie_mpm_params& q = m->params;
    s.gx = q.gravity[0]; s.gy = q.gravity[1]; s.gz = q.gravity[2];
    s.rpic_damping = q.rpic_damping; s.grid_v_damping_scale = q.grid_v_damping_scale; s.alpha = q.alpha;
    s.hardening = q.hardening; s.xi = q.xi; s.plastic_viscosity = q.plastic_viscosity; s.softening = q.softening;
    s.update_cov_with_F = q.update_cov_with_F;
    return s;
}

void mpm_destroy(Mpm* m);
int mpm_sync(Mpm* m, cudaStream_t st);
static void fused_launch(Mpm* m, bool do_g2p, bool do_p2g, bool write_all, float dt, cudaStream_t st);

// ---------------------------------------------------------------------------------- sort scratch (both paths)
static int sort_alloc(Mpm* m) {
    if (m->cell_order) return 0;
    const size_t cap = (size_t)m->n;
    if (cudaMalloc(&m->cell_order, cap * sizeof(int)) != cudaSuccess || cudaMalloc(&m->cell_keys, cap * sizeof(int)) != cudaSuccess ||
        cudaMalloc(&m->cell_keys_sorted, cap * sizeof(int)) != cudaSuccess || cudaMalloc(&m->cell_idx, cap * sizeof(int)) != cudaSuccess) {
        m->error = "cudaMalloc failed (cell order)"; return 1;
    }
    cub::DeviceRadixSort::SortPairs(nullptr, m->cub_bytes, m->cell_keys, m->cell_keys_sorted, m->cell_idx, m->cell_order, (int)cap, 0, 32, 0);
    if (cudaMalloc(&m->cub_tmp, m->cub_bytes) != cudaSuccess) { m->error = "cudaMalloc failed (sort scratch)"; return 1; }
    return 0;
}
static int key_bits(const Mpm* m) {
    int bits = 1;
    while ((1ll << bits) < (long long)m->n_grid * m->n_grid * m->n_grid) ++bits;
    return bits;
}

// ---------------------------------------------------------------------------------- fused path: host
static FsUser fs_user(Mpm* m) {
    FsUser u{};
    auto f = [&](int id) { return reinterpret_cast<float*>(m->fields[id]); };
    u.x = f(PIXIE_MPM_X); u.v = f(PIXIE_MPM_V); u.C = f(PIXIE_MPM_C); u.F = f(PIXIE_MPM_F); u.Ft = f(PIXIE_MPM_F_TRIAL);
    u.stress = f(PIXIE_MPM_STRESS); u.mass = f(PIXIE_MPM_MASS); u.vol = f(PIXIE_MPM_VOL); u.mu = f(PIXIE_MPM_MU); u.lam = f(PIXIE_MPM_LAM);
    u.bulk = f(PIXIE_MPM_BULK); u.ys = f(PIXIE_MPM_YIELD); u.cov = f(PIXIE_MPM_COV);
    u.material = reinterpret_cast<int*>(m->fields[PIXIE_MPM_MATERIAL]);
    u.selection = reinterpret_cast<int*>(m->fields[PIXIE_MPM_SELECTION]);
    return u;
}

static int fused_alloc(Mpm* m) {
    if (m->fs[0].f) return 0;
    m->cap = (m->n + 31) / 32 * 32;
    const size_t cap = (size_t)m->cap;
    bool ok = true;
    for (int b = 0; b < 2 && ok; ++b) {
        Mpm::FsBuf& s = m->fs[b];
        ok = cudaMalloc(&s.f, (size_t)FS_NFLOAT * cap * sizeof(float)) == cudaSuccess && cudaMalloc(&s.material, cap * sizeof(int)) == cudaSuccess &&
             cudaMalloc(&s.selection, cap * sizeof(int)) == cudaSuccess && cudaMalloc(&s.perm, cap * sizeof(int)) == cudaSuccess;
        if (ok) {
            cudaMemset(s.f, 0, (size_t)FS_NFLOAT * cap * sizeof(float));
            cudaMemset(s.material, 0, cap * sizeof(int)); cudaMemset(s.selection, 0, cap * sizeof(int)); cudaMemset(s.perm, 0, cap * sizeof(int));
        }
    }
    if (!ok) { m->error = "cudaMalloc failed (sorted particle state)"; return 1; }
    return sort_alloc(m);
}

// node box of the particles at `x` (+ margin) into m->d_box
static void fused_box(Mpm* m, const float* x, long long stride_comp, long long stride_part, cudaStream_t st) {
    const int init[6] = {m->n_grid, m->n_grid, m->n_grid, 0, 0, 0};
    cudaMemcpyAsync(m->d_box, init, sizeof(init), cudaMemcpyHostToDevice, st);
    const float inv_dx = (float)((double)m->n_grid / (double)m->grid_lim);
    fs_box_kernel<<<148, 256, 0, st>>>(x, stride_comp, stride_part, m->n_active, inv_dx, m->n_grid, kBoxMargin, m->d_box, 0);
    fs_box_kernel<<<1, 32, 0, st>>>(x, stride_comp, stride_part, m->n_active, inv_dx, m->n_grid, kBoxMargin, m->d_box, 1);
    m->launches += 2;
}

static int fused_sort(Mpm* m, const float* x, long long stride_comp, long long stride_part, cudaStream_t st) {
    m->steps_since_sort = 0;
    if (m->n_active <= 0) return 0;
    const float inv_dx = (float)((double)m->n_grid / (double)m->grid_lim);
    fs_key_kernel<<<(m->n_active + 255) / 256, 256, 0, st>>>(x, stride_comp, stride_part, m->n_active, inv_dx, m->n_grid, m->cell_keys, m->cell_idx);
    size_t bytes = m->cub_bytes;
    if (cub::DeviceRadixSort::SortPairs(m->cub_tmp, bytes, m->cell_keys, m->cell_keys_sorted, m->cell_idx, m->cell_order, m->n_active, 0, key_bits(m), st) != cudaSuccess) {
        m->error = "radix sort failed"; return 1;
    }
    m->steps_since_sort = 0;
    m->launches += 1;          // + the radix sort passes of cub (library kernels, not counted)
    return 0;
}

// caller's arrays -> sorted state
static int fused_gather_from_user(Mpm* m, cudaStream_t st) {
    if (fused_alloc(m)) return 1;
    const FsUser u = fs_user(m);
    if (fused_sort(m, u.x, 1, 3, st)) return 1;
    Mpm::FsBuf& d = m->fs[0];
    if (m->n_active > 0) fs_gather_kernel<<<(m->n_active + 255) / 256, 256, 0, st>>>(u, m->cell_order, m->n_active, m->cap, d.f, d.material, d.selection, d.perm,
                                                          m->params.update_cov_with_F ? 1 : 0);
    fused_box(m, u.x, 1, 3, st);
    m->launches += 1;
    m->internal_valid = true;
    m->user_stale = false;
    return cudaGetLastError() != cudaSuccess;
}

// re-sort of the live sorted state (between two launches of the particle kernel)
static int fused_resort(Mpm* m, cudaStream_t st) {
    Mpm::FsBuf& a = m->fs[0];
    Mpm::FsBuf& b = m->fs[1];
    if (fused_sort(m, a.f + (size_t)FS_X * m->cap, m->cap, 1, st)) return 1;
    if (m->n_active <= 0) return 0;
    fs_permute_kernel<<<(m->n_active + 255) / 256, 256, 0, st>>>(a.f, a.material, a.selection, a.perm, m->cell_order, m->n_active, m->cap, b.f, b.material,
                                                           b.selection, b.perm);
    // back into buffer 0: the captured graph and the launch arguments keep pointing at it
    const size_t cap = (size_t)m->cap;
    cudaMemcpyAsync(a.f, b.f, (size_t)FS_NFLOAT * cap * sizeof(float), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(a.material, b.material, cap * sizeof(int), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(a.selection, b.selection, cap * sizeof(int), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(a.perm, b.perm, cap * sizeof(int), cudaMemcpyDeviceToDevice, st);
    fused_box(m, a.f + (size_t)FS_X * m->cap, m->cap, 1, st);
    m->launches += 1;
    return cudaGetLastError() != cudaSuccess;
}

// sorted state -> caller's arrays (if it is ahead); afterwards the caller may mutate its arrays, so the sorted copy is
// considered out of date.
int mpm_sync(Mpm* m, cudaStream_t st) {
    if (m->g2p_pending && m->internal_valid) {        // slab phases: finish the last substep (gather) before anything is read
        fused_launch(m, true, false, true, m->slab_dt, st);
        m->g2p_pending = false;
    }
    if (m->user_stale) {
        const Mpm::FsBuf& s = m->fs[0];
        if (m->n_active > 0) fs_unsort_kernel<<<(m->n_active + 255) / 256, 256, 0, st>>>(fs_user(m), s.perm, m->n_active, m->cap, s.f, m->params.update_cov_with_F ? 1 : 0);
        m->user_stale = false;
        m->launches += 1;
        if (cudaGetLastError() != cudaSuccess) { m->error = "unsort launch failed"; return 1; }
    }
    m->internal_valid = false;
    return 0;
}

// Launch with programmatic stream serialisation (PDL): the kernel may be scheduled while its predecessor in the stream
// (or captured graph) is still draining; both kernels of the substep chain wait for it with griddepcontrol.wait.
template <typename... KArgs, typename... Args>
static void pdl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static inline size_t grid_bytes(const Mpm* m) { return (size_t)m->n_grid * m->n_grid * m->n_grid * sizeof(float4); }
static inline float4* scatter_grid(Mpm* m) { return (m->slab && m->gpar) ? m->grid_mv_alt : m->grid_mv; }
static inline int graph_parity(const Mpm* m) { return m->tpar | (m->gpar << 1); }

static FusedState fused_state(Mpm* m) {
    FusedState t{};
    const Mpm::FsBuf& s = m->fs[0];
    t.f = s.f; t.material = s.material; t.selection = s.selection; t.perm = s.perm;
    t.cap = m->cap; t.n = m->n_active;
    t.grid_v = m->grid_v; t.grid_mv = scatter_grid(m); t.box = m->d_box;
    t.bcs = m->d_bcs; t.n_bc = (int)m->bcs.size();
    t.n_particle_bc = 0;
    for (const DevBC& b : m->bcs) {
        if (b.kind < PIXIE_BC_IMPULSE) continue;
        if (t.n_particle_bc < kInlinePBC) {
            ParticleBC& q = t.pbc[t.n_particle_bc];
            q.kind = b.kind; q.start_time = b.start_time; q.end_time = b.end_time; q.mask = b.mask;
            q.rotation_scale = b.rotation_scale; q.translation_scale = b.translation_scale;
            for (int a = 0; a < 3; ++a) { q.velocity[a] = b.velocity[a]; q.point[a] = b.point[a]; q.normal[a] = b.normal[a]; q.h1[a] = b.h1[a]; q.h2[a] = b.h2[a]; }
        }
        ++t.n_particle_bc;
    }
    t.n_pbc_inline = t.n_particle_bc <= kInlinePBC ? t.n_particle_bc : -1;
    t.n_grid = m->n_grid;
    t.dx = (float)((double)m->grid_lim / (double)m->n_grid);
    t.inv_dx = (float)((double)m->n_grid / (double)m->grid_lim);
    const pixie_mpm_params& q = m->params;
    t.rpic_damping = q.rpic_damping; t.alpha = q.alpha; t.hardening = q.hardening; t.xi = q.xi;
    t.plastic_viscosity = q.plastic_viscosity; t.softening = q.softening;
    t.update_cov_with_F = q.update_cov_with_F;
    if (m->slab) {
        SlabFlags* fl = reinterpret_cast<SlabFlags*>(m->xbuf);
        t.slab_step = &fl->step; t.slab_err = &fl->error;
        t.base_lo = m->peer_xbuf[0] ? m->slab_x0 - m->slab_slack : -(1 << 30);
        t.base_hi = m->peer_xbuf[1] ? m->slab_x1 + m->slab_slack : (1 << 30);
    }
    return t;
}

static void fused_launch(Mpm* m, bool do_g2p, bool do_p2g, bool write_all, float dt, cudaStream_t st) {
    FusedState t = fused_state(m);
    t.do_g2p = do_g2p; t.do_p2g = do_p2g; t.write_all = write_all;
    t.time = m->tslots + m->tpar;                 // clock of the substep whose stress / scatter runs in this launch
    // 88 registers per thread: 32-thread blocks pack 23 per SM (736 threads), so 100k particles are one wave on 148 SMs
    const int blocks = (std::max(m->n_active, 1) + kFusedThreads - 1) / kFusedThreads;
    pdl_launch(mpm_fused_kernel, dim3(blocks), dim3(kFusedThreads), st, t, dt);
    m->launches += 1;
}

static void gridbox_launch(Mpm* m, bool publish_scatter, float dt, double dt_d, cudaStream_t st) {
    GridBoxArgs g{};
    g.grid_mv = scatter_grid(m); g.grid_v = m->grid_v; g.box = m->d_box;
    g.time_in = m->tslots + m->tpar; g.time_out = m->tslots + (m->tpar ^ 1);
    g.pts_in = m->pts + (size_t)m->tpar * kMaxBC * 3; g.pts_out = m->pts + (size_t)(m->tpar ^ 1) * kMaxBC * 3;
    g.bcs = m->d_bcs; g.n_bc = (int)m->bcs.size();
    g.n_grid = m->n_grid; g.x_begin = m->x_begin; g.x_end = m->x_end;
    if (m->slab) {
        g.mine = reinterpret_cast<SlabFlags*>(m->xbuf);
        g.grid_other = m->gpar ? m->grid_mv : m->grid_mv_alt;
        g.publish_scatter = publish_scatter ? 1 : 0;
        for (int sd = 0; sd < 2; ++sd) {
            g.peer[sd] = reinterpret_cast<const SlabFlags*>(m->peer_xbuf[sd]);
            g.peer_mv[sd] = m->peer_xbuf[sd] ? reinterpret_cast<const float4*>(m->peer_xbuf[sd] + sizeof(SlabFlags) + (size_t)m->gpar * grid_bytes(m)) : nullptr;
            g.ov_lo[sd] = m->ov_lo[sd]; g.ov_hi[sd] = m->ov_hi[sd];
        }
    }
    g.dx = (float)((double)m->grid_lim / (double)m->n_grid);
    const pixie_mpm_params& q = m->params;
    g.gx = q.gravity[0]; g.gy = q.gravity[1]; g.gz = q.gravity[2]; g.grid_v_damping_scale = q.grid_v_damping_scale;
    // enough blocks for two per SM; the kernel strides over the (usually much smaller than n_grid^3) node box
    pdl_launch(mpm_gridbox_kernel, dim3(296), dim3(256), st, g, dt, dt_d);
    m->launches += 1;
    m->tpar ^= 1;
    if (m->slab) m->gpar ^= 1;
}

// `count` substeps as: scatter(0) | grid(0) | g2p(0)+scatter(1) | ... | grid(count-1) | g2p(count-1)
static void fused_batch(Mpm* m, int count, float dt, double dt_d, cudaStream_t st) {
    fused_launch(m, false, true, count == 1, dt, st);
    for (int i = 0; i < count; ++i) {
        gridbox_launch(m, true, dt, dt_d, st);
        if (i + 1 < count) fused_launch(m, true, true, i + 2 == count, dt, st);
        else fused_launch(m, true, false, true, dt, st);
    }
}

// CUDA graph of `count` substeps starting at clock parity `m->tpar` (cached: the 50-substep batch of long rollouts and, for
// slab runs, the chunk between two particle migrations)
static cudaGraphExec_t fused_graph(Mpm* m, int count, float dt, double dt_d) {
    for (auto& g : m->graphs)
        if (g.exec && g.count == count && g.parity == graph_parity(m) && g.dt == dt_d) return g.exec;
    Mpm::GraphSlot& slot = m->graphs[m->graph_next];
    m->graph_next = (m->graph_next + 1) % Mpm::kGraphSlots;
    if (slot.exec) { cudaGraphExecDestroy(slot.exec); slot.exec = nullptr; }
    cudaStream_t cs;
    cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
    cudaGraph_t g = nullptr;
    const int par0 = m->tpar, gpar0 = m->gpar, key0 = graph_parity(m);
    const long long launches0 = m->launches;
    bool ok = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
        fused_batch(m, count, dt, dt_d, cs);
        ok = cudaStreamEndCapture(cs, &g) == cudaSuccess && g;
    }
    slot.launches = (int)(m->launches - launches0);
    m->tpar = par0; m->gpar = gpar0;                   // capture did not run anything
    m->launches = launches0;
    if (ok) ok = cudaGraphInstantiate(&slot.exec, g, 0) == cudaSuccess;
    if (g) cudaGraphDestroy(g);
    cudaStreamDestroy(cs);
    if (!ok) { cudaGetLastError(); slot.exec = nullptr; return nullptr; }
    slot.count = count; slot.parity = key0; slot.dt = dt_d;
    return slot.exec;
}

static int mpm_step_fused(Mpm* m, int n_substeps, double dt_d, cudaStream_t st) {
    const float dt = (float)dt_d;
    if (!m->internal_valid && fused_gather_from_user(m, st)) return 1;
    if (!m->graph_valid) {                              // parameters / BCs / bindings changed: captured launches are stale
        for (auto& g : m->graphs) if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
        m->graph_valid = true;
    }
    int done = 0;
    while (done < n_substeps) {
        if (m->steps_since_sort >= kResortEvery && fused_resort(m, st)) return 1;
        int count = std::min(n_substeps - done, kFusedGraphSteps);
        count = std::min(count, std::max(1, kResortEvery - m->steps_since_sort));
        cudaGraphExec_t g = count >= kMinGraphSteps ? fused_graph(m, count, dt, dt_d) : nullptr;
        if (g) {
            if (cudaGraphLaunch(g, st) != cudaSuccess) { m->error = "cudaGraphLaunch failed"; return 1; }
            for (auto& sl : m->graphs) if (sl.exec == g) m->launches += sl.launches;
            if (count & 1) { m->tpar ^= 1; if (m->slab) m->gpar ^= 1; }   // the replay advanced the clock `count` times
        } else {
            fused_batch(m, count, dt, dt_d, st);
        }
        done += count;
        m->steps_since_sort += count;
    }
    m->user_stale = true;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { m->error = std::string("kernel launch failed: ") + cudaGetErrorString(e); return 1; }
    return 0;
}

Mpm* mpm_create(int n_particles, int n_grid, float grid_lim, std::string& err) {
    if (n_particles <= 0 || n_grid <= 0) { err = "n_particles and n_grid must be positive"; return nullptr; }
    auto* m = new Mpm();
    m->n = n_particles; m->n_active = n_particles; m->n_grid = n_grid; m->grid_lim = grid_lim;
    m->x_begin = 0; m->x_end = n_grid;
    m->params.n_grid = n_grid; m->params.grid_lim = grid_lim;
    m->params.grid_v_damping_scale = 1.1f;                 // mpm_solver_warp.py:92
    {
        // friction_angle 25 deg default (:83-86), evaluated like the reference (float math on 3.14159265)
        const double sin_phi = sin(25.0 / 180.0 * 3.14159265);
        m->params.alpha = (float)(sqrt(2.0 / 3.0) * 2.0 * sin_phi / (3.0 - sin_phi));
    }
    m->params.softening = 0.1f;
    const size_t nodes = (size_t)n_grid * n_grid * n_grid;
    if (cudaMalloc(&m->xbuf, sizeof(SlabFlags) + nodes * sizeof(float4)) != cudaSuccess ||
        cudaMalloc(&m->grid_v, nodes * sizeof(float4)) != cudaSuccess ||
        cudaMalloc(&m->d_bcs, kMaxBC * sizeof(DevBC)) != cudaSuccess ||
        cudaMalloc(&m->d_box, 6 * sizeof(int)) != cudaSuccess ||
        cudaMalloc(&m->tslots, 2 * sizeof(double)) != cudaSuccess ||
        cudaMalloc(&m->pts, (size_t)2 * kMaxBC * 3 * sizeof(float)) != cudaSuccess) {
        err = "cudaMalloc failed (no CUDA device?)";
        delete m;
        return nullptr;
    }
    m->grid_mv = reinterpret_cast<float4*>(m->xbuf + sizeof(SlabFlags));
    cudaMemset(m->xbuf, 0, sizeof(SlabFlags) + nodes * sizeof(float4));
    cudaMemset(m->grid_v, 0, nodes * sizeof(float4));
    cudaMemset(m->tslots, 0, 2 * sizeof(double));
    cudaMemset(m->pts, 0, (size_t)2 * kMaxBC * 3 * sizeof(float));
    return m;
}

void mpm_destroy(Mpm* m) {
    if (!m) return;
    cudaFree(m->cell_order); cudaFree(m->cell_keys); cudaFree(m->cell_keys_sorted); cudaFree(m->cell_idx); cudaFree(m->cub_tmp);
    for (int b = 0; b < 2; ++b) { cudaFree(m->fs[b].f); cudaFree(m->fs[b].material); cudaFree(m->fs[b].selection); cudaFree(m->fs[b].perm); }
    cudaFree(m->d_box); cudaFree(m->tslots); cudaFree(m->pts);
    for (auto& g : m->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    cudaFree(m->xbuf);
    cudaFree(m->grid_v); cudaFree(m->d_bcs);
    delete m;
}

int mpm_bind(Mpm* m, int field, void* ptr) {
    if (field < 0 || field >= PIXIE_MPM_FIELD_COUNT) { m->error = "bad field id"; return 1; }
    if (mpm_sync(m, 0)) return 1;          // flush results into the arrays bound so far before one of them changes
    m->fields[field] = ptr;
    return 0;
}
int mpm_set_params(Mpm* m, const pixie_mpm_params& p) {
    if (mpm_sync(m, 0)) return 1;
    if (p.n_grid != m->n_grid) {
        // set_parameters_dict re-allocates the grids when n_grid changes (mpm_solver_warp.py:318-343)
        if (m->slab) { m->error = "n_grid cannot change in slab mode"; return 1; }
        cudaDeviceSynchronize();
        cudaFree(m->xbuf);
        cudaFree(m->grid_v);
        m->xbuf = nullptr;
        const size_t nodes = (size_t)p.n_grid * p.n_grid * p.n_grid;
        if (cudaMalloc(&m->xbuf, sizeof(SlabFlags) + nodes * sizeof(float4)) != cudaSuccess ||
            cudaMalloc(&m->grid_v, nodes * sizeof(float4)) != cudaSuccess) { m->error = "cudaMalloc failed"; return 1; }
        m->grid_mv = reinterpret_cast<float4*>(m->xbuf + sizeof(SlabFlags));
        m->grid_mv_alt = nullptr;
        cudaMemset(m->xbuf, 0, sizeof(SlabFlags) + nodes * sizeof(float4));
        cudaMemset(m->grid_v, 0, nodes * sizeof(float4));
        m->n_grid = p.n_grid;
        m->x_begin = 0; m->x_end = p.n_grid;
    }
    m->grid_lim = p.grid_lim;
    m->params = p;
    m->graph_valid = false;
    return 0;
}
int mpm_add_bc(Mpm* m, const pixie_mpm_bc& b) {
    if ((int)m->bcs.size() >= kMaxBC) { m->error = "too many boundary conditions (limit " + std::to_string(kMaxBC) + ")"; return 1; }
    if (b.kind >= PIXIE_BC_IMPULSE && !b.mask_dev) { m->error = "particle BC needs a mask"; return 1; }
    DevBC d{};
    d.kind = b.kind;
    for (int i = 0; i < 3; ++i) {
        d.point[i] = b.point[i]; d.normal[i] = b.normal[i]; d.size[i] = b.size[i]; d.velocity[i] = b.velocity[i];
        d.h1[i] = b.horizontal_axis_1[i]; d.h2[i] = b.horizontal_axis_2[i];
    }
    d.hhr[0] = b.half_height_and_radius[0]; d.hhr[1] = b.half_height_and_radius[1];
    d.start_time = b.start_time; d.end_time = b.end_time; d.friction = b.friction;
    d.surface_type = b.surface_type; d.reset = b.reset;
    d.rotation_scale = b.rotation_scale; d.translation_scale = b.translation_scale;
    d.mask = b.mask_dev;
    if (mpm_sync(m, 0)) return 1;
    m->bcs.push_back(d);
    // append in place: the device tables also hold the *moved* cuboid positions of earlier BCs
    const size_t k = m->bcs.size() - 1;
    cudaMemcpy(m->d_bcs + k, &d, sizeof(DevBC), cudaMemcpyHostToDevice);
    cudaMemcpy(m->pts + 3 * k, d.point, 3 * sizeof(float), cudaMemcpyHostToDevice);
    cudaMemcpy(m->pts + (size_t)kMaxBC * 3 + 3 * k, d.point, 3 * sizeof(float), cudaMemcpyHostToDevice);
    m->graph_valid = false;
    return 0;
}
int mpm_clear_bcs(Mpm* m) { m->bcs.clear(); m->graph_valid = false; return 0; }
int mpm_set_time(Mpm* m, double t) {
    const double both[2] = {t, t};
    return cudaMemcpy(m->tslots, both, sizeof(both), cudaMemcpyHostToDevice) != cudaSuccess;
}
int mpm_get_time(Mpm* m, double* t) {
    const double* src = m->tslots + m->tpar;
    return cudaMemcpy(t, src, sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess;
}

static int check_bound(Mpm* m) {
    static const int need[] = {PIXIE_MPM_X, PIXIE_MPM_V, PIXIE_MPM_F, PIXIE_MPM_F_TRIAL, PIXIE_MPM_C, PIXIE_MPM_STRESS,
                               PIXIE_MPM_VOL, PIXIE_MPM_MASS, PIXIE_MPM_MU, PIXIE_MPM_LAM, PIXIE_MPM_BULK,
                               PIXIE_MPM_YIELD, PIXIE_MPM_MATERIAL, PIXIE_MPM_SELECTION};
    for (int id : need)
        if (!m->fields[id]) { m->error = "field " + std::to_string(id) + " is not bound"; return 1; }
    if (m->params.update_cov_with_F && !m->fields[PIXIE_MPM_COV]) { m->error = "cov not bound"; return 1; }
    return 0;
}

int mpm_step(Mpm* m, int n_substeps, double dt_d, cudaStream_t st) {
    if (check_bound(m)) return 1;
    if (n_substeps <= 0) return 0;
    if (m->g2p_pending && m->internal_valid) {          // phase-driven substeps came first: complete the last one
        fused_launch(m, true, false, true, m->slab_dt, st);
        m->g2p_pending = false;
    }
    return mpm_step_fused(m, n_substeps, dt_d, st);
}

#define PIXIE_SIMPLE_LAUNCH(kernel)                                                         \
    if (mpm_sync(m, st)) return 1;                                                          \
    const DevState s = make_state(m);                                                       \
    kernel<<<(m->n + 255) / 256, 256, 0, st>>>(s);                                          \
    const cudaError_t e = cudaGetLastError();                                               \
    if (e != cudaSuccess) { m->error = cudaGetErrorString(e); return 1; }                   \
    return 0;

int mpm_compute_mu_lam(Mpm* m, cudaStream_t st) { PIXIE_SIMPLE_LAUNCH(mpm_mu_lam_kernel) }
int mpm_compute_bulk(Mpm* m, cudaStream_t st) { PIXIE_SIMPLE_LAUNCH(mpm_bulk_kernel) }
int mpm_compute_mass(Mpm* m, cudaStream_t st) { PIXIE_SIMPLE_LAUNCH(mpm_mass_kernel) }
int mpm_compute_cov_from_F(Mpm* m, cudaStream_t st) { PIXIE_SIMPLE_LAUNCH(mpm_cov_from_F_kernel) }
int mpm_compute_R_from_F(Mpm* m, cudaStream_t st) { PIXIE_SIMPLE_LAUNCH(mpm_R_from_F_kernel) }

int mpm_apply_additional_params(Mpm* m, const float* boxes_host, int n_boxes, cudaStream_t st) {
    if (n_boxes <= 0) return 0;
    if (mpm_sync(m, st)) return 1;
    float* d = nullptr;
    if (cudaMalloc(&d, (size_t)n_boxes * 10 * 4) != cudaSuccess) { m->error = "cudaMalloc failed"; return 1; }
    cudaMemcpyAsync(d, boxes_host, (size_t)n_boxes * 10 * 4, cudaMemcpyDefault, st);    // host or device source (UVA)
    const DevState s = make_state(m);
    mpm_additional_params_kernel<<<(m->n + 127) / 128, 128, 0, st>>>(s, d, n_boxes);
    cudaStreamSynchronize(st);
    cudaFree(d);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { m->error = cudaGetErrorString(e); return 1; }
    return 0;
}
int mpm_select_box(Mpm* m, const float* point, const float* size, int* mask, cudaStream_t st) {
    if (mpm_sync(m, st)) return 1;
    const DevState s = make_state(m);
    mpm_select_box_kernel<<<(m->n + 255) / 256, 256, 0, st>>>(s, make_float3(point[0], point[1], point[2]),
                                                              make_float3(size[0], size[1], size[2]), mask);
    return cudaGetLastError() != cudaSuccess;
}
int mpm_select_cylinder(Mpm* m, const float* point, const float* normal, float hh, float radius, int* mask, cudaStream_t st) {
    if (mpm_sync(m, st)) return 1;
    const DevState s = make_state(m);
    mpm_select_cyl_kernel<<<(m->n + 255) / 256, 256, 0, st>>>(s, make_float3(point[0], point[1], point[2]),
                                                              make_float3(normal[0], normal[1], normal[2]), hh, radius, mask);
    return cudaGetLastError() != cudaSuccess;
}
int mpm_set_active_count(Mpm* m, int n_active) {
    if (n_active < 0 || n_active > m->n) { m->error = "active count exceeds the bound capacity"; return 1; }
    if (mpm_sync(m, 0)) return 1;          // results of the old live prefix go back first; the next step re-reads the arrays
    m->n_active = n_active;
    m->graph_valid = false;
    if (m->slab && m->grid_mv_alt) {
        // Slab mode calls this after every particle migration (all ranks have finished their substeps: the migration's
        // collectives sit behind them). The shared planes of the grid scattered into last still hold this rank's partial sums
        // (they are cleared one substep late, inside the node box); particles that just LEFT may have put some outside the
        // box of the particles that remain, so both grids' shared planes are cleared outright here.
        const size_t plane = (size_t)m->n_grid * m->n_grid * sizeof(float4);
        for (int sd = 0; sd < 2; ++sd) {
            if (!m->peer_xbuf[sd]) continue;
            const size_t off = (size_t)m->ov_lo[sd] * plane, len = (size_t)(m->ov_hi[sd] - m->ov_lo[sd]) * plane;
            cudaMemsetAsync(reinterpret_cast<uint8_t*>(m->grid_mv) + off, 0, len, 0);
            cudaMemsetAsync(reinterpret_cast<uint8_t*>(m->grid_mv_alt) + off, 0, len, 0);
        }
    }
    return 0;
}
// ---- slab mode (BASELINE config 5, no reference counterpart: the reference hard-wires "cuda:0", gs_simulation.py:441). The exchange buffer [SlabFlags][grid_mv] of each handle is made
//      visible to its x-neighbours (cudaIpc between processes, plain pointers inside one process); scatter, overlap
//      exchange and grid update then chain on the device with flag handshakes, no host in the loop.
int mpm_exchange_buffer(Mpm* m, void** base, size_t* bytes) {
    // slab mode alternates between two {mv, m} grids (see GridBoxArgs): the first request re-allocates the exchange buffer as
    // [SlabFlags][grid 0][grid 1], still ONE allocation = one IPC handle
    const size_t gb = grid_bytes(m);
    if (!m->grid_mv_alt) {
        if (mpm_sync(m, 0)) return 1;
        cudaDeviceSynchronize();
        uint8_t* nb = nullptr;
        if (cudaMalloc(&nb, sizeof(SlabFlags) + 2 * gb) != cudaSuccess) { m->error = "cudaMalloc failed (exchange buffer)"; return 1; }
        cudaMemset(nb, 0, sizeof(SlabFlags) + 2 * gb);
        cudaFree(m->xbuf);
        m->xbuf = nb;
        m->grid_mv = reinterpret_cast<float4*>(nb + sizeof(SlabFlags));
        m->grid_mv_alt = reinterpret_cast<float4*>(nb + sizeof(SlabFlags) + gb);
        m->graph_valid = false;
    }
    *base = m->xbuf;
    *bytes = sizeof(SlabFlags) + 2 * gb;
    return 0;
}
int mpm_slab_attach(Mpm* m, int x0, int x1, int slack, const void* left_xbuf, const void* right_xbuf) {
    if (x0 < 0 || x1 > m->n_grid || x0 >= x1 || slack < 0) { m->error = "bad slab range"; return 1; }
    if ((left_xbuf || right_xbuf) && (x1 - x0) < 2 + 2 * slack) { m->error = "slab narrower than 2 + 2*slack planes"; return 1; }
    if (mpm_sync(m, 0)) return 1;
    const int n = m->n_grid;
    m->slab = true; m->slab_x0 = x0; m->slab_x1 = x1; m->slab_slack = slack;
    m->peer_xbuf[0] = reinterpret_cast<const uint8_t*>(left_xbuf);
    m->peer_xbuf[1] = reinterpret_cast<const uint8_t*>(right_xbuf);
    // planes shared with a neighbour: both of them touch [x - slack, x + 2 + slack) around the interface x
    m->ov_lo[0] = std::max(0, x0 - slack); m->ov_hi[0] = std::min(n, x0 + 2 + slack);
    m->ov_lo[1] = std::max(0, x1 - slack); m->ov_hi[1] = std::min(n, x1 + 2 + slack);
    m->x_begin = left_xbuf ? m->ov_lo[0] : 0;
    m->x_end = right_xbuf ? m->ov_hi[1] : n;
    if (!m->grid_mv_alt) { void* b; size_t nb; if (mpm_exchange_buffer(m, &b, &nb)) return 1; }
    cudaMemset(m->xbuf, 0, sizeof(SlabFlags) + 2 * grid_bytes(m));
    m->gpar = 0;
    m->graph_valid = false;
    m->g2p_pending = false;
    return 0;
}
// One phase of a substep (single-process drivers sequence the phases of all slabs; a multi-process rank calls mpm_step).
int mpm_slab_phase(Mpm* m, int phase, double dt_d, cudaStream_t st) {
    if (!m->slab) { m->error = "not in slab mode"; return 1; }
    if (check_bound(m)) return 1;
    const float dt = (float)dt_d;
    if (phase == 0) {
        if (!m->internal_valid) { if (fused_gather_from_user(m, st)) return 1; m->g2p_pending = false; }
        else if (m->steps_since_sort >= kResortEvery && fused_resort(m, st)) return 1;
        fused_launch(m, m->g2p_pending, true, true, dt, st);
        pdl_launch(mpm_publish_kernel, dim3(1), dim3(32), st, reinterpret_cast<SlabFlags*>(m->xbuf));
        m->launches += 1;
        m->g2p_pending = false;
    } else if (phase == 1) {
        // nothing to launch: the overlap sums are formed inside the grid sweep (kept so that drivers written for the
        // scatter / exchange / finish sequence need no special case)
    } else if (phase == 2) {
        gridbox_launch(m, false, dt, dt_d, st);
        m->g2p_pending = true; m->slab_dt = dt;
        ++m->steps_since_sort;
        m->user_stale = true;
    } else { m->error = "bad phase"; return 1; }
    return cudaGetLastError() != cudaSuccess;
}
// Planes by which the farthest live particle's stencil base lies outside this slab's [x0, x1) (sides without a neighbour do
// not count), max-ed into the device int `d_out` (the caller zeroes it). Reads the sorted state when it is current, so a
// migration check costs one small kernel instead of a write-back of every field.
int mpm_slab_excursion(Mpm* m, int* d_out, cudaStream_t st) {
    if (!m->slab) { m->error = "not in slab mode"; return 1; }
    if (m->n_active <= 0) return 0;
    const float inv_dx = (float)((double)m->n_grid / (double)m->grid_lim);
    const int lo = m->peer_xbuf[0] ? m->slab_x0 : -(1 << 29);
    const int hi = m->peer_xbuf[1] ? m->slab_x1 : (1 << 29);
    const bool sorted = m->internal_valid && m->fs[0].f;
    if (sorted && m->g2p_pending) {                    // phase-driven runs: positions of the last substep first
        fused_launch(m, true, false, true, m->slab_dt, st);
        m->g2p_pending = false;
    }
    const float* x = sorted ? m->fs[0].f + (size_t)FS_X * m->cap : reinterpret_cast<const float*>(m->fields[PIXIE_MPM_X]);
    if (!x) { m->error = "positions not bound"; return 1; }
    fs_excursion_kernel<<<148, 256, 0, st>>>(x, sorted ? 1 : 3, m->n_active, inv_dx, lo, hi, d_out);
    m->launches += 1;
    return cudaGetLastError() != cudaSuccess;
}
int mpm_slab_error(Mpm* m, int* flag) {
    SlabFlags f{};
    if (cudaMemcpy(&f, m->xbuf, sizeof(f), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
    *flag = f.error;
    return 0;
}

int mpm_grid_ptrs(Mpm* m, float** mv4, float** v4) {
    *mv4 = reinterpret_cast<float*>(m->grid_mv);
    *v4 = reinterpret_cast<float*>(m->grid_v);
    return 0;
}
long long mpm_launch_count(Mpm* m) { return m->launches; }
const std::string& mpm_error(Mpm* m) { return m->error; }

}  // namespace pixie
