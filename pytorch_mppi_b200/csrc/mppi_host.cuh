// mppi_host.cuh — host side shared by the translation units of the library: parameter validation, launch geometry,
// argument packing, plans, and the per-model launch/plan templates.  The library is built from several translation
// units (mppi_b200.cu: C ABI + the model-independent kernels; mppi_model_tu.cu compiled once per (model, dtype):
// the fused / resident / states kernels of that model) so that it compiles in parallel; everything here has
// internal linkage (anonymous namespace) except the few declarations in namespace mppi_host that cross units.
#pragma once
#include <cuda_runtime.h>
#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <type_traits>

#include "../../include/mppi_b200.h"
#include "mppi_fused.cuh"
#include "mppi_resident.cuh"
#include "mppi_resident_host.h"

using namespace mppi;

namespace mppi_host {

// last error text of the calling thread (one definition, in mppi_b200.cu)
extern thread_local char g_cuda_err[512];

#define MPPI_MODEL_BLOCK_BYTES 12288     // largest Model::P<real> a kernel takes by value (the MLP's weights: 10 KB in fp64)

struct Geometry {
    int BD, BS, tps, nb, smem, occ, regs;   // BD = BS * tps threads per CTA, BS samples per tile
    int cluster;                            // thread-block-cluster size of the launch (1: none); nb is a multiple of it
    int npub;                               // sharded controllers: records published per rank and command (0: not sharded)
};

// Resident mode: the host side of the protocol (struct Resident, res_*) is csrc/mppi_resident_host.h; this file supplies its
// backend (cooperative launch / stream synchronise / stream query).
struct ResidentDevice {
    unsigned long long* host_box = nullptr;
    unsigned long long* board = nullptr;
    void* action_dev = nullptr;
    cudaStream_t stream = nullptr;
    unsigned long long idle_ns = 0;
};

struct Plan {
    MppiFusedParams p;
    const void* kernel;
    const void* res_kernel;            // resident_command_kernel<Model, real, V, sharded>, or nullptr when this plan cannot run resident
    int res_xchg;                      // always 0 (resident mode serves single-GPU controllers)
    Resident res;
    ResidentDevice resdev;
    Geometry g;
    int is_double, nx, upc_nu, pdl;
    unsigned long long epoch, host_epoch;
    unsigned long long res_epoch_off;  // resident mode: record-mailbox epoch of command seq = res_epoch_off + seq
    alignas(16) unsigned char kargs[sizeof(KArgs<double>)];
    alignas(16) unsigned char mparams[MPPI_MODEL_BLOCK_BYTES];
};

// What one (model, dtype) pair contributes: its kernels (as launchable handles) and how to pack its parameter block.
// The six registry units (mppi_model_tu.cu) each export one statically; a user model compiled at run time with NVRTC
// (mppi_user_model_register) gets one on the heap.  Everything that selects and launches kernels (mppi_fused_host.cuh)
// works on this descriptor, so it is compiled once, not per model.
struct ModelKernels {
    int nx, nu;
    int is_double;
    int is_mlp;                      // PendulumMLP: no split-cost / resident variants; tensor-core kernels in `tc`
    int np;                          // run-time user models: reals in the parameter block (P = { real v[np]; })
    int param_bytes;                 // sizeof(Model::P<real>)
    void (*load)(const ModelKernels* self, void* dst, const double* blob, const double* ext, int n_ext);
    const void* fused[3];            // fused_command_kernel<Model, real, V, false, false>, V = MPPI / SMPPI / KMPPI
    const void* split[3];            // ... SPLIT = true (nullptr: not available)
    const void* batched;             // fused_command_kernel<Model, real, V_MPPI, true>
    const void* resident[3];         // resident_command_kernel<Model, real, V> (nullptr: not available)
    const void* resident_stamped;    // the one instantiation with %globaltimer stamps, or nullptr
    const void* states;              // states_kernel<Model, real>
    const void* tc[3][2][2];         // mlp_tc_command_kernel<V, SPLIT = 2 - mode, FAST>, [V][mode - 1][fast]; fp32 MLP only
    void* library;                   // run-time user models: the cudaLibrary_t that owns the kernels
};
}  // namespace mppi_host

using namespace mppi_host;

namespace {

inline int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return MPPI_ERR_CUDA;
}
inline int unsupported_at(const char* why, const char* file, int line) {
    const char* base = strrchr(file, '/');
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s (%s:%d)", why, base ? base + 1 : file, line);
    return MPPI_ERR_UNSUPPORTED;
}
#define UNSUPPORTED(why) unsupported_at(why, __FILE__, __LINE__)
#define CK(call)                                              \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) return cuda_fail(_e, #call);   \
    } while (0)

struct DevInfo {
    int sm_count = 0;
    int max_smem_optin = 0;
};
inline int get_dev_info(DevInfo& d) {
    static thread_local int cached_dev = -1;
    static thread_local DevInfo cached;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (dev != cached_dev) {
        CK(cudaDeviceGetAttribute(&cached.sm_count, cudaDevAttrMultiProcessorCount, dev));
        CK(cudaDeviceGetAttribute(&cached.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        cached_dev = dev;
    }
    d = cached;
    return MPPI_OK;
}

inline int validate(const MppiFusedParams* p, bool fused = false) {
    if (p == nullptr) return MPPI_ERR_BAD_ARG;
    if (p->struct_size != sizeof(MppiFusedParams)) return MPPI_ERR_ABI;
    if (p->K <= 0 || p->T <= 0 || p->nu <= 0 || p->nu > MPPI_MAX_NU || p->nx <= 0) return MPPI_ERR_BAD_ARG;
    if (fused && p->nx > MPPI_MAX_NX) return MPPI_ERR_BAD_ARG;      // state by value; the per-step entry points never touch the state
    if (p->variant < 0 || p->variant > 2) return MPPI_ERR_BAD_ARG;
    if (p->dtype != MPPI_F32 && p->dtype != MPPI_F64) return MPPI_ERR_BAD_ARG;
    if (p->variant == MPPI_VARIANT_KMPPI && (p->S <= 0 || p->W == nullptr || p->theta == nullptr)) return MPPI_ERR_BAD_ARG;
    if (p->variant == MPPI_VARIANT_SMPPI && (p->A == nullptr || p->T < 2)) return MPPI_ERR_BAD_ARG;
    if ((p->flags & MPPI_FLAG_SHIFT) && p->variant == MPPI_VARIANT_KMPPI && p->Wshift == nullptr) return MPPI_ERR_BAD_ARG;
    if (p->lambda_ <= 0.0) return MPPI_ERR_BAD_ARG;
    if (p->world < 0 || p->world > MPPI_MAX_RANKS) return MPPI_ERR_BAD_ARG;
    if (p->u_per_command < 1 || p->u_per_command > p->T) return MPPI_ERR_BAD_ARG;
    return MPPI_OK;
}

inline int rows_of(const MppiFusedParams* p) { return (p->variant == MPPI_VARIANT_KMPPI ? p->S : p->T) * p->nu; }

// a sharded controller whose kernel exchanges the records with its peers over NVLink (not through a library collective)
inline bool sharded_in_kernel(const MppiFusedParams* p) {
    bool any_peer = false;
    for (int g = 0; g < MPPI_MAX_RANKS; ++g) any_peer = any_peer || p->peer_slots[g] != nullptr;
    return p->world > 1 && any_peer && !(p->flags & MPPI_FLAG_EXPORT_PARTIAL);
}

// make_layout's `extra` word of a kernel that finishes in warp_tail without a cluster, in ticket mode (xchg_npub = 1): the
// softmin_update_kernel and the tcgen05 kernel
inline int ticket_layout_extra(const MppiFusedParams* p) {
    return layout_extra(0, 0, 1, fused_xstage_doubles(sharded_in_kernel(p), p->world, 1, rows_of(p)));
}

template <typename real> void fill_noise_model(const MppiFusedParams* p, NoiseModel<real>& nm) {
    for (int i = 0; i < MPPI_MAX_NU; ++i) {
        nm.mu[i] = (real)p->noise_mu[i];
        nm.u_min[i] = (real)p->u_min[i];
        nm.u_max[i] = (real)p->u_max[i];
        nm.a_min[i] = (real)p->action_min[i];
        nm.a_max[i] = (real)p->action_max[i];
    }
    for (int i = 0; i < MPPI_MAX_NU * MPPI_MAX_NU; ++i) {
        nm.L[i] = (real)p->chol[i];
        nm.Sinv[i] = (real)p->sigma_inv[i];
    }
    nm.lambda_ = (real)p->lambda_;
    nm.neg_inv_lambda = (real)(-(1.0 / p->lambda_));   // mppi.py:256: -factor * (cost - beta), factor = 1/lambda
    nm.u_scale = (real)p->u_scale;
    nm.w_smooth = (real)p->w_action_seq_cost;
    nm.delta_t = (real)p->delta_t;
    nm.diag = (p->flags & MPPI_FLAG_DIAG_SIGMA) ? 1 : 0;
    nm.abs_cost = (p->flags & MPPI_FLAG_ABS_COST) ? 1 : 0;
}

// ticket + the records of (R + 2) doubles the warp-fold tail combines in ticket mode (one per cluster of the grid)
// ... followed by this GPU's own record mailbox (single-GPU LL mode): two epoch parities of MPPI_LL_LOCAL_WORDS flagged words
#define MPPI_LL_STAGE_BYTES 49152                          // finisher staging budget: LL mode needs xw x clusters x (R+2) x 8 <= this
#define MPPI_LL_LOCAL_WORDS (2 * MPPI_LL_STAGE_BYTES / 8)  // words per parity of the local mailbox (2 words per double)
inline uint64_t ws_partials_bytes(int nb, int R) { return (16 + (uint64_t)nb * (uint64_t)(R + 2) * 8 + 255) / 256 * 256; }
inline uint64_t ws_bytes(int nb, int R) { return ws_partials_bytes(nb, R) + 2ull * MPPI_LL_LOCAL_WORDS * 8; }

inline unsigned long long xchg_timeout_ns() {
    // how long a shard waits for its peers' records before giving up (rank skew: a GC pause, a JIT build, a lazy module
    // load on another rank); MPPI_B200_XCHG_TIMEOUT_S overrides the 20 s default
    const char* e = getenv("MPPI_B200_XCHG_TIMEOUT_S");
    double sec = (e != nullptr && atof(e) > 0) ? atof(e) : 20.0;
    return (unsigned long long)(sec * 1e9);
}

template <typename real> int fill_kargs(const MppiFusedParams* p, KArgs<real>& a, int BS, int nb, int tps = 1) {
    memset(&a, 0, sizeof(a));
    fill_noise_model<real>(p, a.nm);
    for (int i = 0; i < MPPI_MAX_NU; ++i) a.u_init[i] = (real)p->u_init[i];
    for (int i = 0; i < MPPI_MAX_NX; ++i) a.x0[i] = (real)p->state[i];
    a.state_dev = (p->flags & MPPI_FLAG_STATE_DEVICE) ? (const real*)p->state_dev : nullptr;
    a.state_per_sample = (p->flags & MPPI_FLAG_STATE_PER_SAMPLE) ? 1 : 0;
    a.U = (real*)p->U;
    a.A = (real*)p->A;
    a.theta = (real*)p->theta;
    a.W = (const real*)p->W;
    a.Wshift = (const real*)p->Wshift;
    a.cost_total = (real*)p->cost_total;
    a.action_out = (real*)p->action_out;
    a.nominal_used = (real*)p->nominal_used;
    a.stats = (double*)p->stats;
    a.z = (const real*)p->z;
    a.z_out = (real*)p->z_out;
    a.K = p->K;
    a.T = p->T;
    a.S = p->S;
    a.R = rows_of(p);
    a.TN = p->T * p->nu;
    a.upc = p->u_per_command;
    a.n_tiles = (p->K + BS - 1) / BS;
    a.tps = tps;
    a.k_offset = p->k_offset;
    a.seed = p->seed;
    a.offset = p->offset;
    a.shift = (p->flags & MPPI_FLAG_SHIFT) ? 1 : 0;
    a.null_action = (p->flags & MPPI_FLAG_NULL_ACTION) ? 1 : 0;
    a.pdl = (p->flags & MPPI_FLAG_PDL) ? 1 : 0;
    const int es = (int)sizeof(real);
    const bool padded = (p->flags & MPPI_FLAG_NOMINAL_PADDED) || ((a.TN * es) % 16 == 0);
    a.tma_ok = padded && ((uintptr_t)p->U % 16 == 0) && (p->variant != MPPI_VARIANT_SMPPI || (uintptr_t)p->A % 16 == 0);
    // workspace carve
    if (p->workspace != nullptr) {
        unsigned char* w = (unsigned char*)p->workspace;
        a.ticket = (unsigned int*)w;
        a.crec = (double*)(w + 16);
    }
    a.xchg_npub = 1;
    a.xchg_parity_words = MPPI_XCHG_PARITY_WORDS;
    a.xchg_timeout_ns = xchg_timeout_ns();
    a.xchg_status_host = (long long*)p->xchg_status_host;
    a.rank = p->rank;
    a.world = p->world <= 0 ? 1 : p->world;
    a.epoch = p->epoch;
    a.export_partial = (p->flags & MPPI_FLAG_EXPORT_PARTIAL) ? 1 : 0;
    a.partial_out = (double*)p->partial_out;
    a.torch_total = p->torch_rng_total;
    a.offset_dev = (unsigned long long*)p->offset_dev;
    a.offset_inc = p->offset_inc;
    a.n_env = p->n_env > 1 ? p->n_env : 1;
    a.env_u_stride = p->env_u_stride;
    a.env_ws_stride = (long long)p->env_ws_stride;
    a.dbg = (unsigned long long*)p->debug_clocks;
    a.host_mailbox = (unsigned long long*)p->host_mailbox;
    a.host_epoch = p->host_epoch;
    bool any_peer = false;
    for (int g = 0; g < MPPI_MAX_RANKS; ++g) {
        a.peers[g] = (unsigned long long*)p->peer_slots[g];
        any_peer = any_peer || p->peer_slots[g] != nullptr;
    }
    if (!any_peer || a.export_partial) a.world = a.export_partial ? a.world : 1;
    if (p->workspace != nullptr && (a.world == 1 || a.export_partial)) {
        // not sharded in-kernel: the record mailbox is this GPU's own, behind the partials in the workspace
        a.peers[0] = (unsigned long long*)((unsigned char*)p->workspace + ws_partials_bytes(nb, a.R));
        a.xchg_parity_words = MPPI_LL_LOCAL_WORDS;
    }
    return MPPI_OK;
}

// launch configuration with the optional attributes: programmatic dependent launch, thread-block clusters (cluster, 1, 1)
inline void launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* at, int nb, int BD, int smem, cudaStream_t stream, bool pdl,
                          int ny, int cluster) {
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(nb, ny);
    cfg.blockDim = dim3(BD);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    int n = 0;
    if (pdl) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = (unsigned)cluster;
        at[n].val.clusterDim.y = 1;
        at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at;
    cfg.numAttrs = n;
}

inline cudaError_t launch_raw(const void* kernel, int nb, int BD, int smem, cudaStream_t stream, void** argv, bool pdl, int ny = 1,
                              int cluster = 1) {
    if (!pdl && cluster <= 1) return cudaLaunchKernel(kernel, dim3(nb, ny), dim3(BD), argv, (size_t)smem, stream);
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[3];
    launch_config(cfg, at, nb, BD, smem, stream, pdl, ny, cluster);
    return cudaLaunchKernelExC(&cfg, kernel, argv);
}

template <typename... Args>
int launch_kernel(void (*kernel)(Args...), int nb, int BD, int smem, cudaStream_t stream, int ny, Args... args) {
    void* argv[] = {(void*)&args...};
    cudaError_t e = cudaLaunchKernel((const void*)kernel, dim3(nb, ny), dim3(BD), argv, (size_t)smem, stream);
    if (e != cudaSuccess) {
        snprintf(g_cuda_err, sizeof(g_cuda_err), "launch grid=%d block=%d smem=%d: %s (%s)", nb, BD, smem,
                 cudaGetErrorName(e), cudaGetErrorString(e));
        return MPPI_ERR_CUDA;
    }
    return MPPI_OK;
}

// LL mode identifies a command's records by its epoch tag: a launch captured into a CUDA graph would replay one tag.
inline int refuse_capture(cudaStream_t stream, const Geometry& g) {
    if (g.npub <= 1) return MPPI_OK;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone)
        return UNSUPPORTED("the fused command cannot be captured into a CUDA graph (its reduction records carry a per-command tag); "
                           "launch it directly — it is one kernel — or set MPPI_B200_XCHG_DIRECT=0");
    return MPPI_OK;
}

struct GeomKey {
    const void* kernel;
    int dev, variant, K, T, nu, S, bt, tp, gb, r2, single, ne;
    bool operator==(const GeomKey& o) const {
        return kernel == o.kernel && dev == o.dev && variant == o.variant && K == o.K && T == o.T && nu == o.nu && S == o.S &&
               bt == o.bt && tp == o.tp && gb == o.gb && r2 == o.r2 && single == o.single && ne == o.ne;
    }
};

// Launch geometry for (kernel, dimensions).  The occupancy / attribute queries cost microseconds, so
// the last few results are cached per thread: a steady-state command() pays only the lookup.
static thread_local int g_tc_kernel = 0;   // set around plan_geometry() for the tcgen05 kernels (see below)
static thread_local int g_tc_cols = 64;    // TMEM columns one CTA of that kernel allocates
template <typename KernelT>
int plan_geometry(KernelT kernel, const MppiFusedParams* p, int es, int need_rows2, bool single_partial_grid, Geometry& g,
                  SmemLayout (*layout)(int, int, int, int, int, int, int, int, int)) {
    static thread_local GeomKey keys[8];
    static thread_local Geometry vals[8];
    static thread_local int n_cached = 0, next_slot = 0;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    const GeomKey key{(const void*)kernel, dev, p->variant, p->K, p->T, p->nu, p->S, p->block_threads, p->threads_per_sample,
                      p->grid_blocks, need_rows2, single_partial_grid ? 1 : 0, p->n_env > 1 ? p->n_env : 1};
    for (int i = 0; i < n_cached; ++i)
        if (keys[i] == key) {
            g = vals[i];
            return MPPI_OK;
        }
    DevInfo di;
    int rc = get_dev_info(di);
    if (rc) return rc;
    const int R = rows_of(p);
    // BS samples per tile; tps threads share one sample's sampling/transform work.
    //
    // Automatic geometry (block_threads == 0): blocks are statically assigned tiles (determinism:
    // the reduction order must not depend on scheduling), so the finish time follows the most
    // loaded SM.  Enumerate BS in steps of a warp and j = resident CTAs per SM, size the grid as
    // min(n_tiles, SMs*j), and keep the candidate with the smallest worst-case samples per SM
    // (ties: fewer passes, then more threads).  Measured on B200 (scripts/geom_sweep.py) this picks
    // the winners of an exhaustive sweep within ~3 %: e.g. K=131072 -> BS=448, 293 CTAs, one pass.
    int BS = p->block_threads;
    int tps = p->threads_per_sample;
    int grid_hint = 0;
    if (BS <= 0) {
        cudaFuncAttributes fa0;
        CK(cudaFuncGetAttributes(&fa0, kernel));
        const int dyn0 = di.max_smem_optin - (int)fa0.sharedSizeBytes;
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn0));
        long long best_load = -1;
        int best_bs = 128, best_passes = 0, best_grid = 0;
        // latency hiding needs ~24 resident warps per SM when the problem is large enough to supply them
        const long long per_sm = ((long long)p->K + di.sm_count - 1) / di.sm_count;
        const long long want_threads = per_sm < 768 ? per_sm : 768;
        for (int bs = 64; bs <= 512; bs += (bs < 128 ? 64 : 32)) {     // 64-sample tiles let K < 128 x SMs reach every SM
            SmemLayout Lc = layout(p->variant, p->T, p->nu, p->S, R, bs, bs, single_partial_grid ? 1 : di.sm_count * 4, need_rows2);
            if (Lc.total > dyn0) continue;
            int occ_c = 0;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_c, kernel, bs, Lc.total));
            if (occ_c < 1) continue;
            const int nt = (p->K + bs - 1) / bs;
            for (int j = 1; j <= occ_c && j <= 8; ++j) {
                const int nbc = nt < di.sm_count * j ? nt : di.sm_count * j;
                const int passes = (nt + nbc - 1) / nbc;
                const int bps = (nbc + di.sm_count - 1) / di.sm_count;
                long long load = (long long)bps * passes * bs;
                const long long resident = (long long)bps * bs;
                if (resident < want_threads) load = load * want_threads / resident;   // under-occupied: proportionally slower
                const bool better = best_load < 0 || load < best_load ||
                                    (load == best_load && (passes < best_passes || (passes == best_passes && bs > best_bs)));
                if (better) {
                    best_load = load;
                    best_bs = bs;
                    best_passes = passes;
                    best_grid = nbc;
                }
            }
        }
        BS = best_bs;
        grid_hint = best_grid;
    }
    if (BS % 32 != 0 || BS < 32 || BS > 512) return MPPI_ERR_BAD_ARG;
    const int n_tiles = (p->K + BS - 1) / BS;
    if (tps <= 0) {
        // helper threads only pay off while an SM hosts a single small CTA
        tps = 1;
        const int envs = p->n_env > 1 ? p->n_env : 1;
        if ((long long)n_tiles * envs <= di.sm_count) tps = 512 / BS >= 8 ? 8 : (512 / BS >= 4 ? 4 : (512 / BS >= 2 ? 2 : 1));
    }
    while (tps > 1 && BS * tps > 512) tps >>= 1;
    if (tps != 1 && tps != 2 && tps != 4 && tps != 8) return MPPI_ERR_BAD_ARG;
    const int BD = BS * tps;
    const int cap = di.sm_count * 16;
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, kernel));
    const int dyn_limit = di.max_smem_optin - (int)fa.sharedSizeBytes;   // static + dynamic <= opt-in maximum
    // The attribute is a per-kernel LIMIT (setting a smaller value later lowers it), so raise it
    // once to the device maximum; the carve-out actually used follows each launch's request.
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit));
    // The layout depends on the grid (rescale factors of nb partials live in shared memory) and the
    // grid on the occupancy the layout allows: iterate from an optimistic guess to a fixed point.
    int nb = n_tiles < cap ? n_tiles : cap;
    int occ = 0;
    SmemLayout L;
    for (int it = 0; it < 4; ++it) {
        L = layout(p->variant, p->T, p->nu, p->S, R, BD, BS, single_partial_grid ? 1 : nb, need_rows2);
        if (L.total > dyn_limit) return UNSUPPORTED("shared-memory tile does not fit");
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, BD, L.total));
        if (occ < 1) return UNSUPPORTED("kernel does not fit on an SM with this block size");
        if (g_tc_kernel) {
            // The occupancy API answers 1 CTA/SM for kernels that allocate tensor memory; measured on B200 the
            // 128-thread tcgen05 CTAs do co-reside (K=131072, T=30: 585 us at 1 CTA/SM, 379 at 2, 311 at 3), so
            // size the grid from the real limits: shared memory, registers, and the CTA's share of the 512 TMEM columns.
            int smem_sm = 0;
            CK(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
            const int by_smem = smem_sm / ((int)fa.sharedSizeBytes + L.total + 1024);
            const int by_regs = 65536 / (((fa.numRegs + 7) / 8 * 8) * BD);
            int o = by_smem < by_regs ? by_smem : by_regs;
            if (o > 512 / g_tc_cols) o = 512 / g_tc_cols;
            const char* e = getenv("MPPI_TC_OCC");
            if (e != nullptr && atoi(e) > 0) o = atoi(e);
            if (o > occ) occ = o;
        }
        int nb2 = n_tiles < di.sm_count * occ ? n_tiles : di.sm_count * occ;
        if (nb2 > cap) nb2 = cap;
        if (p->grid_blocks > 0 && p->grid_blocks < nb2) nb2 = p->grid_blocks;
        if (grid_hint > 0 && grid_hint < nb2) nb2 = grid_hint;
        if (nb2 == nb) break;
        nb = nb2;
    }
    L = layout(p->variant, p->T, p->nu, p->S, R, BD, BS, single_partial_grid ? 1 : nb, need_rows2);
    g.BS = BS;
    g.tps = tps;
    g.BD = BD;
    g.nb = nb;
    g.smem = L.total;
    g.occ = occ;
    g.regs = fa.numRegs;
    g.cluster = 1;
    g.npub = 0;
    (void)es;
    keys[next_slot] = key;
    vals[next_slot] = g;
    next_slot = (next_slot + 1) % 8;
    if (n_cached < 8) ++n_cached;
    return MPPI_OK;
}

template <typename real> SmemLayout layout_fn(int v, int T, int nu, int S, int R, int BD, int BS, int nb, int r2) {
    return make_layout<real>(v, T, nu, S, R, BD, BS, nb, r2);
}


}  // namespace

