// mppi_b200.cu — C-ABI entry points (include/mppi_b200.h) and kernel dispatch.
// Built with: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC
// No torch types cross this boundary; the Python side binds it with ctypes.
//
// Translation units of the library (built in parallel by pytorch_mppi_b200/build.py):
//   mppi_b200.cu        this file: the C ABI, the model-independent kernels (sampling, softmin update, cost
//                       accumulation, omega, apply-partials), plan commands, resident-mode backend, peer mailboxes
//   mppi_model_tu.cu    compiled once per (registered model, dtype): fused / resident / states kernels of that model
#include "mppi_fused_host.cuh"

namespace mppi_host {
thread_local char g_cuda_err[512] = "";

// one getter per (model, dtype) translation unit, all weak: the stock library links the six registry units, an
// nvcc-built user-model variant library links this unit and the two units of that model only
#define MPPI_KERNELS_DECL(name) const ModelKernels* name() __attribute__((weak))
MPPI_KERNELS_DECL(model_kernels_pendulum_f32);
MPPI_KERNELS_DECL(model_kernels_pendulum_f64);
MPPI_KERNELS_DECL(model_kernels_linear_point_f32);
MPPI_KERNELS_DECL(model_kernels_linear_point_f64);
MPPI_KERNELS_DECL(model_kernels_pendulum_mlp_f32);
MPPI_KERNELS_DECL(model_kernels_pendulum_mlp_f64);
MPPI_KERNELS_DECL(model_kernels_user_f32);
MPPI_KERNELS_DECL(model_kernels_user_f64);
}  // namespace mppi_host

namespace {

// a user model compiled at run time (mppi_user_model_register): its descriptor travels in MppiFusedParams.user_model
struct UserModelHandle {
    uint32_t magic;
    ModelKernels mk;
};
constexpr uint32_t kUserMagic = 0x4d505049u;   // "MPPI"

// the (model, dtype) descriptor that serves these parameters, or nullptr
const ModelKernels* find_kernels(const MppiFusedParams* p, int* rc) {
    *rc = MPPI_ERR_UNSUPPORTED;
    const bool f32 = p->dtype == MPPI_F32;
    typedef const ModelKernels* (*Getter)();
    Getter get = nullptr;
    switch (p->model) {
        case MPPI_MODEL_PENDULUM: get = f32 ? model_kernels_pendulum_f32 : model_kernels_pendulum_f64; break;
        case MPPI_MODEL_LINEAR_POINT: get = f32 ? model_kernels_linear_point_f32 : model_kernels_linear_point_f64; break;
        case MPPI_MODEL_PENDULUM_MLP:
            if (p->n_model_params_ext < PendulumMLPModel::N_EXT || p->model_params_ext == nullptr) {
                *rc = MPPI_ERR_BAD_ARG;
                return nullptr;
            }
            get = f32 ? model_kernels_pendulum_mlp_f32 : model_kernels_pendulum_mlp_f64;
            break;
        case MPPI_MODEL_USER:
            if (p->user_model != nullptr) {
                const UserModelHandle* h = reinterpret_cast<const UserModelHandle*>(p->user_model);
                if (h->magic != kUserMagic || h->mk.is_double != (f32 ? 0 : 1)) {
                    *rc = MPPI_ERR_BAD_ARG;
                    return nullptr;
                }
                return &h->mk;
            }
            get = f32 ? model_kernels_user_f32 : model_kernels_user_f64;
            break;
    }
    return get != nullptr ? get() : nullptr;      // nullptr: this library was linked without that unit
}

template <typename real>
inline void plan_update(Plan* pl, const double* state, const void* state_dev, uint32_t flags, uint64_t seed, uint64_t offset,
                        const void* z, void* action_out, void* host_mailbox) {
    KArgs<real>* a = reinterpret_cast<KArgs<real>*>(pl->kargs);
    if (state != nullptr)
        for (int i = 0; i < pl->nx; ++i) a->x0[i] = (real)state[i];
    a->state_dev = (flags & MPPI_FLAG_STATE_DEVICE) ? (const real*)state_dev : nullptr;
    a->state_per_sample = (flags & MPPI_FLAG_STATE_PER_SAMPLE) ? 1 : 0;
    a->shift = (flags & MPPI_FLAG_SHIFT) ? 1 : 0;
    a->seed = seed;
    a->offset = offset;
    a->z = (const real*)z;
    a->action_out = (real*)action_out;
    // one epoch per command on whichever route it takes: the tag of its reduction records (and, sharded, of the exchange)
    if (pl->res.armed && pl->res_epoch_off + pl->res.seq > pl->epoch) pl->epoch = pl->res_epoch_off + pl->res.seq;
    a->epoch = ++pl->epoch;
    a->host_mailbox = (unsigned long long*)host_mailbox;
    if (host_mailbox != nullptr) a->host_epoch = ++pl->host_epoch;
}

inline int plan_launch(Plan* pl, cudaStream_t stream) {
    int rc = refuse_capture(stream, pl->g);
    if (rc) return rc;
    void* argv[2] = {(void*)pl->kargs, (void*)pl->mparams};
    cudaError_t e = launch_raw(pl->kernel, pl->g.nb, pl->g.BD, pl->g.smem, stream, argv, pl->pdl != 0, pl->p.n_env > 1 ? pl->p.n_env : 1,
                               pl->g.cluster);
    if (e != cudaSuccess) {
        snprintf(g_cuda_err, sizeof(g_cuda_err), "plan launch grid=%d block=%d smem=%d cluster=%d: %s (%s)", pl->g.nb, pl->g.BD, pl->g.smem, pl->g.cluster,
                 cudaGetErrorName(e), cudaGetErrorString(e));
        return MPPI_ERR_CUDA;
    }
    return MPPI_OK;
}

// ---- resident mode: the device backend of csrc/mppi_resident_host.h ---------------------------------
template <typename real>
int resident_launch_t(Plan* pl, uint64_t seed, uint64_t offset_pred, int shift_pred, uint64_t seq_start, uint32_t gen) {
    ResidentDevice& d = pl->resdev;
    KArgs<real> a = *reinterpret_cast<KArgs<real>*>(pl->kargs);
    a.seed = seed;
    a.z = nullptr;
    a.z_out = nullptr;
    a.state_dev = nullptr;
    a.action_out = (real*)d.action_dev;
    a.host_mailbox = d.host_box + RES_BOX_ACTION;
    a.pdl = 0;
    ResidentArgs ra;
    memset(&ra, 0, sizeof(ra));
    ra.host_cmd = d.host_box + RES_BOX_RECORD;
    ra.host_status = d.host_box + RES_BOX_DONE;
    ra.board = d.board;
    ra.seq_start = seq_start;
    ra.offset_pred = offset_pred;
    ra.idle_ns = d.idle_ns;
    ra.epoch_off = pl->res_epoch_off;
    ra.gen = gen;
    ra.shift_pred = shift_pred;
    ra.n_words = 3 + pl->nx * (pl->is_double ? 2 : 1);
    DevInfo di;
    int rc = get_dev_info(di);
    if (rc) return rc;
    // the launch route's grid (one tile per CTA, padded to the cluster size) and cluster size: same reduction tree, same
    // bits.  If the driver refuses cooperative + cluster together, the grid is launched without clusters (its results
    // then agree with the launch route to fp64 rounding of the reduction order instead of bit for bit).
    const MppiFusedParams& pp = pl->p;
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, pl->res_kernel));
    const int dyn_limit = di.max_smem_optin - (int)fa.sharedSizeBytes;
    CK(cudaFuncSetAttribute(pl->res_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit));
    CK(cudaMemsetAsync(d.board, 0, MPPI_RES_BOARD_WORDS * sizeof(unsigned long long), d.stream));
    void* argv[3] = {(void*)&a, (void*)pl->mparams, (void*)&ra};
    cudaError_t e = cudaErrorInvalidConfiguration;
    for (int cs = pl->g.cluster; cs >= 1; cs = (cs > 1 ? 1 : 0)) {
        const int nb = cs > 1 ? pl->g.nb : a.n_tiles;
        const int smem = make_layout<real>(pp.variant, pp.T, pp.nu, pp.S, a.R, pl->g.BD, pl->g.BS, fused_layout_nb(nb / cs, a.xchg_npub),
                                           layout_extra(pp.variant != MPPI_VARIANT_MPPI, pl->nx, cs, fused_xstage_doubles(false, 1, a.xchg_npub, a.R))).total;
        if (smem > dyn_limit) return UNSUPPORTED("resident kernel: shared-memory tile does not fit");
        // cooperative: every CTA is resident or the launch fails — the CTAs wait for each other through the board
        cudaLaunchConfig_t cfg;
        cudaLaunchAttribute at[3];
        launch_config(cfg, at, nb, pl->g.BD, smem, d.stream, false, 1, cs);
        at[cfg.numAttrs].id = cudaLaunchAttributeCooperative;
        at[cfg.numAttrs].val.cooperative = 1;
        ++cfg.numAttrs;
        e = cudaLaunchKernelExC(&cfg, pl->res_kernel, argv);
        if (e == cudaSuccess) break;
        cudaGetLastError();
    }
    if (e != cudaSuccess) return cuda_fail(e, "resident launch");
    return MPPI_OK;
}
int resident_be_launch(void* ctx, uint64_t seed, uint64_t offset_pred, int shift_pred, uint64_t seq_start, uint32_t gen) {
    Plan* pl = reinterpret_cast<Plan*>(ctx);
    return pl->is_double ? resident_launch_t<double>(pl, seed, offset_pred, shift_pred, seq_start, gen)
                         : resident_launch_t<float>(pl, seed, offset_pred, shift_pred, seq_start, gen);
}
int resident_be_drain(void* ctx) {
    Plan* pl = reinterpret_cast<Plan*>(ctx);
    CK(cudaStreamSynchronize(pl->resdev.stream));
    return MPPI_OK;
}
int resident_be_health(void* ctx) {
    Plan* pl = reinterpret_cast<Plan*>(ctx);
    cudaError_t q = cudaStreamQuery(pl->resdev.stream);
    if (q != cudaSuccess && q != cudaErrorNotReady) return cuda_fail(q, "cudaStreamQuery while waiting for the resident grid");
    return MPPI_OK;
}
static_assert(MPPI_RES_CMD_SHIFT == (unsigned)RES_CMD_SHIFT && MPPI_RES_CMD_STOP == (unsigned)RES_CMD_STOP, "record flags: host and device disagree");
static_assert((int)RES_ERR_BAD_ARG == (int)MPPI_ERR_BAD_ARG && (int)RES_ERR_TIMEOUT == (int)MPPI_ERR_TIMEOUT, "status codes of the protocol header");

int dispatch_fused(const MppiFusedParams* p, cudaStream_t s, MppiLaunchInfo* info) {
    int rc = validate(p, true);
    if (rc) return rc;
    const ModelKernels* mk = find_kernels(p, &rc);
    if (mk == nullptr) return rc;
    return mk->is_double ? run_fused<double>(mk, p, s, info) : run_fused<float>(mk, p, s, info);
}

// ---- generic path: sample / softmin -------------------------------------------------------------
template <typename real, int V, int NU>
int run_sample(const MppiFusedParams* p, KArgs<real>& a_extra, cudaStream_t stream) {
    auto kernel = sample_kernel<real, V, NU>;
    Geometry g;
    int rc = plan_geometry(kernel, p, (int)sizeof(real), V == V_KMPPI, true, g, layout_fn<real>);
    if (rc) return rc;
    KArgs<real> a;
    fill_kargs<real>(p, a, g.BS, g.nb, g.tps);
    a.out_pa = a_extra.out_pa;
    a.out_noise = a_extra.out_noise;
    a.out_noise_theta = a_extra.out_noise_theta;
    a.out_cost_init = a_extra.out_cost_init;
    a.override_rows = a_extra.override_rows;
    a.n_override = a_extra.n_override;
    a.override_start = a_extra.override_start;
    if (a_extra.shift < 0) {   // materialise from nominal_used: no shift, plain loads
        a.U = (real*)p->nominal_used;
        a.A = a.U + a.TN;
        a.theta = a.U + 2 * a.TN;
        a.shift = 0;
        a.tma_ok = 0;
        a.nominal_used = nullptr;
    }
    return launch_kernel(kernel, g.nb, g.BD, g.smem, stream, a.n_env, a);
}

template <typename real, int V> int run_sample_nu(const MppiFusedParams* p, KArgs<real>& e, cudaStream_t s) {
    switch (p->nu) {
        case 1: return run_sample<real, V, 1>(p, e, s);
        case 2: return run_sample<real, V, 2>(p, e, s);
        case 3: return run_sample<real, V, 3>(p, e, s);
        case 4: return run_sample<real, V, 4>(p, e, s);
    }
    return MPPI_ERR_UNSUPPORTED;
}

template <typename real>
int run_sample_any(const MppiFusedParams* p, void* pa, void* noise, void* noise_theta, void* cost_init, const void* ovr,
                   int n_ovr, int ovr_start, bool from_nominal_used, cudaStream_t s) {
    KArgs<real> e;
    memset(&e, 0, sizeof(e));
    e.out_pa = (real*)pa;
    e.out_noise = (real*)noise;
    e.out_noise_theta = (real*)noise_theta;
    e.out_cost_init = (real*)cost_init;
    e.override_rows = (const real*)ovr;
    e.n_override = n_ovr;
    e.override_start = ovr_start;
    e.shift = from_nominal_used ? -1 : 0;
    switch (p->variant) {
        case MPPI_VARIANT_MPPI: return run_sample_nu<real, V_MPPI>(p, e, s);
        case MPPI_VARIANT_SMPPI: return run_sample_nu<real, V_SMPPI>(p, e, s);
        case MPPI_VARIANT_KMPPI: return run_sample_nu<real, V_KMPPI>(p, e, s);
    }
    return MPPI_ERR_BAD_ARG;
}

template <typename real, int V, int NU>
int run_softmin(const MppiFusedParams* p, const void* cost, const void* eps, cudaStream_t stream) {
    auto kernel = softmin_update_kernel<real, V, NU>;
    Geometry g;
    int rc = plan_geometry(kernel, p, (int)sizeof(real), ticket_layout_extra(p), false, g, layout_fn<real>);
    if (rc) return rc;
    const uint64_t need_ws = ws_bytes(g.nb, rows_of(p));
    if (p->workspace == nullptr || p->workspace_bytes < need_ws) return MPPI_ERR_WORKSPACE;
    if (p->n_env > 1 && (p->env_ws_stride < need_ws || p->workspace_bytes < p->env_ws_stride * (uint64_t)p->n_env)) return MPPI_ERR_WORKSPACE;
    KArgs<real> a;
    fill_kargs<real>(p, a, g.BS, g.nb, g.tps);
    a.in_cost = (const real*)cost;
    a.in_eps = (const real*)eps;
    if (a.world > 1 && rows_of(p) > MPPI_XCHG_MAX_R) return UNSUPPORTED("T*nu exceeds the peer mailbox record size");
    return launch_kernel(kernel, g.nb, g.BD, g.smem, stream, a.n_env, a);
}

template <typename real, int V> int run_softmin_nu(const MppiFusedParams* p, const void* c, const void* e, cudaStream_t s) {
    switch (p->nu) {
        case 1: return run_softmin<real, V, 1>(p, c, e, s);
        case 2: return run_softmin<real, V, 2>(p, c, e, s);
        case 3: return run_softmin<real, V, 3>(p, c, e, s);
        case 4: return run_softmin<real, V, 4>(p, c, e, s);
    }
    return MPPI_ERR_UNSUPPORTED;
}
template <typename real> int run_softmin_any(const MppiFusedParams* p, const void* c, const void* e, cudaStream_t s) {
    switch (p->variant) {
        case MPPI_VARIANT_MPPI: return run_softmin_nu<real, V_MPPI>(p, c, e, s);
        case MPPI_VARIANT_SMPPI: return run_softmin_nu<real, V_SMPPI>(p, c, e, s);
        case MPPI_VARIANT_KMPPI: return run_softmin_nu<real, V_KMPPI>(p, c, e, s);
    }
    return MPPI_ERR_BAD_ARG;
}

template <typename real, int V>
int run_apply(const MppiFusedParams* p, const void* partials, cudaStream_t stream) {
    KArgs<real> a;
    fill_kargs<real>(p, a, 128, 1);
    a.world = p->world <= 0 ? 1 : p->world;
    const int smem = align_up((2 * a.TN + a.R + a.T * a.S) * (int)sizeof(real), 16) + (a.R + 2) * 8 + 16;
    apply_partials_kernel<real, V><<<1, 128, smem, stream>>>(a, (const double*)partials, p->nu);
    CK(cudaGetLastError());
    return MPPI_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int mppi_b200_abi_version(void) { return MPPI_B200_ABI_VERSION; }

uint64_t mppi_abi_layout(int which) {
    switch (which) {
        case 0: return sizeof(MppiFusedParams);
        case 1: return offsetof(MppiFusedParams, seed);
        case 2: return offsetof(MppiFusedParams, state);
        case 3: return offsetof(MppiFusedParams, U);
        case 4: return offsetof(MppiFusedParams, rank);
        case 5: return offsetof(MppiFusedParams, partial_out);
        case 6: return sizeof(MppiLaunchInfo);
    }
    return 0;
}

const char* mppi_status_string(int s) {
    switch (s) {
        case MPPI_OK: return "ok";
        case MPPI_ERR_BAD_ARG: return "bad argument";
        case MPPI_ERR_UNSUPPORTED: return "unsupported (model, variant, dtype, size) combination";
        case MPPI_ERR_WORKSPACE: return "workspace too small";
        case MPPI_ERR_CUDA: return "CUDA error";
        case MPPI_ERR_ABI: return "MppiFusedParams size mismatch (ABI)";
        case MPPI_ERR_TIMEOUT: return "peer exchange timed out";
    }
    return "unknown status";
}

const char* mppi_last_cuda_error(void) { return g_cuda_err; }

int mppi_fused_query(const MppiFusedParams* p, MppiLaunchInfo* out) {
    if (out == nullptr) return MPPI_ERR_BAD_ARG;
    memset(out, 0, sizeof(*out));
    return dispatch_fused(p, nullptr, out);
}

int mppi_fused_command(const MppiFusedParams* p, void* stream) { return dispatch_fused(p, (cudaStream_t)stream, nullptr); }

int mppi_plan_create(const MppiFusedParams* p, void** plan_out) {
    if (plan_out == nullptr) return MPPI_ERR_BAD_ARG;
    int rc = validate(p, true);
    if (rc) return rc;
    Plan* pl = new (std::nothrow) Plan();
    if (pl == nullptr) return MPPI_ERR_BAD_ARG;
    const ModelKernels* mk = find_kernels(p, &rc);
    if (mk != nullptr) rc = mk->is_double ? build_plan<double>(mk, p, pl) : build_plan<float>(mk, p, pl);
    if (rc) {
        delete pl;
        return rc;
    }
    *plan_out = pl;
    return MPPI_OK;
}

int mppi_plan_destroy(void* plan) {
    if (plan == nullptr) return MPPI_ERR_BAD_ARG;
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl->res.armed) mppi_resident_stop(plan);      // the resident grid reads this controller's buffers
    delete pl;
    return MPPI_OK;
}

int mppi_plan_command(void* plan, const double* state, const void* state_dev, uint32_t flags, uint64_t seed, uint64_t offset,
                      const void* z, void* action_out, void* stream) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl == nullptr || action_out == nullptr) return MPPI_ERR_BAD_ARG;
    if (state == nullptr && !(flags & MPPI_FLAG_STATE_DEVICE)) return MPPI_ERR_BAD_ARG;
    if (pl->is_double) plan_update<double>(pl, state, state_dev, flags, seed, offset, z, action_out, nullptr);
    else plan_update<float>(pl, state, state_dev, flags, seed, offset, z, action_out, nullptr);
    return plan_launch(pl, (cudaStream_t)stream);
}

int mppi_plan_command_host(void* plan, const double* state, uint32_t flags, uint64_t seed, uint64_t offset, const void* z,
                           void* action_out_dev, void* host_mailbox, void* action_host_out, void* stream) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl == nullptr || state == nullptr || host_mailbox == nullptr || action_host_out == nullptr || action_out_dev == nullptr)
        return MPPI_ERR_BAD_ARG;
    if (pl->is_double) plan_update<double>(pl, state, nullptr, flags, seed, offset, z, action_out_dev, host_mailbox);
    else plan_update<float>(pl, state, nullptr, flags, seed, offset, z, action_out_dev, host_mailbox);
    int rc = plan_launch(pl, (cudaStream_t)stream);
    if (rc) return rc;
    // every action value arrives as self-validating 8-byte word(s): payload32 | (epoch & 0xffffffff) << 32
    volatile unsigned long long* box = reinterpret_cast<volatile unsigned long long*>(host_mailbox);
    const unsigned long long want = pl->host_epoch & 0xffffffffull;
    const int nwords = pl->upc_nu * (pl->is_double ? 2 : 1);
    unsigned long long spins = 0;
    for (int w = 0; w < nwords; ++w) {
        while ((box[w] >> 32) != want) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
            if ((++spins & 0xFFFFF) == 0) {       // every ~1M spins: has the stream died or finished without publishing?
                cudaError_t q = cudaStreamQuery((cudaStream_t)stream);
                if (q != cudaSuccess && q != cudaErrorNotReady) return cuda_fail(q, "cudaStreamQuery while waiting for the mailbox");
                if (q == cudaSuccess && (box[w] >> 32) != want) return MPPI_ERR_TIMEOUT;
            }
        }
    }
    // the action is returned in the controller's own dtype (f32 words or f64 double-words)
    if (pl->is_double) {
        unsigned long long* out = reinterpret_cast<unsigned long long*>(action_host_out);
        for (int i = 0; i < pl->upc_nu; ++i) out[i] = (box[2 * i] & 0xffffffffull) | (box[2 * i + 1] << 32);
    } else {
        uint32_t* out = reinterpret_cast<uint32_t*>(action_host_out);
        for (int i = 0; i < pl->upc_nu; ++i) out[i] = (uint32_t)box[i];
    }
    return MPPI_OK;
}

int mppi_resident_start(void* plan, void* host_box, void* board_dev, void* action_out_dev, uint64_t idle_us, void* stream) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl == nullptr || host_box == nullptr || board_dev == nullptr || action_out_dev == nullptr || idle_us == 0)
        return MPPI_ERR_BAD_ARG;
    if (pl->res_kernel == nullptr)
        return UNSUPPORTED("resident mode needs a plan on the split-cost rollout (one tile per SM, registered analytic model, in-kernel exchange if sharded)");
    if (pl->p.z_out != nullptr) return UNSUPPORTED("resident mode does not record the noise it draws (z_out)");
    if (pl->res.launched) {                 // re-arming: the old grid leaves first (it polls the box that is about to be cleared)
        int rc = res_halt(pl->res);
        if (rc) return rc;
    }
    ResidentDevice& d = pl->resdev;
    d.host_box = reinterpret_cast<unsigned long long*>(host_box);
    d.board = reinterpret_cast<unsigned long long*>(board_dev);
    d.action_dev = action_out_dev;
    d.idle_ns = idle_us * 1000ull;
    d.stream = (cudaStream_t)stream;
    const ResidentBackend be{pl, resident_be_launch, resident_be_drain, resident_be_health};
    const int rc_arm = res_arm(pl->res, host_box, pl->nx, pl->upc_nu, pl->is_double, be, 0);
    // resident commands continue the plan's epochs: command seq carries epoch res_epoch_off + seq
    pl->res_epoch_off = pl->epoch - pl->res.seq;
    return rc_arm;
}

int mppi_resident_command(void* plan, const double* state, uint32_t flags, uint64_t seed, uint64_t offset, void* action_host_out) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl == nullptr) return MPPI_ERR_BAD_ARG;
    return res_command(pl->res, state, (flags & MPPI_FLAG_SHIFT) ? 1 : 0, seed, offset, action_host_out, 0);
}

int mppi_resident_sync(void* plan) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    return pl == nullptr ? (int)MPPI_ERR_BAD_ARG : res_sync(pl->res);
}

int mppi_resident_stop(void* plan) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    return pl == nullptr ? (int)MPPI_ERR_BAD_ARG : res_stop(pl->res);
}

// ---- user models compiled at run time ----------------------------------------------------------------------------------
// The Python side compiles `mppi_fused.cuh + mppi_resident.cuh + the user's model header` with NVRTC (in process, no
// toolkit) into a cubin and hands it over with the lowered names of the kernels; they are loaded as a cudaLibrary_t and
// wrapped in a ModelKernels table exactly like a registry unit's.  `names`: 6 entries, nullptr = not built:
//   [0] fused (this variant)  [1] split-cost  [2] batched (MPPI variant only)  [3] resident  [4] states  [5] unused
namespace {
void user_load(const ModelKernels* mk, void* dst, const double* blob, const double* ext, int n_ext) {
    for (int i = 0; i < mk->np; ++i) {
        const double v = i < MPPI_MODEL_PARAM_DOUBLES ? blob[i] : ((ext != nullptr && i - MPPI_MODEL_PARAM_DOUBLES < n_ext) ? ext[i - MPPI_MODEL_PARAM_DOUBLES] : 0.0);
        if (mk->is_double) reinterpret_cast<double*>(dst)[i] = v;
        else reinterpret_cast<float*>(dst)[i] = (float)v;
    }
}
}  // namespace

int mppi_user_model_register(const void* cubin, uint64_t cubin_bytes, int32_t nx, int32_t nu, int32_t n_params, int32_t dtype,
                             int32_t variant, const char* const* names, void** handle_out) {
    if (cubin == nullptr || cubin_bytes == 0 || names == nullptr || handle_out == nullptr) return MPPI_ERR_BAD_ARG;
    if (nx < 1 || nx > MPPI_MAX_NX || nu < 1 || nu > MPPI_MAX_NU || n_params < 1 || variant < 0 || variant > 2) return MPPI_ERR_BAD_ARG;
    if (dtype != MPPI_F32 && dtype != MPPI_F64) return MPPI_ERR_BAD_ARG;
    const int es = dtype == MPPI_F64 ? 8 : 4;
    if (n_params * es > MPPI_MODEL_BLOCK_BYTES) return UNSUPPORTED("user model has too many parameters");
    cudaLibrary_t lib = nullptr;
    CK(cudaLibraryLoadData(&lib, cubin, nullptr, nullptr, 0, nullptr, nullptr, 0));
    UserModelHandle* h = new (std::nothrow) UserModelHandle();
    if (h == nullptr) return MPPI_ERR_BAD_ARG;
    memset(h, 0, sizeof(*h));
    h->magic = kUserMagic;
    ModelKernels& mk = h->mk;
    mk.nx = nx;
    mk.nu = nu;
    mk.is_double = dtype == MPPI_F64;
    mk.np = n_params;
    mk.param_bytes = n_params * es;
    mk.load = user_load;
    mk.library = (void*)lib;
    const void** slots[5] = {&mk.fused[variant], &mk.split[variant], &mk.batched, &mk.resident[variant], &mk.states};
    for (int i = 0; i < 5; ++i) {
        if (names[i] == nullptr) continue;
        cudaKernel_t k = nullptr;
        cudaError_t e = cudaLibraryGetKernel(&k, lib, names[i]);
        if (e != cudaSuccess) {
            cudaLibraryUnload(lib);
            delete h;
            return cuda_fail(e, names[i]);
        }
        *slots[i] = (const void*)k;
    }
    if (mk.fused[variant] == nullptr || mk.states == nullptr) {
        cudaLibraryUnload(lib);
        delete h;
        return MPPI_ERR_BAD_ARG;
    }
    *handle_out = h;
    return MPPI_OK;
}

int mppi_user_model_release(void* handle) {
    UserModelHandle* h = reinterpret_cast<UserModelHandle*>(handle);
    if (h == nullptr || h->magic != kUserMagic) return MPPI_ERR_BAD_ARG;
    if (h->mk.library != nullptr) cudaLibraryUnload((cudaLibrary_t)h->mk.library);
    h->magic = 0;
    delete h;
    return MPPI_OK;
}

uint64_t mppi_plan_epoch(void* plan) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    if (pl == nullptr) return 0;
    const unsigned long long res = pl->res.armed ? pl->res_epoch_off + pl->res.seq : 0;
    return res > pl->epoch ? res : pl->epoch;
}

uint64_t mppi_resident_launches(void* plan) {
    Plan* pl = reinterpret_cast<Plan*>(plan);
    return pl == nullptr ? 0 : pl->res.launches;
}

int mppi_apply_partials(const MppiFusedParams* p, const void* partials, void* stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (partials == nullptr || p->nominal_used == nullptr || p->stats == nullptr || p->U == nullptr || p->action_out == nullptr)
        return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (p->dtype == MPPI_F32) {
        switch (p->variant) {
            case MPPI_VARIANT_MPPI: return run_apply<float, V_MPPI>(p, partials, s);
            case MPPI_VARIANT_SMPPI: return run_apply<float, V_SMPPI>(p, partials, s);
            case MPPI_VARIANT_KMPPI: return run_apply<float, V_KMPPI>(p, partials, s);
        }
    } else {
        switch (p->variant) {
            case MPPI_VARIANT_MPPI: return run_apply<double, V_MPPI>(p, partials, s);
            case MPPI_VARIANT_SMPPI: return run_apply<double, V_SMPPI>(p, partials, s);
            case MPPI_VARIANT_KMPPI: return run_apply<double, V_KMPPI>(p, partials, s);
        }
    }
    return MPPI_ERR_BAD_ARG;
}

// two epoch parities of MPPI_XCHG_PARITY_WORDS flagged 8-byte words, records of 2 (R+2) words: world x records per command
// (LL mode: every rank's cluster records, at most the 48 KB staging; rank-record mode: one record per rank)
uint64_t mppi_xchg_bytes(void) { return (uint64_t)2 * MPPI_XCHG_PARITY_WORDS * sizeof(unsigned long long); }
static_assert(MPPI_MAX_RANKS * MPPI_XCHG_MAX_WORDS <= MPPI_XCHG_PARITY_WORDS, "mailbox parity too small for one record per rank");

int mppi_xchg_create(void** mailbox, void* ipc_handle_out_64B) {
    if (mailbox == nullptr || ipc_handle_out_64B == nullptr) return MPPI_ERR_BAD_ARG;
    void* ptr = nullptr;
    CK(cudaMalloc(&ptr, mppi_xchg_bytes()));
    CK(cudaMemset(ptr, 0, mppi_xchg_bytes()));
    CK(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, ptr));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(ipc_handle_out_64B, &h, 64);
    *mailbox = ptr;
    return MPPI_OK;
}

int mppi_xchg_open(const void* ipc_handle_64B, void** peer_mailbox) {
    if (ipc_handle_64B == nullptr || peer_mailbox == nullptr) return MPPI_ERR_BAD_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle_64B, 64);
    void* ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    *peer_mailbox = ptr;
    return MPPI_OK;
}

int mppi_xchg_close(void* peer_mailbox) {
    if (peer_mailbox == nullptr) return MPPI_ERR_BAD_ARG;
    CK(cudaIpcCloseMemHandle(peer_mailbox));
    return MPPI_OK;
}

int mppi_xchg_destroy(void* mailbox) {
    if (mailbox == nullptr) return MPPI_ERR_BAD_ARG;
    CK(cudaFree(mailbox));
    return MPPI_OK;
}

int mppi_materialize(const MppiFusedParams* p, void* perturbed_action, void* noise, void* noise_theta, void* states,
                     void* stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (p->nominal_used == nullptr) return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (states != nullptr && perturbed_action == nullptr) return MPPI_ERR_BAD_ARG;
    rc = p->dtype == MPPI_F32
             ? run_sample_any<float>(p, perturbed_action, noise, noise_theta, nullptr, nullptr, 0, 0, true, s)
             : run_sample_any<double>(p, perturbed_action, noise, noise_theta, nullptr, nullptr, 0, 0, true, s);
    if (rc || states == nullptr) return rc;
    const ModelKernels* mk = find_kernels(p, &rc);
    if (mk == nullptr) return rc;
    return mk->is_double ? run_states<double>(mk, p, perturbed_action, states, s) : run_states<float>(mk, p, perturbed_action, states, s);
}

int mppi_rollout_states(const MppiFusedParams* p, const void* start_states, const void* actions, int64_t actions_stride,
                        int32_t n_rollouts, int32_t T, void* states_out, void* stream) {
    if (p == nullptr || start_states == nullptr || actions == nullptr || states_out == nullptr) return MPPI_ERR_BAD_ARG;
    if (p->struct_size != sizeof(MppiFusedParams)) return MPPI_ERR_ABI;
    if (n_rollouts < 1 || T < 1 || actions_stride < 0) return MPPI_ERR_BAD_ARG;
    if (p->dtype != MPPI_F32 && p->dtype != MPPI_F64) return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    int rc = MPPI_ERR_UNSUPPORTED;
    const ModelKernels* mk = find_kernels(p, &rc);
    if (mk == nullptr) return rc;
    return mk->is_double ? run_rollout_states<double>(mk, p, start_states, actions, actions_stride, n_rollouts, T, states_out, s)
                         : run_rollout_states<float>(mk, p, start_states, actions, actions_stride, n_rollouts, T, states_out, s);
}

int mppi_sample_perturb(const MppiFusedParams* p, void* perturbed_action, void* noise, void* noise_theta, void* cost_init,
                        const void* override_rows, int32_t n_override, int32_t override_start, void* stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (p->U == nullptr || perturbed_action == nullptr || noise == nullptr || p->nominal_used == nullptr) return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    return p->dtype == MPPI_F32 ? run_sample_any<float>(p, perturbed_action, noise, noise_theta, cost_init, override_rows,
                                                        n_override, override_start, false, s)
                                : run_sample_any<double>(p, perturbed_action, noise, noise_theta, cost_init, override_rows,
                                                         n_override, override_start, false, s);
}

int mppi_cost_accumulate(void* cost, const void* c, void* var_acc, int32_t M, int32_t K, double discount, int32_t dtype,
                         void* stream) {
    if (cost == nullptr || c == nullptr || M < 1 || K < 1) return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int BD = 256, nb = (K + BD - 1) / BD;
    if (dtype == MPPI_F32)
        cost_accumulate_kernel<float><<<nb, BD, 0, s>>>((float*)cost, (const float*)c, (float*)var_acc, M, K, (float)discount);
    else if (dtype == MPPI_F64)
        cost_accumulate_kernel<double><<<nb, BD, 0, s>>>((double*)cost, (const double*)c, (double*)var_acc, M, K, discount);
    else
        return MPPI_ERR_BAD_ARG;
    CK(cudaGetLastError());
    return MPPI_OK;
}

int mppi_softmin_update(const MppiFusedParams* p, const void* cost_total, const void* eps, void* stream) {
    int rc = validate(p);
    if (rc) return rc;
    if (cost_total == nullptr || eps == nullptr || p->nominal_used == nullptr || p->U == nullptr || p->action_out == nullptr ||
        p->stats == nullptr)
        return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    return p->dtype == MPPI_F32 ? run_softmin_any<float>(p, cost_total, eps, s) : run_softmin_any<double>(p, cost_total, eps, s);
}

int mppi_omega(const void* cost_total, void* omega_out, const void* stats, double lambda_, int32_t K, int32_t dtype,
               void* stream) {
    if (cost_total == nullptr || omega_out == nullptr || stats == nullptr || K < 1 || lambda_ <= 0) return MPPI_ERR_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int BD = 256, nb = (K + BD - 1) / BD;
    if (dtype == MPPI_F32)
        omega_kernel<float><<<nb, BD, 0, s>>>((const float*)cost_total, (float*)omega_out, (const double*)stats,
                                              (float)(-(1.0 / lambda_)), K);
    else if (dtype == MPPI_F64)
        omega_kernel<double><<<nb, BD, 0, s>>>((const double*)cost_total, (double*)omega_out, (const double*)stats,
                                               -(1.0 / lambda_), K);
    else
        return MPPI_ERR_BAD_ARG;
    CK(cudaGetLastError());
    return MPPI_OK;
}

}  // extern "C"
