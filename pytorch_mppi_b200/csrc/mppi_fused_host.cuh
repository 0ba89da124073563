// mppi_fused_host.cuh — kernel selection, launch geometry, plans and launches of the fused command, for ANY model: the
// model enters through a ModelKernels descriptor (kernel handles + parameter packing), so this is compiled once, in
// mppi_b200.cu, and serves the registry models and NVRTC-compiled user models alike.
#pragma once
#include "mppi_host.cuh"

namespace {

// ---- fused command ----------------------------------------------------------------------------
// PENDULUM_MLP in fp32 with model_params[3] != 0: the tcgen05/TMEM kernel (mppi_mlp_tc.cuh).  One CTA = 256 threads = 128
// samples (two threads per sample) = the 128 lanes of an M=128 accumulator tile; it does not take part in PDL.
inline bool select_tensor_core_route(const ModelKernels* mk, const MppiFusedParams* p, MppiFusedParams& p_tc, const void*& kernel) {
    if (mk->is_mlp && !mk->is_double) {
        int mode = (int)p->model_params[3];            // 1: hi/lo-split bf16 operands ("3 x bf16"), 2: plain bf16, 3: automatic
        // automatic (the Python default): the tensor-core kernel with split operands — the parity route — wherever it
        // exists (fp32, one environment); it is faster than the FFMA kernel at every K from 1024 to 131072
        // (profiles/r02_c4_routes.txt: 78 against 113 us at K = 1024, 102 against 141 at 32768, 320 against 337 at 131072)
        if (mode == 3) mode = 1;
        const int fast = p->model_params[2] != 0.0 ? 1 : 0;
        if ((mode == 1 || mode == 2) && p->n_env <= 1 && mk->tc[p->variant][mode - 1][fast] != nullptr) {
            p_tc = *p;
            p_tc.block_threads = 128;                   // samples per tile
            p_tc.threads_per_sample = 2;
            p_tc.flags &= ~(uint32_t)MPPI_FLAG_PDL;
            kernel = mk->tc[p->variant][mode - 1][fast];
            g_tc_kernel = 1;
            g_tc_cols = 64;                             // tc::TMEM_COLS (mppi_mlp_tc.cuh)
            // co-residency is bounded by shared memory: ask for the largest carve-out
            cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            return true;
        }
    }
    return false;
}

// ---- kernel + launch geometry of one fused command -------------------------------------------------------------------
// What is decided here, once per plan (or per mppi_fused_command call):
//   kernel     fused_command_kernel<Model, real, V, batched, split>  (or the tcgen05 kernel, select_tensor_core_route)
//   geometry   tile size / helper threads / grid (plan_geometry), planned for K_geom samples on sharded controllers so
//              that every rank launches the same grid
//   split      MPPI_FLAG_SPLIT_COST honoured: problems small enough to run with helper threads (threads_per_sample > 1)
//              take the split-cost rollout if its per-step state buffer fits in shared memory
//   cluster    thread-block-cluster size of the warp-fold tail: 8 / 4 / 2 when the whole grid is one wave of at most
//              one CTA per SM and all its clusters are co-resident (cudaOccupancyMaxActiveClusters), else 1
//   npub       sharded controllers: the records a rank publishes to its peers per command — its cluster records when
//              their staging (world x clusters x (R+2) doubles) is small (direct mode), else its one combined record
struct FusedChoice {
    const void* kernel;
    Geometry g;
    int split, wide, tc;
};

template <typename real>
int choose_fused(const ModelKernels* mk, const MppiFusedParams*& p, MppiFusedParams& p_tc, FusedChoice& c) {
    if (p->nx != mk->nx || p->nu != mk->nu) return MPPI_ERR_BAD_ARG;
    const int V = p->variant;
    const bool batched = p->n_env > 1;
    if (batched && (V != V_MPPI || p->world > 1)) return UNSUPPORTED("batched environments: MPPI variant, single GPU only");
    const void* kernel = batched ? mk->batched : mk->fused[V];
    if (kernel == nullptr) return UNSUPPORTED("this model was built without the kernel of this controller variant");
    const bool tc_route = select_tensor_core_route(mk, p, p_tc, kernel);
    if (tc_route) p = &p_tc;
    const int R = rows_of(p), es = (int)sizeof(real);
    const int world = p->world <= 0 ? 1 : p->world;
    const bool sharded = sharded_in_kernel(p);
    MppiFusedParams pg = *p;
    if (p->K_geom > p->K) pg.K = p->K_geom;
    Geometry g;
    int rc;
    if (tc_route) {
        rc = plan_geometry(kernel, &pg, es, ticket_layout_extra(p), false, g, layout_fn<real>);
        g_tc_kernel = 0;
        if (rc) return rc;
        c = FusedChoice{kernel, g, 0, 0, 1};
        return MPPI_OK;
    }
    const int xst1 = sharded ? world * (R + 2) : 0;          // staging of the rank-record exchange
    const int tile2 = V != V_MPPI;                          // SMPPI: effective-noise tile, KMPPI: interpolated-trajectory tile
    rc = plan_geometry(kernel, &pg, es, layout_extra(tile2, 0, 1, xst1), true, g, layout_fn<real>);
    if (rc) return rc;
    int split = 0;
    if (mk->split[V] != nullptr) {      // (the MLP has none: its step is the network, the cost is nothing)
        if (!batched && (p->flags & MPPI_FLAG_SPLIT_COST) && g.tps > 1) {
            const void* k2 = mk->split[V];
            MppiFusedParams p2 = pg;
            p2.block_threads = g.BS;
            p2.threads_per_sample = g.tps;
            p2.grid_blocks = g.nb;
            Geometry g2;
            if (plan_geometry(k2, &p2, es, layout_extra(tile2, mk->nx, 1, xst1), true, g2, layout_fn<real>) == MPPI_OK &&
                g2.BS == g.BS && g2.tps == g.tps) {
                kernel = k2;
                g = g2;
                split = 1;
            }
        }
    }
    // ---- cluster size and exchange mode ------------------------------------------------------------------------------
    DevInfo di;
    rc = get_dev_info(di);
    if (rc) return rc;
    int want = 8;
    if (const char* e = getenv("MPPI_B200_CLUSTER")) want = atoi(e);
    cudaFuncAttributes fa;
    CK(cudaFuncGetAttributes(&fa, kernel));
    const int dyn_limit = di.max_smem_optin - (int)fa.sharedSizeBytes;
    const int envs = batched ? p->n_env : 1;
    g.cluster = 0;
    g.npub = 1;
    for (int cs = 8; cs >= 1; cs >>= 1) {
        if (cs > want && cs > 1) continue;
        const int nbp = (g.nb + cs - 1) / cs * cs;
        if (cs > 2 && nbp > di.sm_count) continue;                        // 8 / 4: one wave of at most one CTA per SM (pairs pack anywhere)
        if (cs > 1 && (g.nb < 2 || nbp > di.sm_count * g.occ)) continue;
        const int NC = nbp / cs;
        // LL mode: the finisher (leader of cluster 0) stages every rank's cluster records: xw x NC x (R+2) doubles
        const int xw = sharded ? world : 1;
        int npub = 1;
        if (NC > 1 && (long long)xw * NC * (R + 2) * 8 <= MPPI_LL_STAGE_BYTES) npub = NC;
        if (const char* e = getenv("MPPI_B200_XCHG_DIRECT"))
            if (atoi(e) == 0) npub = 1;
        const int xst = fused_xstage_doubles(sharded, world, npub, R);
        const SmemLayout L = make_layout<real>(p->variant, p->T, p->nu, p->S, R, g.BD, g.BS, fused_layout_nb(NC, npub),
                                               layout_extra(tile2, split ? mk->nx : 0, cs, xst));
        if (L.total > dyn_limit) continue;
        if (cs > 1) {
            cudaLaunchConfig_t cfg;
            cudaLaunchAttribute at[3];
            launch_config(cfg, at, nbp, g.BD, L.total, nullptr, (p->flags & MPPI_FLAG_PDL) != 0, envs, cs);
            int max_clusters = 0;
            if (cudaOccupancyMaxActiveClusters(&max_clusters, kernel, &cfg) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            if (getenv("MPPI_B200_DEBUG_GEOM"))
                fprintf(stderr, "[mppi_b200] cluster %d: grid %d, smem %d, max active clusters %d (need %d)\n", cs, nbp, L.total, max_clusters, NC * envs);
            if (max_clusters < NC * envs) continue;                       // a cluster left for a second wave doubles the time
        }
        g.cluster = cs;
        g.nb = nbp;
        g.smem = L.total;
        g.npub = npub;
        break;
    }
    if (g.cluster == 0) return UNSUPPORTED("shared-memory tile does not fit");
    c = FusedChoice{kernel, g, split, 0, 0};
    return MPPI_OK;
}

template <typename real> void finish_kargs(const MppiFusedParams* p, const FusedChoice& c, KArgs<real>& a) {
    fill_kargs<real>(p, a, c.g.BS, c.g.nb, c.g.tps);
    a.xchg_npub = c.g.npub > 0 ? c.g.npub : 1;
}

template <typename real>
int run_fused(const ModelKernels* mk, const MppiFusedParams* p, cudaStream_t stream, MppiLaunchInfo* info) {
    const bool batched = p->n_env > 1;
    if (batched && info == nullptr && !(p->flags & MPPI_FLAG_STATE_DEVICE)) return MPPI_ERR_BAD_ARG;   // states are (n_env, nx) on the device
    MppiFusedParams p_tc;
    FusedChoice c;
    int rc = choose_fused<real>(mk, p, p_tc, c);
    if (rc) return rc;
    const Geometry& g = c.g;
    const uint64_t need_ws = ws_bytes(g.nb, rows_of(p));
    KArgs<real> a;
    finish_kargs<real>(p, c, a);
    if (info != nullptr) {
        DevInfo di;
        get_dev_info(di);
        info->block_threads = g.BD;
        info->threads_per_sample = g.tps;
        info->grid_blocks = g.nb;
        info->smem_bytes = g.smem;
        info->regs_per_thread = g.regs;
        info->max_blocks_per_sm = g.occ;
        info->sm_count = di.sm_count;
        // report the worst case so one allocation serves any later geometry for these dimensions
        info->workspace_bytes = ws_bytes(di.sm_count * 16, rows_of(p));
        info->tma_staging = a.tma_ok;
        info->split_cost = c.split;
        info->wide_regs = c.wide;
        info->cluster_size = g.cluster;
        info->xchg_records = g.npub;
        return MPPI_OK;
    }
    if (p->U == nullptr || p->cost_total == nullptr || p->action_out == nullptr || p->nominal_used == nullptr ||
        p->stats == nullptr || p->workspace == nullptr)
        return MPPI_ERR_BAD_ARG;
    if (p->workspace_bytes < need_ws) return MPPI_ERR_WORKSPACE;
    if (batched && (p->env_ws_stride < need_ws || p->workspace_bytes < p->env_ws_stride * (uint64_t)p->n_env ||
                    p->env_u_stride < p->T * p->nu))
        return MPPI_ERR_WORKSPACE;
    if (a.world > 1 && rows_of(p) > MPPI_XCHG_MAX_R) return UNSUPPORTED("T*nu exceeds the peer mailbox record size");
    if (a.export_partial && p->partial_out == nullptr) return MPPI_ERR_BAD_ARG;
    alignas(16) unsigned char mp[MPPI_MODEL_BLOCK_BYTES];
    if (mk->param_bytes > (int)sizeof(mp)) return UNSUPPORTED("model parameter block too large");
    mk->load(mk, mp, p->model_params, p->model_params_ext, p->n_model_params_ext);
    if ((rc = refuse_capture(stream, g)) != MPPI_OK) return rc;
    if (a.world == 1 || a.export_partial) {       // plan-less single-GPU launches draw their record tags from one process-wide counter
        static unsigned long long s_epoch = 0;
        a.epoch = __atomic_add_fetch(&s_epoch, 1ull, __ATOMIC_RELAXED);
    }
    void* argv2[2] = {(void*)&a, (void*)mp};
    cudaError_t e = launch_raw(c.kernel, g.nb, g.BD, g.smem, stream, argv2, a.pdl != 0, a.n_env, g.cluster);
    if (e != cudaSuccess) return cuda_fail(e, "fused launch");
    return MPPI_OK;
}

template <typename real> int build_plan(const ModelKernels* mk, const MppiFusedParams* p, Plan* pl) {
    const bool batched = p->n_env > 1;
    const int V = p->variant;
    MppiFusedParams p_tc;
    FusedChoice c;
    int rc = choose_fused<real>(mk, p, p_tc, c);
    if (rc) return rc;
    pl->g = c.g;
    if (p->U == nullptr || p->cost_total == nullptr || p->nominal_used == nullptr || p->stats == nullptr || p->workspace == nullptr)
        return MPPI_ERR_BAD_ARG;
    if (p->workspace_bytes < ws_bytes(pl->g.nb, rows_of(p))) return MPPI_ERR_WORKSPACE;
    if (mk->param_bytes > (int)sizeof(pl->mparams)) return UNSUPPORTED("model parameter block too large");
    KArgs<real>* a = reinterpret_cast<KArgs<real>*>(pl->kargs);
    finish_kargs<real>(p, c, *a);
    if (a->world > 1 && rows_of(p) > MPPI_XCHG_MAX_R) return UNSUPPORTED("T*nu exceeds the peer mailbox record size");
    mk->load(mk, pl->mparams, p->model_params, p->model_params_ext, p->n_model_params_ext);
    pl->kernel = c.kernel;
    pl->res_kernel = nullptr;
    pl->res_xchg = 0;
    // resident mode runs the split-cost rollout with one tile per CTA: exactly the single-GPU plans that took it, with
    // the launch route's grid and cluster size (mppi_resident.cuh)
    if (c.split && !batched && !a->export_partial && a->world == 1 && a->n_tiles <= pl->g.nb && pl->g.nb <= a->n_tiles + pl->g.cluster - 1) {
        pl->res_kernel = mk->resident[V];
        // the one instantiation with %globaltimer stamps (a profiling aid, scripts/resident_timeline.py)
        if (pl->res_kernel != nullptr && p->debug_clocks != nullptr && V == V_MPPI && mk->resident_stamped != nullptr)
            pl->res_kernel = mk->resident_stamped;
    }
    pl->is_double = sizeof(real) == 8;
    pl->nx = mk->nx;
    pl->upc_nu = p->u_per_command * p->nu;
    pl->pdl = (p->flags & MPPI_FLAG_PDL) ? 1 : 0;
    pl->epoch = p->epoch;
    pl->res_epoch_off = 0;
    pl->host_epoch = p->host_epoch;      // monotonic across re-plans: a stale mailbox tag of an earlier plan can never match
    pl->p = *p;
    return MPPI_OK;
}

template <typename real>
int launch_states(const ModelKernels* mk, const MppiFusedParams* p, KArgs<real>& a, int n, const void* actions, void* states,
                  long long stride, cudaStream_t stream) {
    alignas(16) unsigned char mp[MPPI_MODEL_BLOCK_BYTES];
    if (mk->param_bytes > (int)sizeof(mp)) return UNSUPPORTED("model parameter block too large");
    mk->load(mk, mp, p->model_params, p->model_params_ext, p->n_model_params_ext);
    const real* pa = (const real*)actions;
    real* st = (real*)states;
    void* argv[5] = {(void*)&pa, (void*)&st, (void*)&a, (void*)mp, (void*)&stride};
    cudaError_t e = cudaLaunchKernel(mk->states, dim3((n + 127) / 128), dim3(128), argv, 0, stream);
    if (e != cudaSuccess) return cuda_fail(e, "states launch");
    return MPPI_OK;
}

// states along the rollouts of the last command's perturbed actions (mppi.py:307-322)
template <typename real>
int run_states(const ModelKernels* mk, const MppiFusedParams* p, const void* pa, void* states, cudaStream_t stream) {
    if (p->nx != mk->nx || p->nu != mk->nu) return MPPI_ERR_BAD_ARG;
    KArgs<real> a;
    fill_kargs<real>(p, a, 128, 1);
    return launch_states<real>(mk, p, a, p->K, pa, states, (long long)p->T * p->nu, stream);
}

// get_rollouts (mppi.py:425-448): n start states, each rolled through an action sequence
template <typename real>
int run_rollout_states(const ModelKernels* mk, const MppiFusedParams* p, const void* start_states, const void* actions, long long stride,
                       int n, int T, void* states, cudaStream_t stream) {
    if (p->nx != mk->nx || p->nu != mk->nu) return MPPI_ERR_BAD_ARG;
    KArgs<real> a;
    memset(&a, 0, sizeof(a));
    a.nm.u_scale = (real)p->u_scale;
    a.K = n;
    a.T = T;
    a.state_dev = (const real*)start_states;
    a.state_per_sample = 1;
    return launch_states<real>(mk, p, a, n, actions, states, stride, stream);
}

}  // namespace

