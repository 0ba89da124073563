// mppi_fused.cuh — device side of the MPPI engine.
//
// fused_command_kernel: one kernel per MPPI/SMPPI/KMPPI command() for registered analytic models.
// One thread rolls out one sample; a CTA owns tiles of `blockDim.x` samples (grid-stride over tiles,
// so grid <= SMs x resident CTAs for any K).  Per tile:
//   A. standard normals -> shared-memory tile rows[R][BD+1]  (in-kernel Philox4x32-10 keyed by the
//      GLOBAL sample index, or an injected z tensor loaded coalesced)
//   B. colour with the Cholesky factor, add the nominal sequence (staged in shared memory by a TMA
//      bulk copy), clamp -> the tile now holds the perturbed actions (KMPPI: the control points)
//   C. T-step rollout with the state in registers, cost accumulated in the reference's op order
//   D. online-softmin fold: every rollout warp folds its 32 samples into its own running record (warp_fold)
// The tail (warp_tail) combines the warp records of a CTA or cluster, then those of the grid (last arrival of an atomic
// ticket, or a poller of flagged records), optionally exchanges the rank record with peer GPUs through NVLink mailboxes,
// and writes the updated nominal sequence: `U += sum_k w_k eps_k / eta` lands without a second launch.
//
// sample_kernel / softmin_update_kernel: the same stages split at the Python T-loop, for arbitrary
// dynamics/cost callables (A+B with coalesced write-out; D + the same tail from materialised tensors).
//
// Reference lines replaced: mppi.py:232-238, 375-385, 297-332, 407-417, 254-259, 268-270
// (SMPPI :489-493, 520-570; KMPPI :617-619, 657-688).
#pragma once

#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#endif
#include "mppi_math.cuh"

#ifndef MPPI_ROLLOUT_PIPELINED
#define MPPI_ROLLOUT_PIPELINED 0
#endif
#ifndef MPPI_ROLLOUT_UNROLL
#define MPPI_ROLLOUT_UNROLL 2
#endif
// minimum resident CTAs per SM promised to ptxas for the fused kernel: 2 keeps 512-thread CTAs at 64 registers, two per
// SM — what large K wants (left unspecified, ptxas sizes the kernel for its out-of-line tail functions: 128 registers,
// one CTA per SM, and BASELINE config 5 loses 25 %); the split-cost variant (small K, one CTA per SM) lifts the cap
#ifndef MPPI_FUSED_MIN_BLOCKS
#define MPPI_FUSED_MIN_BLOCKS 2
#endif
#define MPPI_PRAGMA_(x) _Pragma(#x)
#define MPPI_UNROLL_N(n) MPPI_PRAGMA_(unroll n)

namespace mppi {

enum { V_MPPI = 0, V_SMPPI = 1, V_KMPPI = 2 };

template <typename real> struct KArgs {
    NoiseModel<real> nm;
    real u_init[MPPI_MAX_NU];
    real x0[MPPI_MAX_NX];
    const real* state_dev;
    real* U;
    real* A;
    real* theta;
    const real* W;
    const real* Wshift;
    real* cost_total;
    real* action_out;
    real* nominal_used;
    double* stats;
    const real* z;
    real* z_out;
    // workspace carve
    unsigned int* ticket;
    double* crec;                 // cluster records (n_clusters, R+2) doubles: (beta, eta, V[R])
    // multi-GPU
    unsigned long long* peers[8];
    double* partial_out;
    unsigned long long epoch;
    int rank, world, export_partial;
    int xchg_npub;                // records each rank publishes per command: its cluster records (LL mode) or 1
    unsigned int xchg_parity_words;   // 8-byte words between the two epoch parities of a record mailbox
    unsigned long long xchg_timeout_ns;
    long long* xchg_status_host;  // optional pinned host word: set to MPPI_ERR_TIMEOUT when a peer exchange timed out
    // sizes
    int K, T, S, R, TN, upc, n_tiles;
    long long k_offset;
    unsigned long long seed, offset;
    int shift, null_action, tma_ok, state_per_sample;
    int tps;   // threads cooperating on one sample's sampling/transform phases (1, 2 or 4)
    int pdl;   // launched with programmatic stream serialization
    unsigned long long torch_total;   // > 0: reproduce torch.randn's CUDA stream (256 * grid of the ATen kernel)
    unsigned long long* offset_dev;   // optional device-resident Philox counter base (CUDA-graph replays)
    unsigned long long offset_inc;
    // batched environments (MPPI_Batched, mppi.py:691-873): gridDim.y = n_env independent problems that
    // share the noise stream; per-environment buffers are strided
    int n_env;
    long long env_u_stride;      // elements between consecutive environments' U
    long long env_ws_stride;     // BYTES between consecutive environments' workspace
    unsigned long long* dbg;   // optional (grid,16) globaltimer stamps
    unsigned long long* host_mailbox;   // optional pinned host memory: [0]=epoch flag, [2..]=action values
    unsigned long long host_epoch;
    // generic-path extras (sample_kernel / softmin_update_kernel)
    real* out_pa;
    real* out_noise;
    real* out_noise_theta;
    real* out_cost_init;
    const real* override_rows;
    int n_override, override_start;
    const real* in_cost;
    const real* in_eps;
    real* out_omega;
};

// ---- shared-memory carve, computed identically on host and device -------------------------------
struct SmemLayout {
    int off_uraw, off_araw, off_thraw, off_us, off_as, off_ths, off_w, off_wsh, off_rows, off_rows2, off_part2, off_numd,
        off_xs, off_wrec, off_xstage, off_sqd, total;
    int LD;
};

// `extra` word of make_layout: bit 0 = rows2 tile; bits 8..15 = nx of the split-cost state buffer; bits 16..19 = cluster
// size of the warp-record area (0 = the kernel does not use the warp-fold tail); bits 20..30 = record staging of the
// finisher in units of 16 doubles (at most 8208 doubles: 8 ranks x 1026, or the 48 KB LL budget)
__host__ __device__ inline int layout_extra(int rows2, int nx_split, int cluster, int xstage_doubles) {
    return (rows2 & 1) | (nx_split << 8) | (cluster << 16) | (((xstage_doubles + 15) / 16) << 20);
}

__host__ __device__ inline int align_up(int x, int a) { return (x + a - 1) / a * a; }

// BD = threads per CTA, BS = samples per tile (BD / threads-per-sample)
// `extra` (layout_extra): bit 0 = rows2 tile (a second TN-row tile: the fused kernels' SMPPI / KMPPI tile, sample_kernel's
// KMPPI trajectories); bits 8.. = nx of the split-cost rollout's per-step state buffer xs[T*nx][BS] (0 = none; see
// fused_command_kernel<..., SPLIT>); the warp-record area and the finisher's staging (see above)
// nb = records the finisher reads from the L2 workspace (ticket mode; 1 otherwise): their rescale factors live in sqd
template <typename real>
__host__ __device__ inline SmemLayout make_layout(int variant, int T, int nu, int S, int R, int BD, int BS, int nb, int extra) {
    SmemLayout L;
    const int need_rows2 = extra & 1, nx_split = (extra >> 8) & 0xff, cluster = (extra >> 16) & 0xf, xstage = (extra >> 20) * 16;
    const int es = (int)sizeof(real);
    const int TN = T * nu, SN = S * nu, nw = BD / 32;
    int o = 16;  // [0,8): mbarrier
    L.off_uraw = o; o = align_up(o + TN * es, 16);
    L.off_araw = o; o = align_up(o + (variant == V_SMPPI ? TN : 0) * es, 16);
    L.off_thraw = o; o = align_up(o + (variant == V_KMPPI ? SN : 0) * es, 16);
    L.off_us = o; o = align_up(o + TN * es, 16);
    L.off_as = o; o = align_up(o + (variant == V_SMPPI ? TN : 0) * es, 16);
    L.off_ths = o; o = align_up(o + (variant == V_KMPPI ? SN : 0) * es, 16);
    L.off_w = o; o = align_up(o + (variant == V_KMPPI ? T * S : 0) * es, 16);
    L.off_wsh = o; o = align_up(o + (variant == V_KMPPI ? S * S : 0) * es, 16);
    L.LD = BS + 1;
    L.off_rows = o; o = align_up(o + R * L.LD * es, 16);
    L.off_rows2 = o; o = align_up(o + (need_rows2 ? TN * L.LD : 0) * es, 16);
    // combine_*: (BD / 64) groups x (R + 1) columns, and one group in a CTA of one warp
    L.off_part2 = o; o = align_up(o + (nw > 1 ? nw * R : R + 1) * 8, 16);
    L.off_numd = o; o = align_up(o + (R + 2) * 8, 16);
    L.off_xs = o; o = align_up(o + T * nx_split * BS * es, 16);
    // warp-fold tail: (cluster x rollout warps) records of (R+2) doubles — slots [0, BS/32) are this CTA's own running
    // records, the cluster leader also receives its peers' through distributed shared memory
    L.off_wrec = o; o = align_up(o + cluster * (BS / 32) * (R + 2) * 8, 16);
    L.off_xstage = o; o = align_up(o + xstage * 8, 16);
    // rescale factors of combine_records: one per record — the cluster's warp records, the staged records, or (ticket
    // mode: the caller passes nb = number of cluster records of the grid) the records in the L2 workspace
    {
        int nsq = cluster * (BS / 32);
        if (xstage / (R + 2) > nsq) nsq = xstage / (R + 2);
        if (nb > nsq) nsq = nb;
        L.off_sqd = o; o = align_up(o + (cluster > 0 ? nsq : 0) * 8, 16);
    }
    L.total = o;
    return L;
}

#define MPPI_XCHG_MAX_R 1024                            // rows of a record a sharded controller exchanges
#define MPPI_XCHG_MAX_WORDS (2 * (MPPI_XCHG_MAX_R + 2))  // mailbox words of such a record

#if defined(__CUDACC__)

// ---- mbarrier + TMA bulk copy (cp.async.bulk; SASS: UBLKCP) --------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, void* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t phase) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    }
}

__device__ __forceinline__ void stamp(unsigned long long* dbg, int slot) {
    if (dbg != nullptr && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        dbg[(size_t)blockIdx.x * 16 + slot] = t;
    }
}

// ---- warp reductions (deterministic: fixed shuffle tree) -----------------------------------------
template <typename T> __device__ __forceinline__ T warp_min(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T other = __shfl_xor_sync(0xffffffffu, v, o);
        v = other < v ? other : v;
    }
    return v;
}
template <typename T> __device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- shared-memory view ---------------------------------------------------------------------
template <typename real> struct Smem {
    unsigned long long* bar;
    real *Uraw, *Araw, *thraw, *Us, *As, *ths, *Ws, *Wsh, *rows, *rows2, *xs;
    double *part2, *numd, *wrec, *xstage, *sqd;
    int LD;
    __device__ Smem(unsigned char* smem, const SmemLayout& L) {
        bar = reinterpret_cast<unsigned long long*>(smem);
        Uraw = reinterpret_cast<real*>(smem + L.off_uraw);
        Araw = reinterpret_cast<real*>(smem + L.off_araw);
        thraw = reinterpret_cast<real*>(smem + L.off_thraw);
        Us = reinterpret_cast<real*>(smem + L.off_us);
        As = reinterpret_cast<real*>(smem + L.off_as);
        ths = reinterpret_cast<real*>(smem + L.off_ths);
        Ws = reinterpret_cast<real*>(smem + L.off_w);
        Wsh = reinterpret_cast<real*>(smem + L.off_wsh);
        rows = reinterpret_cast<real*>(smem + L.off_rows);
        rows2 = reinterpret_cast<real*>(smem + L.off_rows2);
        part2 = reinterpret_cast<double*>(smem + L.off_part2);
        numd = reinterpret_cast<double*>(smem + L.off_numd);
        xs = reinterpret_cast<real*>(smem + L.off_xs);
        wrec = reinterpret_cast<double*>(smem + L.off_wrec);
        xstage = reinterpret_cast<double*>(smem + L.off_xstage);
        sqd = reinterpret_cast<double*>(smem + L.off_sqd);
        LD = L.LD;
    }
};

// ---- stage 0: nominal sequence(s) into shared memory, shift folded in ----------------------------
// stage_issue starts the (asynchronous) TMA bulk copy; stage_finish waits for it and builds the
// shifted nominal.  The first tile's Philox draws run in between, hiding the global-memory latency.
template <typename real, int VARIANT, int NU>
__device__ void stage_issue(const KArgs<real>& a, Smem<real>& sm) {
    const int tid = threadIdx.x, BD = blockDim.x;
    const int T = a.T, S = a.S, R = a.R, TN = a.TN;
    if (tid == 0) mbar_init(sm.bar, 1);
    __syncthreads();
    if (a.tma_ok) {
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)align_up(TN * (int)sizeof(real), 16);
            mbar_expect_tx(sm.bar, VARIANT == V_SMPPI ? 2 * bytes : bytes);
            tma_bulk_g2s(sm.Uraw, a.U, bytes, sm.bar);
            if (VARIANT == V_SMPPI) tma_bulk_g2s(sm.Araw, a.A, bytes, sm.bar);
        }
    } else {
        for (int j = tid; j < TN; j += BD) {
            sm.Uraw[j] = a.U[j];
            if (VARIANT == V_SMPPI) sm.Araw[j] = a.A[j];
        }
    }
    if (VARIANT == V_KMPPI) {
        for (int j = tid; j < R; j += BD) sm.thraw[j] = a.theta[j];
        for (int j = tid; j < T * S; j += BD) sm.Ws[j] = a.W[j];
        if (a.shift)
            for (int j = tid; j < S * S; j += BD) sm.Wsh[j] = a.Wshift[j];
    }
}

template <typename real, int VARIANT, int NU>
__device__ void stage_finish(const KArgs<real>& a, Smem<real>& sm) {
    typedef Ops<real> O;
    const int tid = threadIdx.x, BD = blockDim.x;
    const int T = a.T, S = a.S, R = a.R, TN = a.TN;
    if (a.tma_ok) mbar_wait(sm.bar, 0);
    __syncthreads();
    for (int j = tid; j < TN; j += BD) {
        const int t = j / NU, n = j - t * NU;
        sm.Us[j] = a.shift ? (t + 1 < T ? sm.Uraw[j + NU] : a.u_init[n]) : sm.Uraw[j];               // mppi.py:237-238
        if (VARIANT == V_SMPPI) sm.As[j] = a.shift ? (t + 1 < T ? sm.Araw[j + NU] : sm.Araw[j]) : sm.Araw[j];  // :492-493
    }
    if (VARIANT == V_KMPPI) {
        for (int j = tid; j < R; j += BD) {
            const int s = j / NU, n = j - s * NU;
            if (a.shift) {                                                                 // mppi.py:619
                real acc = O::mul(sm.Wsh[s * S], sm.thraw[n]);
                for (int q = 1; q < S; ++q) acc = O::add(acc, O::mul(sm.Wsh[s * S + q], sm.thraw[q * NU + n]));
                sm.ths[j] = acc;
            } else {
                sm.ths[j] = sm.thraw[j];
            }
        }
    }
    __syncthreads();
}

template <typename real, int VARIANT, int NU>
__device__ void stage_nominal(const KArgs<real>& a, Smem<real>& sm) {
    stage_issue<real, VARIANT, NU>(a, sm);
    stage_finish<real, VARIANT, NU>(a, sm);
}

// ---- stage A: standard normals into the tile ------------------------------------------------------
// (thread -> sample s = tid % BS, chunk lane g = tid / BS: the tps threads of a sample split its
// Philox chunks)
// the rarely-taken sources of normals, out of line so that they do not sit in the hot path's instruction stream:
// injected z (parity tests), the torch-compatible stream (one Philox call per element), recording of the draws (z_out)
template <typename real>
__device__ __noinline__ void fill_normals_rare(const KArgs<real>& a, real* rows, int LD, int tile, bool active, unsigned long long kg, int nvalid) {
    const int tid = threadIdx.x, BD = blockDim.x, R = a.R;
    const int BS = BD / a.tps, s_ = tid % BS, g_ = tid / BS;
    if (a.z != nullptr) {
        const size_t base = (size_t)tile * BS * R;
        const int count = nvalid * R;
        for (int e = tid; e < count; e += BD) {
            const int s = e / R, j = e - s * R;
            rows[j * LD + s] = a.z[base + e];
        }
        __syncthreads();
    } else if (a.torch_total > 0 && active) {
        // torch-compatible stream: one Philox call per element (the ATen kernel scatters each call's
        // outputs `total` elements apart), 4x the generator work of the native stream
        constexpr int UN = TorchNormal<real>::UNROLL;
        real* col = rows + s_;
        const unsigned long long off = a.offset_dev != nullptr ? __ldcg(a.offset_dev) : a.offset;
        for (int j = g_; j < R; j += a.tps) {
            const unsigned long long li = kg * (unsigned long long)R + (unsigned long long)j;
            const unsigned long long idx = li % a.torch_total, m = li / a.torch_total;
            col[j * LD] = TorchNormal<real>::one(a.seed, idx, off + m / UN, (int)(m % UN));
        }
    }
}
template <typename real>
__device__ __noinline__ void record_normals(const KArgs<real>& a, const real* rows, int LD, int tile, int nvalid) {
    const int tid = threadIdx.x, BD = blockDim.x, R = a.R, BS = BD / a.tps;
    __syncthreads();
    const size_t base = (size_t)tile * BS * R;
    const int count = nvalid * R;
    for (int e = tid; e < count; e += BD) {
        const int s = e / R, j = e - s * R;
        a.z_out[base + e] = rows[j * LD + s];
    }
    __syncthreads();
}

template <typename real>
__device__ void fill_normals(const KArgs<real>& a, Smem<real>& sm, int tile, bool active, unsigned long long kg, int nvalid) {
    const int tid = threadIdx.x, BD = blockDim.x, R = a.R, LD = sm.LD;
    const int BS = BD / a.tps, s_ = tid % BS, g_ = tid / BS;
    if (a.z != nullptr || a.torch_total > 0) {
        fill_normals_rare<real>(a, sm.rows, LD, tile, active, kg, nvalid);
    } else if (active) {
        constexpr int PER = Normals<real>::PER_CALL;
        real* col = sm.rows + s_;
        const unsigned long long off = a.offset_dev != nullptr ? __ldcg(a.offset_dev) : a.offset;
        for (int c = g_; c * PER < R; c += a.tps) {
            real tmp[PER];
            Normals<real>::draw(a.seed, kg, off + (unsigned long long)c, tmp);
#pragma unroll
            for (int q = 0; q < PER; ++q)
                if (c * PER + q < R) col[(c * PER + q) * LD] = tmp[q];
        }
    }
    if (a.z_out != nullptr) record_normals<real>(a, sm.rows, LD, tile, nvalid);
}

// value that overrides the sampled action before the clamp: null action (mppi.py:390-392) or a
// SpecificActionSampler row (mppi.py:393-399); returns true if overridden
template <typename real>
__device__ __forceinline__ bool override_value(const KArgs<real>& a, unsigned long long kg, int j, real& p) {
    if (a.null_action && kg == 0ull) { p = (real)0; return true; }
    if (a.override_rows != nullptr) {
        const long long r = (long long)kg - a.override_start;
        if (r >= 0 && r < a.n_override) { p = a.override_rows[(size_t)r * a.TN + j]; return true; }
    }
    return false;
}

// ---- stage B: colour + nominal + clamp, in place in this thread's column --------------------------
// TILE2 (fused / resident kernels): a second tile `rows2` of T*nu rows per sample keeps what the serial rollout thread
// would otherwise recompute per step — SMPPI: the effective noise eps = (v - A)/dt - U (one IEEE division per element,
// needed by the action cost and by the softmin fold); KMPPI: the interpolated, clamped trajectory (interp_column).
template <typename real, int VARIANT, int NU, bool TILE2 = false>
__device__ __forceinline__ void transform_column(const KArgs<real>& a, Smem<real>& sm, unsigned long long kg) {
    typedef Ops<real> O;
    const NoiseModel<real>& nm = a.nm;
    const int LD = sm.LD;
    const int BS = blockDim.x / a.tps, s_ = threadIdx.x % BS, g_ = threadIdx.x / BS;
    real* col = sm.rows + s_;
    if (VARIANT == V_KMPPI) {
        for (int s = g_; s < a.S; s += a.tps) {                                           // mppi.py:660-664
            real zr[NU], e[NU];
#pragma unroll
            for (int n = 0; n < NU; ++n) zr[n] = col[(s * NU + n) * LD];
            colour<real, NU>(nm, zr, e);
#pragma unroll
            for (int n = 0; n < NU; ++n)
                col[(s * NU + n) * LD] = clamp<real>(O::add(sm.ths[s * NU + n], e[n]), nm.u_min[n], nm.u_max[n]);
        }
    } else {
        for (int t = g_; t < a.T; t += a.tps) {
            real zr[NU], e[NU];
#pragma unroll
            for (int n = 0; n < NU; ++n) zr[n] = col[(t * NU + n) * LD];
            colour<real, NU>(nm, zr, e);
#pragma unroll
            for (int n = 0; n < NU; ++n) {
                real p = O::add(sm.Us[t * NU + n], e[n]);                                 // mppi.py:380 / :544
                if (VARIANT == V_SMPPI) {
                    p = O::add(sm.As[t * NU + n], O::mul(p, nm.delta_t));                 // mppi.py:548
                    override_value<real>(a, kg, t * NU + n, p);                           // mppi.py:549
                    p = clamp<real>(p, nm.a_min[n], nm.a_max[n]);                         // mppi.py:550
                    if (TILE2)                                                            // mppi.py:552
                        sm.rows2[(t * NU + n) * LD + s_] = O::sub(O::div(O::sub(p, sm.As[t * NU + n]), nm.delta_t), sm.Us[t * NU + n]);
                } else {
                    override_value<real>(a, kg, t * NU + n, p);                           // mppi.py:381
                    p = clamp<real>(p, nm.u_min[n], nm.u_max[n]);                         // mppi.py:383
                }
                col[(t * NU + n) * LD] = p;
            }
        }
    }
}

// KMPPI, TILE2: interpolate this sample's control points onto the horizon ONCE, with all its tps threads
// (mppi.py:665-668: W @ theta_k, specific actions, clamp), after the barrier that completes the control-point tile
template <typename real, int NU>
__device__ __forceinline__ void interp_column(const KArgs<real>& a, Smem<real>& sm, unsigned long long kg) {
    typedef Ops<real> O;
    const int LD = sm.LD, S = a.S;
    const int BS = blockDim.x / a.tps, s_ = threadIdx.x % BS, g_ = threadIdx.x / BS;
    const real* col = sm.rows + s_;
    for (int t = g_; t < a.T; t += a.tps) {
#pragma unroll
        for (int n = 0; n < NU; ++n) {
            real acc = O::mul(sm.Ws[t * S], col[n * LD]);
            for (int s = 1; s < S; ++s) acc = O::add(acc, O::mul(sm.Ws[t * S + s], col[(s * NU + n) * LD]));
            override_value<real>(a, kg, t * NU + n, acc);
            sm.rows2[(t * NU + n) * LD + s_] = clamp<real>(acc, a.nm.u_min[n], a.nm.u_max[n]);
        }
    }
}

// perturbed action at step t for this thread (KMPPI interpolates the control points: mppi.py:665-668)
template <typename real, int VARIANT, int NU, bool TILE2 = false>
__device__ __forceinline__ void action_at(const KArgs<real>& a, const Smem<real>& sm, unsigned long long kg, int t, real* v) {
    typedef Ops<real> O;
    const int LD = sm.LD;
    const real* col = sm.rows + (threadIdx.x % (blockDim.x / a.tps));
    if (VARIANT == V_KMPPI && TILE2) {
        const real* col2 = sm.rows2 + (threadIdx.x % (blockDim.x / a.tps));
#pragma unroll
        for (int n = 0; n < NU; ++n) v[n] = col2[(t * NU + n) * LD];
    } else if (VARIANT == V_KMPPI) {
        const int S = a.S;
#pragma unroll
        for (int n = 0; n < NU; ++n) {
            real acc = O::mul(sm.Ws[t * S], col[n * LD]);
            for (int s = 1; s < S; ++s) acc = O::add(acc, O::mul(sm.Ws[t * S + s], col[(s * NU + n) * LD]));
            override_value<real>(a, kg, t * NU + n, acc);
            v[n] = clamp<real>(acc, a.nm.u_min[n], a.nm.u_max[n]);
        }
    } else {
#pragma unroll
        for (int n = 0; n < NU; ++n) v[n] = col[(t * NU + n) * LD];
    }
}

// effective noise entering the action cost at step t (mppi.py:385 / :552 / :670)
template <typename real, int VARIANT, int NU, bool TILE2 = false>
__device__ __forceinline__ void noise_at(const KArgs<real>& a, const Smem<real>& sm, int t, const real* v, real* eps) {
    typedef Ops<real> O;
#pragma unroll
    for (int n = 0; n < NU; ++n) {
        if (VARIANT == V_SMPPI && TILE2)
            eps[n] = sm.rows2[(t * NU + n) * sm.LD + (threadIdx.x % (blockDim.x / a.tps))];
        else if (VARIANT == V_SMPPI)
            eps[n] = O::sub(O::div(O::sub(v[n], sm.As[t * NU + n]), a.nm.delta_t), sm.Us[t * NU + n]);
        else
            eps[n] = O::sub(v[n], sm.Us[t * NU + n]);
    }
}

// the weighted quantity for row j given the stored tile value (the thing the softmin averages)
template <typename real, int VARIANT>
__device__ __forceinline__ real eps_of(const NoiseModel<real>& nm, real val, real us, real as_or_ths) {
    typedef Ops<real> O;
    if (VARIANT == V_MPPI) return O::sub(val, us);                                          // mppi.py:385
    if (VARIANT == V_SMPPI) return O::sub(O::div(O::sub(val, as_or_ths), nm.delta_t), us);  // mppi.py:552
    return O::sub(val, as_or_ths);                                                          // mppi.py:664
}

// ---- flagged 8-byte words (payload32 | flag32): peer mailboxes, the local record mailbox, host delivery ----------
// (the record layout of a mailbox: xchg_publish_words below)
// relaxed.sys, not volatile: the words are self-validating, so nothing orders one against another — and ptxas completes
// every volatile access before it issues the next (a thread polling 8 words paid 8 L2 round trips per sweep; the same
// serialisation made a 32-record combine from shared memory cost 1.5 us)
__device__ __forceinline__ void st_peer(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_poll(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// value i of the action as flagged 8-byte word(s) in pinned host memory (float: 1 word, double: 2)
template <typename real>
__device__ __forceinline__ void host_store(unsigned long long* box, int i, real v, unsigned long long epoch);
template <>
__device__ __forceinline__ void host_store<float>(unsigned long long* box, int i, float v, unsigned long long epoch) {
    st_peer(box + i, ((epoch & 0xffffffffull) << 32) | (unsigned long long)__float_as_uint(v));
}
template <>
__device__ __forceinline__ void host_store<double>(unsigned long long* box, int i, double v, unsigned long long epoch) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    st_peer(box + 2 * i, ((epoch & 0xffffffffull) << 32) | (bits & 0xffffffffull));
    st_peer(box + 2 * i + 1, ((epoch & 0xffffffffull) << 32) | (bits >> 32));
}

// ---- final update from (beta, eta, numerators) with the post-shift nominal in shared memory -----
template <typename real, int VARIANT>
__device__ void finish_update(const KArgs<real>& a, const double* numd, const real* Us, const real* As, real* ths,
                              const real* Ws, int nu) {
    typedef Ops<real> O;
    const int tid = threadIdx.x, BD = blockDim.x;
    const int TN = a.TN, R = a.R;
    const double eta = numd[1];
    const double inv_eta = 1.0 / eta;
    // nominal_used: U | A | theta slots, as sampled from (post-shift, pre-update)
    for (int j = tid; j < TN; j += BD) {
        a.nominal_used[j] = Us[j];
        if (VARIANT == V_SMPPI) a.nominal_used[TN + j] = As[j];
    }
    if (VARIANT == V_KMPPI)
        for (int j = tid; j < R; j += BD) a.nominal_used[2 * TN + j] = ths[j];
    if (tid == 0) {
        a.stats[0] = numd[0];
        a.stats[1] = eta;
        if (a.offset_dev != nullptr && blockIdx.y == 0) *a.offset_dev += a.offset_inc;   // every sampler of this command is done
    }
    // Host delivery: each action value goes out as self-validating 8-byte words (payload32 | epoch32), so
    // the host sees a value as soon as its own store lands — no system-wide fence, no separate flag.
    unsigned long long* hact = a.host_mailbox;
    if (VARIANT == V_MPPI) {
        for (int j = tid; j < TN; j += BD) {
            const real un = O::add(Us[j], (real)(numd[2 + j] * inv_eta));                // mppi.py:270
            a.U[j] = un;
            if (j < a.upc * nu) {                                                          // mppi.py:271-275
                a.action_out[j] = un;
                if (hact != nullptr) host_store<real>(hact, j, un, a.host_epoch);
            }
        }
    } else if (VARIANT == V_SMPPI) {
        for (int j = tid; j < TN; j += BD) {
            const real un = O::add(Us[j], (real)(numd[2 + j] * inv_eta));                // mppi.py:529
            const real an = O::add(As[j], O::mul(un, a.nm.delta_t));                       // mppi.py:531
            a.U[j] = un;
            a.A[j] = an;
            if (j < a.upc * nu) {                                                          // mppi.py:533-537
                a.action_out[j] = an;
                if (hact != nullptr) host_store<real>(hact, j, an, a.host_epoch);
            }
        }
    } else {
        __syncthreads();
        for (int j = tid; j < R; j += BD) {
            const real tn = O::add(ths[j], (real)(numd[2 + j] * inv_eta));              // mppi.py:681
            ths[j] = tn;
            a.theta[j] = tn;
        }
        __syncthreads();
        const int S = a.S;
        for (int j = tid; j < TN; j += BD) {                                               // mppi.py:682  U = W theta
            const int t = j / nu, n = j - t * nu;
            real acc = O::mul(Ws[t * S], ths[n]);
            for (int s = 1; s < S; ++s) acc = O::add(acc, O::mul(Ws[t * S + s], ths[s * nu + n]));
            a.U[j] = acc;
            if (j < a.upc * nu) {
                a.action_out[j] = acc;
                if (hact != nullptr) host_store<real>(hact, j, acc, a.host_epoch);
            }
        }
    }
}

// =================================================================================================
// Warp-fold tail: the softmin reduction of every command kernel (fused, resident, tcgen05 and the stepped route's
// softmin_update_kernel) — no CTA-wide barriers in the fold, a thread-block-cluster stage through distributed shared
// memory (fused / resident kernels), and a finisher that works on a handful of records.
//
//   per tile   each ROLLOUT WARP folds its 32 samples into its own running record (beta_w, eta_w, V_w[R]) — shuffles
//              only, fp64 accumulation, record in shared memory (warp-private: no barrier)
//   per CTA    the warp records go to the cluster LEADER's shared memory (st.shared::cluster), one cluster barrier
//   leader     combines cluster_size x warps records into ONE cluster record and publishes it: to the L2 workspace
//              (ticket among the leaders — 16 atomics instead of 128 at BASELINE config 2), or, on a sharded controller
//              in direct mode, straight into every peer GPU's mailbox over NVLink
//   finisher   (last leader) combines the n_clusters (x world) records and writes the update
// Every combination is in fixed record order and fp64, so the result does not depend on scheduling and is bit-identical
// on all ranks of a sharded controller.   Reference lines: mppi.py:254-259, 268-270 (and the SMPPI / KMPPI forms).
// =================================================================================================
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ void st_dsmem_f64(uint32_t addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

#define MPPI_XCHG_PARITY_WORDS 65536       // 8-byte words per epoch parity of a peer mailbox (mppi_xchg_bytes = 2 x this x 8)

// doubles of the finisher's staging area: every record it polls (LL mode: xw x npub cluster records; sharded rank-record
// mode: one per rank); a single GPU in ticket mode stages nothing
__host__ __device__ inline int fused_xstage_doubles(bool sharded, int world, int npub, int R) {
    const int xw = sharded ? world : 1;
    return (npub > 1 || sharded) ? xw * npub * (R + 2) : 0;
}

// the `nb` argument of make_layout for the warp-fold tail: the records combine_records reads from the L2 workspace
// (ticket mode: the grid's NC cluster records), 1 when they arrive as flagged words (LL mode) or there is one cluster
__host__ __device__ inline int fused_layout_nb(int NC, int npub) { return (NC > 1 && npub != NC) ? NC : 1; }

// this CTA's running warp records: (beta = +inf, eta = 0, V = 0); call before the first barrier of the kernel
template <typename real>
__device__ __forceinline__ void warp_records_init(const KArgs<real>& a, Smem<real>& sm) {
    const int RW = a.R + 2, n = (blockDim.x / a.tps >> 5) * RW;
    for (int i = threadIdx.x; i < n; i += blockDim.x) sm.wrec[i] = (i % RW == 0) ? (double)INFINITY : 0.0;
}

// ---- per tile: fold this warp's 32 samples into its running record (rollout warps only; warp-synchronous) ----------
// Where the weighted quantity of row j comes from:
enum {
    FOLD_ROWS = 0,    // eps_of(rows): the tile holds the perturbed actions / control points
    FOLD_ROWS2 = 1,   // rows2 holds the effective noise (SMPPI with TILE2: written once by transform_column)
    FOLD_EPS = 2      // rows holds eps itself (softmin_update_kernel: the materialised noise)
};
template <typename real, int VARIANT, int SRC>
__device__ __forceinline__ void warp_fold(const KArgs<real>& a, Smem<real>& sm, real c_tot, bool active, int nvalid) {
    typedef Ops<real> O;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int R = a.R, LD = sm.LD, i0 = w * 32;
    double* rec = sm.wrec + (size_t)w * (R + 2);
    const real nfl = a.nm.neg_inv_lambda;
    // the fused kernels: the 32 columns this warp reads below were written by its own lanes (one sample per thread: no
    // CTA barrier in between) — order them.  (Kernels whose tile is written by other warps put a CTA barrier first.)
    __syncwarp();
    const real cmin = warp_min<real>(active ? c_tot : O::inf());
    const real beta_run = (real)rec[0];                 // a value of type `real`, kept in a double slot
    const real beta_new = cmin < beta_run ? cmin : beta_run;
    if (beta_new == O::inf()) return;                   // warp-uniform: no sample of this warp has a cost yet
    const real wgt = active ? O::exp_(nfl * (c_tot - beta_new)) : (real)0;                       // mppi.py:12-13, 256
    const double resc = (beta_run == O::inf()) ? 0.0 : (double)O::exp_(nfl * (beta_run - beta_new));
    const double eta_tile = (double)warp_sum<real>(wgt);
    const int nv = min(32, nvalid - i0);
    for (int jb = 0; jb < R; jb += 32) {
        const int j = jb + lane;
        const bool jv = j < R;
        const int jc = jv ? j : 0;
        const real us = (VARIANT == V_KMPPI || SRC != FOLD_ROWS) ? (real)0 : sm.Us[jc];
        const real a2 = SRC != FOLD_ROWS ? (real)0 : (VARIANT == V_SMPPI ? sm.As[jc] : (VARIANT == V_KMPPI ? sm.ths[jc] : (real)0));
        const real* row = (SRC == FOLD_ROWS2 ? sm.rows2 : sm.rows) + (size_t)jc * LD + i0;
        // the 32 products of a warp are added in the controller's precision (as the reference's einsum does, in its own
        // order); everything ACROSS warps, CTAs and GPUs is fp64 (measured: an fp64 inner sum costs the large-K
        // geometry, where every warp folds, 5 us per command through F2F.F64 / DADD issue)
        real acc = (real)0;
        for (int i = 0; i < nv; ++i) {
            const real wi = __shfl_sync(0xffffffffu, wgt, i);
            const real e = SRC == FOLD_ROWS ? eps_of<real, VARIANT>(a.nm, row[i], us, a2) : row[i];
            acc += wi * e;                                                                      // mppi.py:268
        }
        if (jv) rec[2 + j] = rec[2 + j] * resc + (double)acc;
    }
    __syncwarp();                    // every lane has read the running record
    if (lane == 0) {
        rec[0] = (double)beta_new;
        rec[1] = rec[1] * resc + eta_tile;
    }
    __syncwarp();
}

// ---- fixed-order fp64 combination of records (beta_q, eta_q, V_q[R]) -----------------------------------------------
//   beta = min beta_q ; s_q = exp(nfl (beta_q - beta)) ; eta = sum s_q eta_q ; V[j] = sum s_q V_q[j]   -> numd[0 .. R+2)
// CTA-wide (every thread calls it; three barriers).  Record q is recs[q * (R+2) ..] in shared or global memory (generic
// pointer, volatile loads: L2 for global).  Threads are (group g = tid / W, column jl = tid % W; W = 64, or 32 in a CTA of
// one warp, so that every group is complete): group g adds the records q = g, g + nG, ... for its columns (column 0 = eta, column 1 + j = V[j]) into part2[g][..], the groups are added
// in order — the result does not depend on timing.  Deliberately SMALL and out of line (one copy for every call site):
// the tail runs once per command on a cold instruction cache, where instruction count, not arithmetic, sets its time
// (ncu: `no_instruction` is the third-largest stall of the kernel).
template <typename real>
__device__ __noinline__ void combine_records(const double* recs, int nrec, int R, double nfl, double* part2, double* sq,
                                             double* numd) {
    typedef Ops<real> O;
    const int RW = R + 2, C = R + 1;                      // columns: eta, V[0..R)
    const int BD = blockDim.x, lw = BD < 64 ? 5 : 6, W = 1 << lw;
    const int tid = threadIdx.x, nG = BD >> lw, g = tid >> lw, jl = tid & (W - 1), nw = BD >> 5;
    // beta: ONE load per thread (record tid; more only for grids above blockDim records), warp minima through sq[]
    const double b_mine = tid < nrec ? recs[(size_t)tid * RW] : (double)INFINITY;
    double b = b_mine;
    for (int q = tid + BD; q < nrec; q += BD) b = fmin(b, recs[(size_t)q * RW]);
    b = warp_min<double>(b);
    if ((tid & 31) == 0) part2[tid >> 5] = b;
    __syncthreads();
    double beta = part2[0];
    for (int w = 1; w < nw; ++w) beta = fmin(beta, part2[w]);
    // the rescale factors in the controller's precision (exact for equal betas; beta_q - beta is exact in fp64); an empty
    // record weighs 0
    if (tid < nrec) sq[tid] = b_mine == (double)INFINITY ? 0.0 : (double)O::exp_((real)(nfl * (b_mine - beta)));
    for (int q = tid + BD; q < nrec; q += BD) {
        const double bq = recs[(size_t)q * RW];
        sq[q] = bq == (double)INFINITY ? 0.0 : (double)O::exp_((real)(nfl * (bq - beta)));
    }
    __syncthreads();
    if (tid == 0) numd[0] = beta;
    // the loads of a batch are issued together, THEN used: written as `acc += sq[q] * recs[..]` in one loop, ptxas keeps
    // every volatile load next to its DFMA and a thread waits one L2 round trip per record (K = 131072: 293 records in
    // the L2 workspace, 42 per thread — 9 us; batched: 6 round trips)
    constexpr int UB = 8;
    for (int j = jl; j < C; j += W) {
        double acc = 0.0;
        const double* col = recs + 1 + j;
        for (int q0 = g; q0 < nrec; q0 += nG * UB) {
            double v[UB];
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int q = q0 + u * nG;
                v[u] = q < nrec ? col[(unsigned)(q * RW)] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int q = q0 + u * nG;
                if (q < nrec) acc += sq[q] * v[u];
            }
        }
        part2[g * C + j] = acc;
    }
    __syncthreads();
    for (int j = tid; j < C; j += BD) {
        double t = part2[j];
        for (int w = 1; w < nG; ++w) t += part2[(size_t)w * C + j];
        numd[1 + j] = t;
    }
    __syncthreads();
}

// ---- the same combination for records in the L2 workspace (ticket mode: grids of hundreds of CTAs) ---------------------
// ld.global.cg loads (L2; no SM of this launch has the lines in L1), UB of them in flight per thread before the first is
// used.  The volatile form above leaves one L2 round trip per record on the critical path — at K = 131072 (293 records,
// 42 per thread) that was 9 us of a 47 us command.
template <typename real>
__device__ __noinline__ void combine_global(const double* recs, int nrec, int R, double nfl, double* part2, double* sq, double* numd) {
    typedef Ops<real> O;
    const int RW = R + 2, C = R + 1;
    const int BD = blockDim.x, lw = BD < 64 ? 5 : 6, W = 1 << lw;     // column groups of 64 (32 in a CTA of one warp)
    const int tid = threadIdx.x, nG = BD >> lw, g = tid >> lw, jl = tid & (W - 1), nw = BD >> 5;
    double b = (double)INFINITY;
    for (int q = tid; q < nrec; q += BD) b = fmin(b, __ldcg(recs + (size_t)q * RW));
    b = warp_min<double>(b);
    if ((tid & 31) == 0) part2[tid >> 5] = b;
    __syncthreads();
    double beta = part2[0];
    for (int w = 1; w < nw; ++w) beta = fmin(beta, part2[w]);
    for (int q = tid; q < nrec; q += BD) {
        const double bq = __ldcg(recs + (size_t)q * RW);
        sq[q] = bq == (double)INFINITY ? 0.0 : (double)O::exp_((real)(nfl * (bq - beta)));
    }
    __syncthreads();
    if (tid == 0) numd[0] = beta;
    constexpr int UB = 8;
    for (int j = jl; j < C; j += W) {
        double acc = 0.0;
        const double* col = recs + 1 + j;
        for (int q0 = g; q0 < nrec; q0 += nG * UB) {
            double v[UB];
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int q = q0 + u * nG;
                v[u] = q < nrec ? __ldcg(col + (size_t)q * RW) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                const int q = q0 + u * nG;
                if (q < nrec) acc += sq[q] * v[u];
            }
        }
        part2[g * C + j] = acc;
    }
    __syncthreads();
    for (int j = tid; j < C; j += BD) {
        double t = part2[j];
        for (int w = 1; w < nG; ++w) t += part2[w * C + j];
        numd[1 + j] = t;
    }
    __syncthreads();
}

// ---- the same combination for at most 64 records, WITHOUT CTA barriers or scratch -------------------------------------
// Only the warps that own a column block take part (warp w: columns 32 w + lane, stride 32 P): each computes beta and the
// rescale factors for itself (lane l holds those of records l and l + 32, handed round with shuffles) and adds its columns
// over the records in ascending order (two interleaved chains).  The other warps of the CTA go straight to the one
// barrier at the end.  This is the form the tail uses at every size that matters for latency: 16 warp records per cluster
// and 32 cluster records per GPU at BASELINE config 2 — the barrier-and-scratch form above cost 2.3 + 2.9 us there
// (every warp of the CTA walks its ~600 instructions, contending with the co-resident CTA at large K), this one a fraction.
template <typename real>
__device__ __noinline__ void combine_narrow(const double* recs, int nrec, int R, double nfl, double* numd) {
    typedef Ops<real> O;
    const int RW = R + 2, C = R + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int P = min(nw, (C + 31) >> 5);
    if (warp < P) {
        const double b0 = lane < nrec ? recs[lane * RW] : (double)INFINITY;
        const double b1 = lane + 32 < nrec ? recs[(lane + 32) * RW] : (double)INFINITY;
        const double beta = warp_min<double>(fmin(b0, b1));
        // in the controller's precision (exact for equal betas; beta_q - beta is exact in fp64); an empty record weighs 0
        const double s0 = b0 == (double)INFINITY ? 0.0 : (double)O::exp_((real)(nfl * (b0 - beta)));
        const double s1 = b1 == (double)INFINITY ? 0.0 : (double)O::exp_((real)(nfl * (b1 - beta)));
        for (int jb = warp * 32; jb < C; jb += P * 32) {
            const int j = jb + lane;
            const double* col = recs + 1 + (j < C ? j : 0);
            double acc0 = 0.0, acc1 = 0.0;
            for (int q0 = 0; q0 < nrec; q0 += 4) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = q0 + u < nrec ? col[(q0 + u) * RW] : 0.0;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int q = q0 + u;                       // q >= nrec: that lane's factor is 0 and v is 0
                    const double sq = __shfl_sync(0xffffffffu, q < 32 ? s0 : s1, q & 31);
                    if (u & 1) acc1 += sq * v[u];
                    else acc0 += sq * v[u];
                }
            }
            if (j < C) numd[1 + j] = acc0 + acc1;
        }
        if (threadIdx.x == 0) numd[0] = beta;
    }
    __syncthreads();
}
#define MPPI_COMBINE_NARROW_MAX 64

template <typename real>
__device__ __forceinline__ void combine(Smem<real>& sm, const double* recs, int nrec, int R, double nfl) {
    if (nrec <= MPPI_COMBINE_NARROW_MAX) combine_narrow<real>(recs, nrec, R, nfl, sm.numd);
    else combine_records<real>(recs, nrec, R, nfl, sm.part2, sm.sqd, sm.numd);
}

// ---- record mailboxes: records of (R+2) doubles as LL words (payload32 | flag32), record r at word r * 2 (R+2) ------
// a.peers[g], g < xw, are the mailboxes the record goes to: every rank's (sharded controller, over NVLink) or just this
// GPU's own (single GPU: a region of the workspace) — self-validating words need no fence and no ticket, the finisher
// sees a record one store-to-poll latency after it was written.
static __device__ __noinline__ void xchg_publish_words(unsigned long long* const* peers, int xw, unsigned long long epoch, unsigned int parity_words,
                                                int rec_index, int R, const double* src) {
    const int nwords = 2 * (R + 2);
    const uint32_t flag = (uint32_t)(epoch & 0x7fffffffull) | 0x80000000u;
    const size_t off = (size_t)(epoch & 1ull) * parity_words + (size_t)rec_index * nwords;
    for (int i = threadIdx.x; i < nwords; i += blockDim.x) {
        const unsigned long long bits = (unsigned long long)__double_as_longlong(src[i >> 1]);
        const uint32_t half = (i & 1) ? (uint32_t)(bits >> 32) : (uint32_t)bits;
        const unsigned long long word = ((unsigned long long)flag << 32) | half;
        for (int g = 0; g < xw; ++g) st_peer(peers[g] + off + i, word);
    }
    // (measured and rejected: a system-scope fence after the remote stores, meant to push the posted NVLink writes out
    // sooner, costs 4.5 us per command at two GPUs — 24.2 against 19.7 us back to back)
}
template <typename real>
__device__ __forceinline__ void xchg_publish(const KArgs<real>& a, int xw, int rec_index, const double* src) {
    xchg_publish_words(a.peers, xw, a.epoch, a.xchg_parity_words, rec_index, a.R, src);
}
// all threads of the CTA; nrec records from this rank's own mailbox into sm.xstage (doubles), PB polls in flight per
// thread.  Returns 0, or 1 on timeout.
static __device__ __noinline__ int xchg_collect_words(const unsigned long long* mine, unsigned long long epoch, unsigned long long timeout_ns,
                                               int nwords, uint32_t* dst) {
    constexpr int PB = 8;
    const int BD = blockDim.x;
    const uint32_t flag = (uint32_t)(epoch & 0x7fffffffull) | 0x80000000u;
    __shared__ int s_timeout;
    if (threadIdx.x == 0) s_timeout = 0;
    __syncthreads();
    unsigned long long t0 = 0;
    for (int base = threadIdx.x; base < nwords; base += BD * PB) {
        unsigned int pending = 0;
#pragma unroll
        for (int u = 0; u < PB; ++u)
            if (base + u * BD < nwords) pending |= 1u << u;
        unsigned int spins = 0;
        while (pending) {
            unsigned long long w[PB];
#pragma unroll
            for (int u = 0; u < PB; ++u)
                if (pending & (1u << u)) w[u] = ld_poll(mine + base + u * BD);
#pragma unroll
            for (int u = 0; u < PB; ++u)
                if ((pending & (1u << u)) && (uint32_t)(w[u] >> 32) == flag) {
                    dst[base + u * BD] = (uint32_t)w[u];
                    pending &= ~(1u << u);
                }
            if (pending && (++spins & 255u) == 0) {
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                if (now - t0 > timeout_ns || s_timeout) {
                    s_timeout = 1;
                    break;
                }
            }
        }
    }
    __syncthreads();
    return s_timeout;
}
template <typename real>
__device__ __forceinline__ int xchg_collect(const KArgs<real>& a, Smem<real>& sm, int own, int nrec) {
    return xchg_collect_words(a.peers[own] + (size_t)(a.epoch & 1ull) * a.xchg_parity_words, a.epoch, a.xchg_timeout_ns,
                              nrec * 2 * (a.R + 2), reinterpret_cast<uint32_t*>(sm.xstage));
}

// a peer never delivered: report it (device stats, pinned host word) and return a DEFINED action — the nominal the
// command sampled around, not updated.  This rank's U then lags its peers by one update: the host raises on the next
// command (mppi.py reads the status word), it does not continue silently.
template <typename real, int VARIANT>
__device__ void xchg_timed_out(const KArgs<real>& a, Smem<real>& sm, int nu) {
    const real* nom = VARIANT == V_SMPPI ? sm.As : sm.Us;
    for (int j = threadIdx.x; j < a.upc * nu; j += blockDim.x) {
        a.action_out[j] = nom[j];
        if (a.host_mailbox != nullptr) host_store<real>(a.host_mailbox, j, nom[j], a.host_epoch);
    }
    if (threadIdx.x == 0) {
        a.stats[3] = -6.0;     // MPPI_ERR_TIMEOUT
        if (a.xchg_status_host != nullptr) {
            *reinterpret_cast<volatile long long*>(a.xchg_status_host) = -6;
            __threadfence_system();
        }
        *a.ticket = 0u;
    }
}

// ---- the tail: returns true in the CTA that finished the command --------------------------------------------------
// PERSISTENT (resident kernel): the grid outlives the command, so the non-leader CTAs of a cluster complete the barrier
// phase (arrive + wait) instead of exiting after their arrive.
template <typename real, int VARIANT, int NU, bool PERSISTENT = false>
__device__ bool warp_tail(const KArgs<real>& a, Smem<real>& sm) {
    const int tid = threadIdx.x, BD = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int R = a.R, RW = R + 2;
    const int nrw = (BD / a.tps) >> 5;                       // rollout warps = records per CTA
    const int cs = (int)cluster_nctarank();                  // cluster dims are (cs, 1, 1)
    const int cr = blockIdx.x % cs, cid = blockIdx.x / cs, NC = gridDim.x / cs;
    const double nfl = (double)a.nm.neg_inv_lambda;
    const bool sharded = a.world > 1 && !a.export_partial;
    const int xw = sharded ? a.world : 1;                    // ranks whose records the finisher combines
    const int xr = sharded ? a.rank : 0;                     // this rank's slot among them
    // LL mode: the cluster records go out as flagged words (to this GPU's mailbox, and every peer's on a sharded
    // controller); the leader of cluster 0 polls for all xw x NC of them — no fence, no ticket.  Otherwise (grids whose
    // records do not fit the finisher's staging area): records to the L2 workspace, ticket among the leaders.
    const bool ll = NC > 1 && a.xchg_npub == NC;
    __shared__ int s_is_last;

    // (1) warp records -> the cluster leader's shared memory
    if (cs > 1) {
        if (!PERSISTENT) cluster_wait_acquire();             // phase 0 (arrived at kernel entry): every CTA of the cluster runs
        if (cr != 0 && warp < nrw) {
            const uint32_t dst = mapa_shared(smem_u32(sm.wrec), 0) + (uint32_t)(((cr * nrw + warp) * RW) * 8);
            const double* rec = sm.wrec + (size_t)warp * RW;
            for (int i = lane; i < RW; i += 32) st_dsmem_f64(dst + i * 8, rec[i]);
        }
        cluster_arrive_release();
        if (cr != 0) {
            if (PERSISTENT) cluster_wait_acquire();
            return false;
        }
        cluster_wait_acquire();
    } else {
        __syncthreads();
    }
    stamp(a.dbg, 6);

    // (2) leader: cs x nrw warp records -> one cluster record in sm.numd
    {
        combine<real>(sm, sm.wrec, cs * nrw, R, nfl);
    }
    stamp(a.dbg, 9);
    // (3) publish the cluster record
    if (ll) {
        xchg_publish<real>(a, xw, xr * NC + cid, sm.numd);
        if (cid != 0) return false;                          // the leader of cluster 0 finishes the command
    } else if (NC > 1) {
        for (int i = tid; i < RW; i += BD) a.crec[(size_t)cid * RW + i] = sm.numd[i];
        __syncthreads();        // every thread's stores precede thread 0's release (one MEMBAR per leader)
        if (tid == 0) {
            unsigned int t;
            asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(t) : "l"(a.ticket), "r"(1u) : "memory");
            s_is_last = (t == (unsigned int)NC - 1);
        }
        __syncthreads();
        if (!s_is_last) return false;
        if (tid == 0) *a.ticket = 0u;   // self-reset: the next launch needs no memset
    }
    stamp(a.dbg, 8);

    // (4) finisher: all records -> (beta, eta, numerators) in sm.numd
    if (ll) {
        if (xchg_collect<real>(a, sm, xr, xw * NC)) {
            xchg_timed_out<real, VARIANT>(a, sm, NU);
            return true;
        }
        stamp(a.dbg, 12);
        combine<real>(sm, sm.xstage, xw * NC, R, nfl);
    } else if (NC > 1) {
        combine_global<real>(a.crec, NC, R, nfl, sm.part2, sm.sqd, sm.numd);
    }
    stamp(a.dbg, 10);
    if (a.export_partial) {   // library-collective route: caller all-gathers, mppi_apply_partials finishes
        const int TN = a.TN;
        for (int j = tid; j < RW; j += BD) a.partial_out[j] = sm.numd[j];
        for (int j = tid; j < TN; j += BD) {
            a.nominal_used[j] = sm.Us[j];
            if (VARIANT == V_SMPPI) a.nominal_used[TN + j] = sm.As[j];
        }
        if (VARIANT == V_KMPPI)
            for (int j = tid; j < R; j += BD) a.nominal_used[2 * TN + j] = sm.ths[j];
        if (tid == 0) {
            a.stats[0] = sm.numd[0];
            a.stats[1] = sm.numd[1];
            a.stats[3] = 0.0;
        }
        return true;
    }
    if (sharded && !ll) {
        // rank-record mode: this rank's combined record is its one published record
        xchg_publish<real>(a, xw, xr, sm.numd);
        if (xchg_collect<real>(a, sm, xr, xw)) {
            xchg_timed_out<real, VARIANT>(a, sm, NU);
            return true;
        }
        combine<real>(sm, sm.xstage, xw, R, nfl);
    }
    stamp(a.dbg, 11);
    finish_update<real, VARIANT>(a, sm.numd, sm.Us, sm.As, sm.ths, sm.Ws, NU);
    if (tid == 0) a.stats[3] = 0.0;
    return true;
}

// ---- per-environment view of the kernel arguments (batched launches) -------------------------------
// The argument block lives in constant (parameter) space; a batched CTA needs its environment's
// pointers, so it builds an adjusted copy in shared memory once and every stage reads that copy.
template <typename real, int NXv, int NUv>
__device__ void make_env_args(const KArgs<real>& in, KArgs<real>* out) {
    const int tid = threadIdx.x, BD = blockDim.x;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&in);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out);
    for (int i = tid; i < (int)(sizeof(KArgs<real>) / 4); i += BD) dst[i] = src[i];
    __syncthreads();
    if (tid == 0) {
        const long long e = blockIdx.y;
        const long long K = in.K, TN = in.TN, R = in.R;
        out->U = in.U + e * in.env_u_stride;
        if (in.cost_total) out->cost_total = in.cost_total + e * K;
        if (in.action_out) out->action_out = in.action_out + e * in.upc * NUv;
        if (in.nominal_used) out->nominal_used = in.nominal_used + e * (3 * TN + 4);
        if (in.stats) out->stats = in.stats + e * 4;
        if (in.state_dev) out->state_dev = in.state_dev + e * NXv;
        if (in.ticket) {
            const long long off = e * in.env_ws_stride;
            out->ticket = reinterpret_cast<unsigned int*>(reinterpret_cast<unsigned char*>(in.ticket) + off);
            out->crec = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(in.crec) + off);
            if (in.world == 1 || in.export_partial)      // this GPU's own record mailbox lives in the environment's workspace
                out->peers[0] = reinterpret_cast<unsigned long long*>(reinterpret_cast<unsigned char*>(in.peers[0]) + off);
        }
        if (in.out_pa) out->out_pa = in.out_pa + e * K * TN;
        if (in.out_noise) out->out_noise = in.out_noise + e * K * TN;
        if (in.out_cost_init) out->out_cost_init = in.out_cost_init + e * K;
        if (in.in_cost) out->in_cost = in.in_cost + e * K;
        if (in.in_eps) out->in_eps = in.in_eps + e * K * R;
    }
    __syncthreads();
}

// ---- stage C', split-cost rollout as a function: recurrence on the rollout thread | running costs on all tps
// threads of the sample | ordered sum.  Returns the sample's total cost on its rollout thread (+inf elsewhere) and
// stores it to cost_total[k].  Contains two CTA barriers: every thread must call it.
// Shared by fused_command_kernel<..., SPLIT = true> and the resident kernel (mppi_resident.cuh).
template <class Model, typename real, int VARIANT>
__device__ __forceinline__ real split_cost_rollout(const KArgs<real>& a, const typename Model::template P<real>& mp, Smem<real>& sm,
                                                   int k, unsigned long long kg, bool in_range, bool active) {
    typedef Ops<real> O;
    constexpr int NX = Model::NX, NU = Model::NU;
    const NoiseModel<real>& nm = a.nm;
    const int tid = threadIdx.x, BS = blockDim.x / a.tps, T = a.T;
    real c_tot = O::inf();
    real* xcol = sm.xs + (tid % BS);
    real x[NX];
    real pert = (real)0, smooth = (real)0;
    if (active) {
        if (a.state_dev != nullptr) {
            const real* sp = a.state_dev + (a.state_per_sample ? (size_t)k * NX : 0);
#pragma unroll
            for (int i = 0; i < NX; ++i) x[i] = sp[i];
        } else {
#pragma unroll
            for (int i = 0; i < NX; ++i) x[i] = a.x0[i];
        }
        real vprev[NU];
#pragma unroll
        for (int n = 0; n < NU; ++n) vprev[n] = (real)0;
MPPI_UNROLL_N(MPPI_ROLLOUT_UNROLL)
        for (int t = 0; t < T; ++t) {
            real v[NU], u[NU], eps[NU];
            action_at<real, VARIANT, NU, true>(a, sm, kg, t, v);
            noise_at<real, VARIANT, NU, true>(a, sm, t, v, eps);
#pragma unroll
            for (int n = 0; n < NU; ++n) u[n] = O::mul(nm.u_scale, v[n]);            // mppi.py:313
            Model::template step<real>(mp, x, u);                                     // mppi.py:314
#pragma unroll
            for (int i = 0; i < NX; ++i) xcol[(t * NX + i) * BS] = x[i];
            pert = O::add(pert, action_cost_term<real, NU>(nm, eps, sm.Us + t * NU));
            if (VARIANT == V_SMPPI) {
                if (t > 0) {
#pragma unroll
                    for (int n = 0; n < NU; ++n) {
                        const real d = O::mul(nm.u_scale, O::sub(v[n], vprev[n]));    // mppi.py:559
                        smooth = O::add(smooth, O::mul(d, d));
                    }
                }
#pragma unroll
                for (int n = 0; n < NU; ++n) vprev[n] = v[n];
            }
        }
    }
    __syncthreads();
    if (in_range) {
MPPI_UNROLL_N(2)
        for (int t = tid / BS; t < T; t += a.tps) {      // independent across t: two in flight per thread
            real v[NU], u[NU], xt[NX];
            action_at<real, VARIANT, NU, true>(a, sm, kg, t, v);
#pragma unroll
            for (int n = 0; n < NU; ++n) u[n] = O::mul(nm.u_scale, v[n]);
#pragma unroll
            for (int i = 0; i < NX; ++i) xt[i] = xcol[(t * NX + i) * BS];
            xcol[(t * NX) * BS] = Model::template cost<real>(mp, xt, u);              // mppi.py:318
        }
    }
    __syncthreads();
    if (active) {
        real roll = (real)0;
        for (int t = 0; t < T; ++t) roll = O::add(roll, xcol[(t * NX) * BS]);         // mppi.py:319, t = 0..T-1
        if (Model::template has_terminal<real>(mp)) roll = O::add(roll, Model::template terminal<real>(mp, x));
        c_tot = O::add(roll, pert);                                                   // mppi.py:416
        if (VARIANT == V_SMPPI) c_tot = O::add(c_tot, O::mul(smooth, nm.w_smooth));   // mppi.py:562,569
        a.cost_total[k] = c_tot;
    }
    return c_tot;
}

// =================================================================================================
// The fused command kernel
// =================================================================================================
// SPLIT (threads_per_sample > 1 only, i.e. problems too small to fill the machine): the rollout is the one
// phase a sample's helper threads cannot share — the state recurrence is serial.  But only the DYNAMICS are:
// the running cost of step t depends on x_t alone.  So the rollout thread runs the bare recurrence and parks
// every x_t in shared memory (xs[T*NX][BS]); then all tps threads of the sample evaluate the T running costs
// in parallel (in place: cost_t overwrites x_t[0]); then the rollout thread adds them up in the reference's
// order t = 0..T-1.  Same operations, same rounding, same summation order as the fused loop — the single
// resident warp just stops carrying the cost's ~45 instructions per step on its critical path.
//
// MINB: minimum resident CTAs per SM promised to ptxas.  The split-cost kernels (one CTA per SM by construction) get 1: the
// whole register file.  The single-loop kernels of the analytic models get 2 = a 64-register cap (20 B of spill): the
// two-CTA-per-SM geometry of large K needs it, and without the promise the out-of-line tail functions push ptxas to 128
// registers and one CTA per SM (measured at K = 131072: 42 -> 53 us).  The MLP's step keeps 64 activations live: it gets
// the whole register file (one CTA per SM) — under the cap it spilled 340 B per thread.
template <class Model> struct FusedMinBlocks { static constexpr int value = MPPI_FUSED_MIN_BLOCKS; };
template <> struct FusedMinBlocks<PendulumMLPModel> { static constexpr int value = 1; };

template <class Model, typename real, int VARIANT, bool BATCHED, bool SPLIT = false, int MINB = (SPLIT ? 1 : FusedMinBlocks<Model>::value)>
__global__ void __launch_bounds__(512, MINB) fused_command_kernel(const __grid_constant__ KArgs<real> a_in,
                                                            const __grid_constant__ typename Model::template P<real> mp) {
    typedef Ops<real> O;
    constexpr int NX = Model::NX, NU = Model::NU;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, BD = blockDim.x;
    __shared__ __align__(16) unsigned char a_env_raw[BATCHED ? sizeof(KArgs<real>) : 16];
    if (BATCHED) make_env_args<real, NX, NU>(a_in, reinterpret_cast<KArgs<real>*>(a_env_raw));
    const KArgs<real>& a = BATCHED ? *reinterpret_cast<const KArgs<real>*>(a_env_raw) : a_in;
    const int BS = BD / a.tps;
    const int xst = fused_xstage_doubles(a.world > 1 && !a.export_partial, a.world, a.xchg_npub, a.R);
    const int cs_ = (int)cluster_nctarank(), NC_ = (int)gridDim.x / cs_;
    const SmemLayout L = make_layout<real>(VARIANT, a.T, NU, a.S, a.R, BD, BS, fused_layout_nb(NC_, a.xchg_npub),
                                           layout_extra(VARIANT != V_MPPI, SPLIT ? NX : 0, cs_, xst));
    Smem<real> sm(smem, L);
    const NoiseModel<real>& nm = a.nm;
    const int T = a.T;
    warp_records_init<real>(a, sm);      // published by the barrier in stage_issue
    // phase 0 of the cluster barrier: "this CTA has started" — the tail waits for it before the first store into the
    // leader's shared memory (distributed shared memory may only be touched once its CTA is known to be running)
    if (cs_ > 1) cluster_arrive_relaxed();

    stamp(a.dbg, 0);
    // Programmatic dependent launch: this grid may be resident while the previous kernel on the stream is
    // still finishing.  Let our own successor start early too, draw the first tile's normals (pure
    // compute into shared memory), and only then wait for the predecessor's memory to be visible.
    const bool early_fill = a.pdl && a.z == nullptr && a.z_out == nullptr && blockIdx.x < a.n_tiles;
    if (a.pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (early_fill) {
        const int k0 = blockIdx.x * BS + (tid % BS);
        fill_normals<real>(a, sm, blockIdx.x, k0 < a.K, (unsigned long long)(a.k_offset + k0), min(BS, a.K - blockIdx.x * BS));
    }
    if (a.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
    stage_issue<real, VARIANT, NU>(a, sm);
    stamp(a.dbg, 1);
    bool staged = false;

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int k = tile * BS + (tid % BS);
        const bool in_range = k < a.K;
        const bool active = in_range && tid < BS;      // the rollout thread of sample k
        const int nvalid = min(BS, a.K - tile * BS);
        const unsigned long long kg = (unsigned long long)(a.k_offset + k);

        if (!(early_fill && tile == blockIdx.x)) fill_normals<real>(a, sm, tile, in_range, kg, nvalid);
        if (!staged) {   // the nominal sequence is first needed now; its TMA copy flew during the draws
            stage_finish<real, VARIANT, NU>(a, sm);
            staged = true;
        } else if (a.tps > 1) {
            __syncthreads();
        }
        if (tile == blockIdx.x) stamp(a.dbg, 2);
        if (in_range) transform_column<real, VARIANT, NU, true>(a, sm, kg);
        if (a.tps > 1) __syncthreads();
        if (VARIANT == V_KMPPI) {      // the control points of the sample are complete: interpolate them onto the horizon
            if (in_range) interp_column<real, NU>(a, sm, kg);
            if (a.tps > 1) __syncthreads();
        }
        if (tile == blockIdx.x) stamp(a.dbg, 3);

        real c_tot = O::inf();
        if constexpr (SPLIT) {
            // C'. split rollout: recurrence (rollout thread) | running costs (all tps threads) | ordered sum
            c_tot = split_cost_rollout<Model, real, VARIANT>(a, mp, sm, k, kg, in_range, active);
        } else if (active) {

            // C. rollout (mppi.py:297-332) + action cost (mppi.py:409,415) [+ smoothness :559-562]
            real x[NX];
            if (a.state_dev != nullptr) {
                const real* sp = a.state_dev + (a.state_per_sample ? (size_t)k * NX : 0);
#pragma unroll
                for (int i = 0; i < NX; ++i) x[i] = sp[i];
            } else {
#pragma unroll
                for (int i = 0; i < NX; ++i) x[i] = a.x0[i];
            }
            // Software-pipelined T-loop: the running cost of the state reached at step t-1 and the
            // dynamics of step t both depend only on x_t, so issuing them back to back gives the
            // single resident warp two independent dependency chains.  The arithmetic and the
            // order of every accumulation are exactly the reference's (cost summed t = 0..T-1).
            real roll = (real)0, pert = (real)0, smooth = (real)0;
            real vprev[NU], uprev[NU];
#pragma unroll
            for (int n = 0; n < NU; ++n) { vprev[n] = (real)0; uprev[n] = (real)0; }
MPPI_UNROLL_N(MPPI_ROLLOUT_UNROLL)
            for (int t = 0; t < T; ++t) {
                real v[NU], u[NU], eps[NU], xs[NX];
                action_at<real, VARIANT, NU, true>(a, sm, kg, t, v);
                noise_at<real, VARIANT, NU, true>(a, sm, t, v, eps);
#pragma unroll
                for (int n = 0; n < NU; ++n) u[n] = O::mul(nm.u_scale, v[n]);            // mppi.py:313
#pragma unroll
                for (int i = 0; i < NX; ++i) xs[i] = x[i];
#if MPPI_ROLLOUT_PIPELINED
                Model::template step<real>(mp, x, u);                                     // mppi.py:314
                if (t > 0) roll = O::add(roll, Model::template cost<real>(mp, xs, uprev));   // mppi.py:318-319 (step t-1)
#else
                Model::template step<real>(mp, x, u);                                     // mppi.py:314
                roll = O::add(roll, Model::template cost<real>(mp, x, u));                // mppi.py:318-319
#endif
                pert = O::add(pert, action_cost_term<real, NU>(nm, eps, sm.Us + t * NU));
                if (VARIANT == V_SMPPI) {
                    if (t > 0) {
#pragma unroll
                        for (int n = 0; n < NU; ++n) {
                            const real d = O::mul(nm.u_scale, O::sub(v[n], vprev[n]));    // mppi.py:559
                            smooth = O::add(smooth, O::mul(d, d));
                        }
                    }
#pragma unroll
                    for (int n = 0; n < NU; ++n) vprev[n] = v[n];
                }
#pragma unroll
                for (int n = 0; n < NU; ++n) uprev[n] = u[n];
            }
#if MPPI_ROLLOUT_PIPELINED
            roll = O::add(roll, Model::template cost<real>(mp, x, uprev));                // step T-1
#endif
            if (Model::template has_terminal<real>(mp)) roll = O::add(roll, Model::template terminal<real>(mp, x));
            c_tot = O::add(roll, pert);                                                   // mppi.py:416
            if (VARIANT == V_SMPPI) c_tot = O::add(c_tot, O::mul(smooth, nm.w_smooth));   // mppi.py:562,569
            a.cost_total[k] = c_tot;
        }
        if (tile == blockIdx.x) stamp(a.dbg, 4);
        // D. every rollout warp folds its 32 samples into its own running record (no CTA barrier)
        if (tid < BS) warp_fold<real, VARIANT, VARIANT == V_SMPPI ? FOLD_ROWS2 : FOLD_ROWS>(a, sm, c_tot, active, nvalid);
        if (tile == blockIdx.x) stamp(a.dbg, 5);
        if (tile + (int)gridDim.x < a.n_tiles) __syncthreads();      // the tile is refilled by the next pass
    }
    if (!staged) stage_finish<real, VARIANT, NU>(a, sm);
    warp_tail<real, VARIANT, NU>(a, sm);
    stamp(a.dbg, 7);
}

// =================================================================================================
// Generic path, part 1: sample + perturb with coalesced write-out (mppi.py:375-385, 409, 415;
// SMPPI :539-562; KMPPI :657-670).  Also used to materialise noise/perturbed_action lazily.
// =================================================================================================
template <typename real, int VARIANT, int NU>
__global__ void __launch_bounds__(512) sample_kernel(const __grid_constant__ KArgs<real> a_in) {
    typedef Ops<real> O;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, BD = blockDim.x;
    __shared__ __align__(16) unsigned char a_env_raw[sizeof(KArgs<real>)];
    if (a_in.n_env > 1) make_env_args<real, 0, NU>(a_in, reinterpret_cast<KArgs<real>*>(a_env_raw));
    const KArgs<real>& a = a_in.n_env > 1 ? *reinterpret_cast<const KArgs<real>*>(a_env_raw) : a_in;
    const int BS = BD / a.tps;
    const SmemLayout L = make_layout<real>(VARIANT, a.T, NU, a.S, a.R, BD, BS, 1, VARIANT == V_KMPPI);
    Smem<real> sm(smem, L);
    const NoiseModel<real>& nm = a.nm;
    const int T = a.T, R = a.R, TN = a.TN, LD = sm.LD;

    stage_nominal<real, VARIANT, NU>(a, sm);
    if (blockIdx.x == 0 && a.nominal_used != nullptr) {
        for (int j = tid; j < TN; j += BD) {
            a.nominal_used[j] = sm.Us[j];
            if (VARIANT == V_SMPPI) a.nominal_used[TN + j] = sm.As[j];
        }
        if (VARIANT == V_KMPPI)
            for (int j = tid; j < R; j += BD) a.nominal_used[2 * TN + j] = sm.ths[j];
    }

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int k = tile * BS + (tid % BS);
        const bool in_range = k < a.K;
        const bool active = in_range && tid < BS;
        const int nvalid = min(BS, a.K - tile * BS);
        const unsigned long long kg = (unsigned long long)(a.k_offset + k);
        fill_normals<real>(a, sm, tile, in_range, kg, nvalid);
        if (a.tps > 1) __syncthreads();
        if (in_range) transform_column<real, VARIANT, NU>(a, sm, kg);
        if (a.tps > 1) __syncthreads();
        if (active) {
            real pert = (real)0, smooth = (real)0;
            real vprev[NU];
#pragma unroll
            for (int n = 0; n < NU; ++n) vprev[n] = (real)0;
            for (int t = 0; t < T; ++t) {
                real v[NU], eps[NU];
                action_at<real, VARIANT, NU>(a, sm, kg, t, v);
                noise_at<real, VARIANT, NU>(a, sm, t, v, eps);
                pert = O::add(pert, action_cost_term<real, NU>(nm, eps, sm.Us + t * NU));
                if (VARIANT == V_KMPPI) {
#pragma unroll
                    for (int n = 0; n < NU; ++n) sm.rows2[(t * NU + n) * LD + tid] = v[n];
                }
                if (VARIANT == V_SMPPI) {
                    if (t > 0) {
#pragma unroll
                        for (int n = 0; n < NU; ++n) {
                            const real d = O::mul(nm.u_scale, O::sub(v[n], vprev[n]));
                            smooth = O::add(smooth, O::mul(d, d));
                        }
                    }
#pragma unroll
                    for (int n = 0; n < NU; ++n) vprev[n] = v[n];
                }
            }
            if (a.out_cost_init != nullptr) {
                real c0 = pert;
                if (VARIANT == V_SMPPI) c0 = O::add(c0, O::mul(smooth, nm.w_smooth));
                a.out_cost_init[k] = c0;
            }
        }
        __syncthreads();
        // coalesced write-out of the tile: (K,T,nu) row-major == [sample][j]
        {
            const real* vt = (VARIANT == V_KMPPI) ? sm.rows2 : sm.rows;
            const size_t base = (size_t)tile * BS * TN;
            const int count = nvalid * TN;
            for (int e = tid; e < count; e += BD) {
                const int s = e / TN, j = e - s * TN;
                const real val = vt[j * LD + s];
                if (a.out_pa != nullptr) a.out_pa[base + e] = val;
                if (a.out_noise != nullptr) {
                    real ep;
                    if (VARIANT == V_SMPPI) ep = O::sub(O::div(O::sub(val, sm.As[j]), nm.delta_t), sm.Us[j]);
                    else ep = O::sub(val, sm.Us[j]);
                    a.out_noise[base + e] = ep;
                }
            }
            if (VARIANT == V_KMPPI && a.out_noise_theta != nullptr) {
                const size_t base2 = (size_t)tile * BS * R;
                const int count2 = nvalid * R;
                for (int e = tid; e < count2; e += BD) {
                    const int s = e / R, j = e - s * R;
                    a.out_noise_theta[base2 + e] = O::sub(sm.rows[j * LD + s], sm.ths[j]);
                }
            }
        }
        __syncthreads();
    }
}

// states along the rollout of given perturbed actions (mppi.py:307-322), for registered models.
// pa_stride = elements between consecutive samples' action sequences: T*nu for a (K,T,nu) tensor, 0 when every
// sample replays the SAME (T,nu) sequence (get_rollouts, mppi.py:425-448).
template <class Model, typename real>
__global__ void states_kernel(const real* __restrict__ pa, real* __restrict__ states, const KArgs<real> a,
                              const typename Model::template P<real> mp, long long pa_stride) {
    typedef Ops<real> O;
    constexpr int NX = Model::NX, NU = Model::NU;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.K) return;
    pa += (size_t)k * (size_t)pa_stride;
    real x[NX];
    if (a.state_dev != nullptr) {
        const real* sp = a.state_dev + (a.state_per_sample ? (size_t)k * NX : 0);
        for (int i = 0; i < NX; ++i) x[i] = sp[i];
    } else {
        for (int i = 0; i < NX; ++i) x[i] = a.x0[i];
    }
    for (int t = 0; t < a.T; ++t) {
        real u[NU];
        for (int n = 0; n < NU; ++n) u[n] = O::mul(a.nm.u_scale, pa[t * NU + n]);                 // mppi.py:313 / :445
        Model::template step<real>(mp, x, u);
        for (int i = 0; i < NX; ++i) states[((size_t)k * a.T + t) * NX + i] = x[i];
    }
}

// =================================================================================================
// Generic path, part 2: softmin + weighted update from materialised cost_total (K) and eps (K,R)
// (mppi.py:254-259, 268-270).  HBM-bound: reads 4*K*(R+1) bytes once, coalesced.  The rollout warps fold the tile with
// warp_fold, and the command finishes in warp_tail without a cluster: the grid's CTA records combine through the ticket
// (one record per rank, exchanged with the peers, on a sharded controller).  Never LL mode: the launch may be captured
// into a CUDA graph, whose replays would repeat an LL record's per-command tag.
// (512, 1): without the minimum ptxas squeezes some instantiations to 64 registers and spills in the tail.
// =================================================================================================
template <typename real, int VARIANT, int NU>
__global__ void __launch_bounds__(512, 1) softmin_update_kernel(const __grid_constant__ KArgs<real> a_in) {
    typedef Ops<real> O;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, BD = blockDim.x;
    __shared__ __align__(16) unsigned char a_env_raw[sizeof(KArgs<real>)];
    if (a_in.n_env > 1) make_env_args<real, 0, NU>(a_in, reinterpret_cast<KArgs<real>*>(a_env_raw));
    const KArgs<real>& a = a_in.n_env > 1 ? *reinterpret_cast<const KArgs<real>*>(a_env_raw) : a_in;
    const int BS = BD / a.tps;
    const SmemLayout L = make_layout<real>(VARIANT, a.T, NU, a.S, a.R, BD, BS, fused_layout_nb((int)gridDim.x, 1),
                                           layout_extra(0, 0, 1, fused_xstage_doubles(a.world > 1 && !a.export_partial, a.world, 1, a.R)));
    Smem<real> sm(smem, L);
    const int R = a.R, TN = a.TN, LD = sm.LD;
    warp_records_init<real>(a, sm);
    // post-shift nominal comes from nominal_used (written by sample_kernel)
    for (int j = tid; j < TN; j += BD) {
        sm.Us[j] = a.nominal_used[j];
        if (VARIANT == V_SMPPI) sm.As[j] = a.nominal_used[TN + j];
    }
    if (VARIANT == V_KMPPI) {
        for (int j = tid; j < R; j += BD) sm.ths[j] = a.nominal_used[2 * TN + j];
        for (int j = tid; j < a.T * a.S; j += BD) sm.Ws[j] = a.W[j];
    }
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int k = tile * BS + tid;
        const bool active = tid < BS && k < a.K;
        const int nvalid = min(BS, a.K - tile * BS);
        const size_t base = (size_t)tile * BS * R;
        const int count = nvalid * R;
        for (int e = tid; e < count; e += BD) {
            const int s = e / R, j = e - s * R;
            sm.rows[j * LD + s] = a.in_eps[base + e];
        }
        const real c = active ? a.in_cost[k] : O::inf();
        __syncthreads();                                              // the tile was loaded by every warp
        if (tid < BS) warp_fold<real, VARIANT, FOLD_EPS>(a, sm, c, active, nvalid);
        if (tile + (int)gridDim.x < a.n_tiles) __syncthreads();      // the tile is refilled by the next pass
    }
    warp_tail<real, VARIANT, NU>(a, sm);
}

// omega_k = exp(-(c_k - beta)/lambda) / eta from the stats a command left behind (mppi.py:256-258)
template <typename real>
__global__ void omega_kernel(const real* __restrict__ cost, real* __restrict__ omega, const double* __restrict__ stats,
                             real neg_inv_lambda, int K) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const real beta = (real)stats[0];
    const real inv_eta = (real)(1.0 / stats[1]);
    omega[k] = inv_eta * Ops<real>::exp_(neg_inv_lambda * (cost[k] - beta));
}

// cost[m,k] += c[m,k]  (mppi.py:319 / 363); M>1: var_acc[k] += var_m(c[:,k]) * discount (mppi.py:364)
template <typename real>
__global__ void cost_accumulate_kernel(real* __restrict__ cost, const real* __restrict__ c, real* __restrict__ var_acc,
                                       int M, int K, real discount) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    real mean = (real)0;
    for (int m = 0; m < M; ++m) {
        const real v = c[(size_t)m * K + k];
        cost[(size_t)m * K + k] += v;
        mean += v;
    }
    if (var_acc != nullptr && M > 1) {
        mean /= (real)M;
        real ss = (real)0;
        for (int m = 0; m < M; ++m) {
            const real d = c[(size_t)m * K + k] - mean;
            ss += d * d;
        }
        var_acc[k] += ss / (real)(M - 1) * discount;
    }
}

// ---- finish from all-gathered partials (library-collective route) --------------------------------
template <typename real, int VARIANT>
__global__ void apply_partials_kernel(const KArgs<real> a, const double* partials, int nu) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, BD = blockDim.x;
    const int TN = a.TN, R = a.R, T = a.T, S = a.S;
    real* Us = reinterpret_cast<real*>(smem);
    real* As = Us + TN;
    real* ths = As + TN;
    real* Ws = ths + R;
    double* numd = reinterpret_cast<double*>(smem + align_up((2 * TN + R + T * S) * (int)sizeof(real), 16));
    for (int j = tid; j < TN; j += BD) {
        Us[j] = a.nominal_used[j];
        As[j] = (VARIANT == V_SMPPI) ? a.nominal_used[TN + j] : (real)0;
    }
    if (VARIANT == V_KMPPI) {
        for (int j = tid; j < R; j += BD) ths[j] = a.nominal_used[2 * TN + j];
        for (int j = tid; j < T * S; j += BD) Ws[j] = a.W[j];
    }
    const double nfl = (double)a.nm.neg_inv_lambda;
    double beta = partials[0];
    for (int g = 1; g < a.world; ++g) beta = fmin(beta, partials[(size_t)g * (R + 2)]);
    for (int j = tid; j < R + 1; j += BD) {
        double acc = 0.0;
        for (int g = 0; g < a.world; ++g) {
            const double* rec = partials + (size_t)g * (R + 2);
            acc += exp(nfl * (rec[0] - beta)) * rec[1 + j];
        }
        numd[1 + j] = acc;
    }
    if (tid == 0) numd[0] = beta;
    __syncthreads();
    finish_update<real, VARIANT>(a, numd, Us, As, ths, Ws, nu);
    if (tid == 0) a.stats[3] = 0.0;
}

#endif  // __CUDACC__

}  // namespace mppi
