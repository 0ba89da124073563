// mppi_resident.cuh — the resident command kernel: command() without a kernel launch.
//
// A host control loop that calls command() at 10-50 kHz (mppi.py:240-252 once per control step) pays, on the
// launch route, ~12 us of launch + completion latency around a ~15 us kernel (DESIGN.md §4.4).  Here the kernel
// stays resident: one cooperative launch puts the command's grid on the SMs, and every following command is a
// RECORD the host writes into pinned memory (flags, Philox counter, start state — self-validating 8-byte words,
// payload32 | seq32) and an ACTION the finishing CTA writes back the same way.  Per command:
//
//   host  : write record seq+1 -> spin on the action words
//   CTA 0 : warp 0 polls the record over PCIe, re-publishes it on a device-memory board
//   all   : warp 0 of every CTA polls the board (L2), decodes it into the CTA's shared-memory argument block
//   all   : split-cost rollout -> softmin fold -> ticket; the last CTA combines, updates U, stores the action to
//           the host, fences, and publishes `done = seq+1` (device board + host status word)
//
// Everything that does not depend on the start state is done BEFORE the record arrives, overlapped with the
// host's turnaround: as soon as `done` says the previous update of U is visible, every CTA draws the next
// command's normals (the Philox counter advances by a known increment), stages + shifts U and builds the
// perturbed-action tile, predicting that the next command repeats the last one's shift flag.  A record that
// contradicts the prediction (other counter, other shift flag) just redoes that preparation — same results.
//
// Arithmetic: the stages are the functions of mppi_fused.cuh (fill_normals, stage_finish, transform_column,
// split_cost_rollout, warp_fold, warp_tail — launched with the same cluster size), so a resident command is bit-identical to a launched one
// with the same (state, seed, counter, flags) — tests/test_gpu_resident.py.
//
// Safety: the kernel cannot outlive its usefulness.  CTA 0 exits after `idle_ns` without a record (it tells the
// board, so every CTA leaves, and writes an exit word the host sees: the next command simply relaunches); every
// other spin loop carries the same clock check with a margin.  Launched cooperatively, so all CTAs are resident or
// the launch fails.  One tile per CTA (the small-problem geometry the split-cost rollout serves).
//
// Single-GPU controllers only (a sharded controller's ranks would each need their own host record in lock-step; the
// launch route with its in-kernel NVLink exchange serves them).
//
// Reference lines replaced: the same as fused_command_kernel (mppi.py:232-275, 297-417 and the SMPPI / KMPPI forms).
#pragma once

#include "mppi_fused.cuh"

namespace mppi {

#define MPPI_RES_MAX_WORDS 32             // command record: 3 + nx (f32) or 3 + 2 nx (f64) words
#define MPPI_RES_BOARD_DONE 64            // board[64] = seq of the last finished command
#define MPPI_RES_BOARD_WORDS 128
#define MPPI_RES_CMD_SHIFT 1u
#define MPPI_RES_CMD_STOP 2u

struct ResidentArgs {
    const unsigned long long* host_cmd;   // pinned host memory: the command record
    unsigned long long* host_status;      // pinned host memory: [0] = seq of the last finished command, [1] = exit word
    unsigned long long* board;            // device memory, MPPI_RES_BOARD_WORDS words, zeroed before every launch
    unsigned long long seq_start;         // commands up to here are done; the kernel waits for seq_start + 1
    unsigned long long offset_pred;       // Philox counter the next command is expected to carry
    unsigned long long idle_ns;           // leave after this long without a record
    unsigned long long epoch_off;         // record-mailbox epoch of command seq = epoch_off + seq (continues the plan's epochs)
    unsigned int gen;                     // launch generation, echoed in the exit word
    int shift_pred;                       // shift flag the next command is expected to carry
    int n_words;                          // words per record
};

#if defined(__CUDACC__)

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// nominal sequence(s) into shared memory with L2 loads: another SM rewrote them during this kernel's life, so the
// (incoherent) L1 must not serve them.  Replaces stage_issue's staging; stage_finish then builds the shifted copy.
template <typename real, int VARIANT>
__device__ void stage_resident(const KArgs<real>& a, Smem<real>& sm) {
    const int tid = threadIdx.x, BD = blockDim.x;
    const int T = a.T, S = a.S, R = a.R, TN = a.TN;
    for (int j = tid; j < TN; j += BD) {
        sm.Uraw[j] = __ldcg(a.U + j);
        if (VARIANT == V_SMPPI) sm.Araw[j] = __ldcg(a.A + j);
    }
    if (VARIANT == V_KMPPI) {
        for (int j = tid; j < R; j += BD) sm.thraw[j] = __ldcg(a.theta + j);
        for (int j = tid; j < T * S; j += BD) sm.Ws[j] = a.W[j];            // constants of the controller
        if (a.shift)
            for (int j = tid; j < S * S; j += BD) sm.Wsh[j] = a.Wshift[j];
    }
}

// everything of a command that does not need the start state: normals, shifted nominal, perturbed-action tile
template <typename real, int VARIANT, int NU>
__device__ __forceinline__ void resident_prepare(const KArgs<real>& a, Smem<real>& sm, bool in_range, unsigned long long kg, int nvalid) {
    warp_records_init<real>(a, sm);                  // this command's softmin records (published by the barriers below)
    fill_normals<real>(a, sm, blockIdx.x, in_range, kg, nvalid);
    stage_resident<real, VARIANT>(a, sm);
    stage_finish<real, VARIANT, NU>(a, sm);          // tma_ok == 0: barrier, shifted copy, barrier
    if (in_range) transform_column<real, VARIANT, NU, true>(a, sm, kg);
    __syncthreads();
    if (VARIANT == V_KMPPI) {
        if (in_range) interp_column<real, NU>(a, sm, kg);
        __syncthreads();
    }
}

// __launch_bounds__(640, 1): CTAs have at most 512 threads; promising 640 makes ptxas stop at 96 registers
// (65,536 / 640), so a resident 512-thread CTA leaves a quarter of its SM's register file to the kernels other
// streams launch meanwhile (torch ops reading U or cost_total) instead of taking all of it at 128.
//
// STAMPS = true (one debug instantiation: pendulum, fp32, MPPI; chosen when the plan carries debug_clocks): %globaltimer
// stamps of the last command's phases per CTA, slots of the (grid, 16) debug_clocks array:
//   14 previous update visible | 0 prepared, polling | 13 (CTA 0) record seen in host memory | 1 record seen by this CTA |
//   2 decoded | 3 rolled out | 4 folded | 6 ticket taken | 8, 10, 11 finisher: partials acquired, eta, numerators |
//   12 finisher: action stored, fence done, done word written.   scripts/resident_timeline.py reads them.
template <class Model, typename real, int VARIANT, bool STAMPS = false>
__global__ void __launch_bounds__(640, 1) resident_command_kernel(const __grid_constant__ KArgs<real> a_in,
                                                                  const __grid_constant__ typename Model::template P<real> mp,
                                                                  const __grid_constant__ ResidentArgs ra) {
    typedef Ops<real> O;
    constexpr int NX = Model::NX, NU = Model::NU;
    constexpr int WPV = sizeof(real) / 4;             // record words per state value
    static_assert(5 + 2 * MPPI_MAX_NX <= MPPI_RES_MAX_WORDS, "command record does not fit one warp");
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ __align__(16) unsigned char a_raw[sizeof(KArgs<real>)];
    __shared__ unsigned int s_cmd[MPPI_RES_MAX_WORDS];
    __shared__ int s_stop;
    const int tid = threadIdx.x, BD = blockDim.x, lane = tid & 31, warp = tid >> 5;

    // the argument block lives in shared memory: thread 0 rewrites its per-command fields
    KArgs<real>& a = *reinterpret_cast<KArgs<real>*>(a_raw);
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&a_in);
        uint32_t* dst = reinterpret_cast<uint32_t*>(a_raw);
        for (int i = tid; i < (int)(sizeof(KArgs<real>) / 4); i += BD) dst[i] = src[i];
        __syncthreads();
        if (tid == 0) {
            a.tma_ok = 0;          // nominal staged with L2 loads (stage_resident)
            a.pdl = 0;
            a.z = nullptr;
            a.z_out = nullptr;
            if (!STAMPS) a.dbg = nullptr;
            a.offset_dev = nullptr;
            a.state_dev = nullptr;
            a.world = 1;
            a.export_partial = 0;
            a.offset = ra.offset_pred;
            a.shift = ra.shift_pred;
        }
        __syncthreads();
    }
    const int BS = BD / a.tps;
    const int cs_ = (int)cluster_nctarank();
    const SmemLayout L = make_layout<real>(VARIANT, a.T, NU, a.S, a.R, BD, BS, fused_layout_nb((int)gridDim.x / cs_, a.xchg_npub),
                                           layout_extra(VARIANT != V_MPPI, NX, cs_, fused_xstage_doubles(false, 1, a.xchg_npub, a.R)));
    Smem<real> sm(smem, L);
    // distributed shared memory may only be touched once its CTA is known to be running: one cluster barrier at entry
    if (cs_ > 1) {
        cluster_arrive_relaxed();
        cluster_wait_acquire();
    }

    // one tile per CTA
    const int k = blockIdx.x * BS + (tid % BS);
    const bool in_range = k < a.K;
    const bool active = in_range && tid < BS;
    const int nvalid = min(BS, a.K - blockIdx.x * BS);
    const unsigned long long kg = (unsigned long long)(a.k_offset + k);

    unsigned long long seq = ra.seq_start;
    unsigned long long offset_pred = ra.offset_pred;
    int shift_pred = ra.shift_pred;
    unsigned long long t_idle0 = global_ns();
    const unsigned long long slack_ns = 2000000000ull;   // non-polling CTAs give CTA 0 this much more before leaving
    int exit_reason = 0;

    for (;;) {
        // (1) the previous command's update of U / A / theta must be visible before it is staged again
        if (seq != ra.seq_start) {
            if (tid == 0) {
                const unsigned long long* done = ra.board + MPPI_RES_BOARD_DONE;
                int lost = 0;
                while (ld_poll(done) != seq) {
                    if (global_ns() - t_idle0 > ra.idle_ns + slack_ns) { lost = 1; break; }
                }
                __threadfence();       // acquire side of the finisher's fence
                s_stop = lost;
            }
            __syncthreads();
            if (s_stop) { exit_reason = 3; break; }
        }
        if constexpr (STAMPS) stamp(a.dbg, 14);

        // (2) state-independent work, on the predicted counter / shift flag
        resident_prepare<real, VARIANT, NU>(a, sm, in_range, kg, nvalid);
        if constexpr (STAMPS) stamp(a.dbg, 0);

        // (3) the record of command seq + 1
        const unsigned int want = (unsigned int)((seq + 1) & 0xffffffffull);
        if (warp == 0) {
            const int nw = ra.n_words;
            const unsigned long long* src = blockIdx.x == 0 ? ra.host_cmd : ra.board;
            const unsigned long long limit = blockIdx.x == 0 ? ra.idle_ns : ra.idle_ns + slack_ns;
            unsigned int payload = 0;
            int timed_out = 0;
            for (;;) {
                const unsigned long long v = lane < nw ? ld_poll(src + lane) : ((unsigned long long)want << 32);
                const bool ok = (unsigned int)(v >> 32) == want;
                if (__all_sync(0xffffffffu, ok)) {
                    payload = (unsigned int)v;
                    break;
                }
                if (lane == 0 && global_ns() - t_idle0 > limit) timed_out = 1;
                timed_out = __shfl_sync(0xffffffffu, timed_out, 0);
                if (timed_out) break;
            }
            if (timed_out) payload = lane == 0 ? MPPI_RES_CMD_STOP : 0u;
            if constexpr (STAMPS) {
                if (!timed_out && !(payload & MPPI_RES_CMD_STOP)) stamp(a.dbg, blockIdx.x == 0 ? 13 : 1);   // lane 0 == thread 0
            }
            if (blockIdx.x == 0 && lane < nw) st_peer(ra.board + lane, ((unsigned long long)want << 32) | payload);
            if (lane < nw) s_cmd[lane] = payload;
            if (lane == 0) s_stop = timed_out ? 1 : ((payload & MPPI_RES_CMD_STOP) ? 2 : 0);
        }
        __syncthreads();
        if (s_stop) { exit_reason = s_stop; break; }
        t_idle0 = global_ns();       // every thread restarts its idle clock at the record's arrival

        // (4) decode; redo the preparation if the record is not the predicted one
        const int shift = (s_cmd[0] & MPPI_RES_CMD_SHIFT) ? 1 : 0;
        const unsigned long long offset = (unsigned long long)s_cmd[1] | ((unsigned long long)s_cmd[2] << 32);
        if (tid == 0) {
            a.offset = offset;
            a.shift = shift;
            a.host_epoch = seq + 1;
            a.epoch = ra.epoch_off + seq + 1;
            uint32_t* x0w = reinterpret_cast<uint32_t*>(a.x0);
            for (int i = 0; i < NX * WPV; ++i) x0w[i] = s_cmd[3 + i];
        }
        __syncthreads();
        if (offset != offset_pred || shift != shift_pred) resident_prepare<real, VARIANT, NU>(a, sm, in_range, kg, nvalid);
        if constexpr (STAMPS) stamp(a.dbg, 2);

        // (5) rollout, fold, tail — the launched kernel's stages
        const real c_tot = split_cost_rollout<Model, real, VARIANT>(a, mp, sm, k, kg, in_range, active);
        if constexpr (STAMPS) stamp(a.dbg, 3);
        if (tid < BS) warp_fold<real, VARIANT, VARIANT == V_SMPPI ? FOLD_ROWS2 : FOLD_ROWS>(a, sm, c_tot, active, nvalid);
        if constexpr (STAMPS) stamp(a.dbg, 4);
        const bool finisher = warp_tail<real, VARIANT, NU, true>(a, sm);
        if (finisher) {
            __syncthreads();           // every store of the update precedes thread 0's fence
            if (tid == 0) {
                __threadfence_system();
                st_peer(ra.board + MPPI_RES_BOARD_DONE, seq + 1);
                st_peer(ra.host_status, seq + 1);
                if constexpr (STAMPS) stamp(a.dbg, 12);
            }
        }
        ++seq;
        offset_pred = offset + a_in.offset_inc;
        shift_pred = shift;
        __syncthreads();               // thread 0 rewrites the argument block at the top of the next pass
        if (tid == 0) {
            a.offset = offset_pred;
            a.shift = shift_pred;
        }
        __syncthreads();
    }
    if (blockIdx.x == 0 && tid == 0) st_peer(ra.host_status + 1, ((unsigned long long)ra.gen << 32) | (unsigned long long)exit_reason);
}

#endif  // __CUDACC__

}  // namespace mppi
