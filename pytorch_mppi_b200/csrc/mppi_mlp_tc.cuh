// mppi_mlp_tc.cuh — tensor-core variant of the fused command kernel for the learned pendulum model
// (BASELINE config 4: 3-32-32-2 tanh residual MLP, /root/reference/tests/pendulum_approximate.py:47-67).
//
// The network's three layers are genuine dense contractions, so per rollout step a CTA of 128 samples (= the 128 TMEM
// lanes of one M=128 UMMA tile) runs them on the 5th-gen tensor cores:
//   registers -> bf16 operand tile in shared memory (canonical K-major, no swizzle)
//   tcgen05.mma.cta_group::1.kind::f16  (one elected thread)  -> fp32 accumulators in TMEM
//   tcgen05.commit -> mbarrier -> tcgen05.ld of the thread's own row (lane = sample) -> tanh -> next operand row
// three times per step.  Everything else (sampling, clamp, cost, the warp-fold softmin and its tail) is the
// code of mppi_fused.cuh.
//
// Round 2: a step is a serial chain of three MMA round trips (7,090 clocks per step measured at BASELINE config 4, the
// tensor pipe itself 7 % busy), so the kernel shortens the chain instead of widening the MMAs:
//   * TWO threads per sample (256-thread CTAs): warps w and w+4 own the same 32 TMEM lanes and split the 32 hidden
//     units — 16 tanh + 16 packs each instead of 32 (`tcgen05.ld.32x32b.x16` on their half of the columns);
//   * layer 1 (3 inputs -> 32 units, 96 FMAs per sample) runs on the FP32 pipe, in exact fp32, straight from the state in
//     shared memory: TWO MMA round trips per step instead of three (measured per step and layer: 416 clocks to issue the
//     K-steps + commit, 170-400 to the mbarrier, 150 for the TMEM load — profiles/r02_tc_phase_clocks_v2.txt);
//   * the running cost of the state a step produced is evaluated one step LATER, in the shadow of the layer-2 MMA
//     (same values, same summation order);
//   * tanh = FMUL, MUFU.EX2, FADD, MUFU.RCP, FFMA (mppi_math.cuh).
// Tried and dropped: four independent TMEM accumulators per layer (chains of two dependent MMAs instead of seven) —
// 5 % slower: the MMA chain is not what the round trip waits for.
//
// Precision: operands are bf16.  In the default (SPLIT) mode activations and weights are split into hi + lo
// bf16 parts and each layer is issued as  a_hi*w_hi + a_lo*w_hi + a_hi*w_lo  ("3 x bf16": the a_hi chunks are
// read twice, against the w_hi and the w_lo tile), which costs almost nothing here (the step is latency-bound;
// the extra K-steps are a few more MMA issues) and brings the layer outputs to ~2^-16 relative accuracy
// instead of bf16's 2^-8.  The biases ride along as two extra K columns (constant 1 x [b_hi, b_lo]).
// Measured on B200 (K=32768, T=30): 112 us per command against 160 us for the FFMA kernel at the same
// tolerance; "bf16" mode with MUFU.TANH: 74 us.
#pragma once

#include <cuda_bf16.h>
#include "mppi_fused.cuh"

namespace mppi {

#if defined(__CUDACC__)

namespace tc {

constexpr int H = 32;             // hidden width
constexpr int KX3 = 64;           // SPLIT: activations of layers 2 and 3 are stored as [a_hi(32) | a_lo(32)]
constexpr int CH = 128;           // bytes of one 8-row x 16-byte core matrix
constexpr int TMEM_COLS = 64;     // D2: columns [0,32), D3: [32,48)

// shared-memory operand tiles (bytes); canonical K-major/no-swizzle: core (row group g, k-chunk c) at
// g*SBO + c*LBO, rows 16 B apart inside a core, LBO = 128 B (adjacent chunks), SBO = chunks*128 B
constexpr int B1_BYTES = 32 * 16 * 2;

__device__ __forceinline__ uint64_t smem_desc(const void* base, int sbo_bytes) {
    // SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout none
    const uint64_t addr = (uint64_t)(smem_u32(base) >> 4) & 0x3FFF;
    const uint64_t lbo = (uint64_t)(CH >> 4) & 0x3FFF;
    const uint64_t sbo = (uint64_t)(sbo_bytes >> 4) & 0x3FFF;
    return addr | (lbo << 16) | (sbo << 32) | (1ull << 46);
}
// InstrDescriptor: c=F32 (1<<4) | a=BF16 (1<<7) | b=BF16 (1<<10) | K-major both | N>>3 at [17,23) | M>>4 at [24,29)
__device__ __forceinline__ constexpr uint32_t instr_desc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// one thread of a CONVERGED warp (elect.sync).  The MMA issue must be guarded by this, not by `tid == 0`: ptxas wraps every
// tcgen05 instruction it cannot prove single-threaded in an ELECT / BRA.U.ANY loop (~80 clocks per MMA, measured)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mma_commit(void* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// bounded mbarrier wait: a wedged MMA becomes a trap (kernel error), never a hung GPU
__device__ __forceinline__ void mbar_wait_bounded(void* bar, uint32_t phase) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
        if (!done && clock64() - t0 > 2000000000ll) __trap();
    }
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld2_nowait(uint32_t taddr, float& v0, float& v1) {
    uint32_t r0, r1;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr) : "memory");
    v0 = __uint_as_float(r0);
    v1 = __uint_as_float(r1);
}
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, float& v0, float& v1) {
    uint32_t r0, r1;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    v0 = __uint_as_float(r0);
    v1 = __uint_as_float(r1);
}

__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}
// two floats -> packed bf16 pair (a in the low half): one cvt.rn.bf16x2.f32
__device__ __forceinline__ uint32_t cvt2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
// element (row, k) of a canonical K-major tile with `chunks` k-chunks: byte offset
__device__ __forceinline__ int tile_off(int row, int k, int chunks) {
    return (row >> 3) * (chunks * CH) + (k >> 3) * CH + (row & 7) * 16 + (k & 7) * 2;
}

// this thread's 32 activations -> its row of the operand tile.
//   SPLIT: [hi(32) | lo(32)] with lo = bf16(h - hi);   else [bf16(h)]
template <int SPLIT, int CHUNKS> __device__ __forceinline__ void write_a_row(unsigned char* A, int row, const float* h) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        hi[i] = cvt2(h[2 * i], h[2 * i + 1]);
        if (SPLIT) {
            const float r0 = h[2 * i] - __uint_as_float(hi[i] << 16);
            const float r1 = h[2 * i + 1] - __uint_as_float(hi[i] & 0xFFFF0000u);
            lo[i] = cvt2(r0, r1);
        }
    }
    unsigned char* base = A + (row >> 3) * (CHUNKS * CH) + (row & 7) * 16;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        *reinterpret_cast<uint4*>(base + c * CH) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
        if (SPLIT) *reinterpret_cast<uint4*>(base + (4 + c) * CH) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    }
}

// 16 of a thread-pair's 32 activations -> its two chunks of the operand row (half = 0: hidden units 0..15, 1: 16..31)
template <int SPLIT, int CHUNKS> __device__ __forceinline__ void write_a_half(unsigned char* A, int row, int half, const float* h) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        hi[i] = cvt2(h[2 * i], h[2 * i + 1]);
        if (SPLIT) {
            const float r0 = h[2 * i] - __uint_as_float(hi[i] << 16);
            const float r1 = h[2 * i + 1] - __uint_as_float(hi[i] & 0xFFFF0000u);
            lo[i] = cvt2(r0, r1);
        }
    }
    unsigned char* base = A + (row >> 3) * (CHUNKS * CH) + (row & 7) * 16;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        *reinterpret_cast<uint4*>(base + (2 * half + c) * CH) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
        if (SPLIT) *reinterpret_cast<uint4*>(base + (4 + 2 * half + c) * CH) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
    }
}

}  // namespace tc

// =================================================================================================
template <int VARIANT, int SPLIT, int FAST>
__global__ void __launch_bounds__(256, 2) mlp_tc_command_kernel(const __grid_constant__ KArgs<float> a,
                                                             const __grid_constant__ PendulumMLPModel::P<float> mp) {
    typedef float real;
    typedef Ops<real> O;
    typedef PendulumMLPModel Model;
    constexpr int NX = 2, NU = 1, H = tc::H;
    // K of layers 2 and 3: the activations (split or not) plus one 16-wide K-step whose columns 9 and 10 are the
    // constant 1: the matching rows of B hold bias_hi and bias_lo, so the MMA adds the bias for free
    constexpr int KB = SPLIT ? tc::KX3 : H;
    constexpr int KX = KB + 16;
    constexpr int CHUNKS = KX / 8, NSTEP = KX / 16;
    constexpr int TMEM_COLS = tc::TMEM_COLS, C2 = 0, C3 = 32;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ __align__(128) unsigned char sA2[128 * KX * 2];                 // operand tile of layers 2 and 3
    __shared__ __align__(128) unsigned char sB2[32 * KX * 2];
    __shared__ __align__(128) unsigned char sB3[16 * KX * 2];
    __shared__ __align__(128) unsigned char sB2lo[SPLIT ? 32 * H * 2 : 128];    // w_lo tiles (K = 32), SPLIT only
    __shared__ __align__(128) unsigned char sB3lo[SPLIT ? 16 * H * 2 : 128];
    __shared__ __align__(16) float sX[128 * 4];                                 // (x0, x1, clamped u) of every sample: layer 1's input
    __shared__ __align__(8) unsigned long long s_mma_bar;
    __shared__ uint32_t s_tmem_base;
    const int tid = threadIdx.x, BD = blockDim.x;      // BD == 256: thread = (sample row tid % 128, half tid / 128)
    const int warp = tid >> 5;
    const int row = tid & 127, half = tid >> 7;
    const SmemLayout L = make_layout<real>(VARIANT, a.T, NU, a.S, a.R, BD, BD / a.tps, fused_layout_nb((int)gridDim.x, 1),
                                           layout_extra(0, 0, 1, fused_xstage_doubles(a.world > 1 && !a.export_partial, a.world, 1, a.R)));
    Smem<real> sm(smem, L);
    warp_records_init<real>(a, sm);      // published by the setup barrier below
    const NoiseModel<real>& nm = a.nm;
    const int T = a.T;
    if (a.dbg != nullptr && tid == 32) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        a.dbg[(size_t)blockIdx.x * 16 + 12] = gt;
    }
    // prologue / epilogue wall-clock stamps of thread 32 go to a second block of rows (gridDim.x + blockIdx.x): the debug
    // buffer scripts/tc_phase_clocks.py hands in has 2 x grid rows
#define TC_STAMP(slot)                                                               \
    if (a.dbg != nullptr && tid == 32) {                                             \
        unsigned long long gt_;                                                      \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                      \
        a.dbg[((size_t)gridDim.x + blockIdx.x) * 16 + (slot)] = gt_;                 \
    }

    // ---- one-time setup: TMEM, MMA barrier, bf16 weight tiles (hi/lo split, K-extended) -----------------
    // The weights are kernel parameters (constant bank), cold in this SM's constant cache at every launch: the tile build
    // below walked them with one dependent miss after another (the setup took 5-6 us of a 100 us command).  Every thread
    // now requests its words first — all lines in flight while TMEM is allocated and the tiles are zeroed — and parks
    // them in shared memory, which the tile build reads.
    constexpr int NPW = (int)(sizeof(PendulumMLPModel::P<float>) / 4);
    __shared__ __align__(16) float sP[NPW];
    float pw_reg[(NPW + 255) / 256];
    {
        const float* pw = reinterpret_cast<const float*>(&mp);
#pragma unroll
        for (int i = 0; i < (NPW + 255) / 256; ++i) pw_reg[i] = tid + i * 256 < NPW ? pw[tid + i * 256] : 0.0f;
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)),
                     "r"((uint32_t)TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&s_mma_bar)), "r"(1u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 128 * KX * 2 / 4; i += BD) reinterpret_cast<uint32_t*>(sA2)[i] = 0u;
    for (int i = tid; i < 32 * KX * 2 / 4; i += BD) reinterpret_cast<uint32_t*>(sB2)[i] = 0u;
    for (int i = tid; i < 16 * KX * 2 / 4; i += BD) reinterpret_cast<uint32_t*>(sB3)[i] = 0u;
    if (SPLIT)
        for (int i = tid; i < 16 * H * 2 / 4; i += BD) reinterpret_cast<uint32_t*>(sB3lo)[i] = 0u;
#pragma unroll
    for (int i = 0; i < (NPW + 255) / 256; ++i)
        if (tid + i * 256 < NPW) sP[tid + i * 256] = pw_reg[i];
    __syncthreads();
    const PendulumMLPModel::P<float>& ms = *reinterpret_cast<const PendulumMLPModel::P<float>*>(sP);
    // the bias K-step of the operand tile: columns KB+9, KB+10 are the constant 1 in every row (written once)
    for (int r = tid; r < 128; r += BD) {
        __nv_bfloat16* A = reinterpret_cast<__nv_bfloat16*>(sA2);
        A[tc::tile_off(r, KB + 9, CHUNKS) / 2] = __float2bfloat16_rn(1.0f);
        A[tc::tile_off(r, KB + 10, CHUNKS) / 2] = __float2bfloat16_rn(1.0f);
    }
    for (int n = tid; n < H; n += BD) {
        __nv_bfloat16 bh, bl;
        __nv_bfloat16* B = reinterpret_cast<__nv_bfloat16*>(sB2);
        tc::split_bf16(ms.b2[n], bh, bl);
        B[tc::tile_off(n, KB + 9, CHUNKS) / 2] = bh;
        B[tc::tile_off(n, KB + 10, CHUNKS) / 2] = bl;
        if (n < 2) {
            B = reinterpret_cast<__nv_bfloat16*>(sB3);
            tc::split_bf16(ms.b3[n], bh, bl);
            B[tc::tile_off(n, KB + 9, CHUNKS) / 2] = bh;
            B[tc::tile_off(n, KB + 10, CHUNKS) / 2] = bl;
        }
    }
    // B2 (N=32 x K).  SPLIT: the product  a_hi*w_hi + a_lo*w_hi + a_hi*w_lo  is issued as
    //   [a_hi | a_lo | 1 1] x [w_hi ; w_hi ; b_hi b_lo]   (the main tile, K = 80)
    // + [a_hi]              x [w_lo]                      (the same a_hi chunks against the w_lo tile, K = 32)
    // non-SPLIT: [bf16(a) | 1 1] x [bf16(w) ; b_hi b_lo].
    for (int e = tid; e < H * H; e += BD) {
        const int n = e / H, k = e - n * H;
        __nv_bfloat16 wh, wl;
        tc::split_bf16(ms.W2[k * H + n], wh, wl);                 // W2t[k][n] = W2[n][k]
        __nv_bfloat16* B = reinterpret_cast<__nv_bfloat16*>(sB2);
        B[tc::tile_off(n, k, CHUNKS) / 2] = wh;
        if (SPLIT) {
            B[tc::tile_off(n, 32 + k, CHUNKS) / 2] = wh;
            reinterpret_cast<__nv_bfloat16*>(sB2lo)[tc::tile_off(n, k, 4) / 2] = wl;
        }
    }
    // B3 (N=16 x K): rows 0,1 hold the output layer, rows 2..15 stay zero
    for (int e = tid; e < 2 * H; e += BD) {
        const int n = e / H, k = e - n * H;
        __nv_bfloat16 wh, wl;
        tc::split_bf16(ms.W3[n * H + k], wh, wl);
        __nv_bfloat16* B = reinterpret_cast<__nv_bfloat16*>(sB3);
        B[tc::tile_off(n, k, CHUNKS) / 2] = wh;
        if (SPLIT) {
            B[tc::tile_off(n, 32 + k, CHUNKS) / 2] = wh;
            reinterpret_cast<__nv_bfloat16*>(sB3lo)[tc::tile_off(n, k, 4) / 2] = wl;
        }
    }
    tc::fence_async_smem();
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    TC_STAMP(0)     // TMEM allocated, weight tiles built
    const uint32_t tmem = s_tmem_base;
    const uint32_t my_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);   // warps w and w+4 own TMEM lanes 32 (w % 4) ..: lane = sample row
    uint32_t mma_phase = 0;
    const uint64_t dA2 = tc::smem_desc(sA2, CHUNKS * tc::CH), dB2 = tc::smem_desc(sB2, CHUNKS * tc::CH),
                   dB3 = tc::smem_desc(sB3, CHUNKS * tc::CH);
    const uint64_t dB2lo = tc::smem_desc(sB2lo, 4 * tc::CH), dB3lo = tc::smem_desc(sB3lo, 4 * tc::CH);
    constexpr uint32_t I32 = tc::instr_desc(128, 32), I16 = tc::instr_desc(128, 16);
    constexpr uint64_t KSTEP = (2 * tc::CH) >> 4;                     // one K=16 step = two 8-element chunks, in 16-byte units
    // layer 1 on the FP32 pipe: this thread's 16 hidden units (W1 is stored transposed, W1t[c][unit])
    const int hb = 16 * half;

    stage_issue<real, VARIANT, NU>(a, sm);
    bool staged = false;

    // Tile = 128 samples; the two threads of a sample share its draws and its colour/clamp pass (a.tps == 2), thread 0
    // of the pair (half 0, warps 0-3) carries the state and the cost.
    const int BS = BD / a.tps;
    const bool roller = half == 0;                     // warp-uniform
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int k = tile * BS + (tid % BS);
        const bool in_range = k < a.K;
        const bool active = in_range && roller;
        const int nvalid = min(BS, a.K - tile * BS);
        const unsigned long long kg = (unsigned long long)(a.k_offset + k);
        fill_normals<real>(a, sm, tile, in_range, kg, nvalid);
        if (tile == blockIdx.x) TC_STAMP(1)     // normals drawn
        if (!staged) {
            stage_finish<real, VARIANT, NU>(a, sm);
            staged = true;
        } else {
            __syncthreads();
        }
        if (tile == blockIdx.x) TC_STAMP(2)     // nominal staged
        if (in_range) transform_column<real, VARIANT, NU>(a, sm, kg);
        __syncthreads();
        if (tile == blockIdx.x) TC_STAMP(3)     // perturbed actions built

        // ---- rollout: the MMAs are CTA-wide, so every thread keeps the step's three barriers ----------------
        real x[NX] = {(real)0, (real)0};
        if (active) {
            if (a.state_dev != nullptr) {
                const real* sp = a.state_dev + (a.state_per_sample ? (size_t)k * NX : 0);
                x[0] = sp[0];
                x[1] = sp[1];
            } else {
                x[0] = a.x0[0];
                x[1] = a.x0[1];
            }
        }
        real roll = (real)0, pert = (real)0, smooth = (real)0, vprev = (real)0, u_prev = (real)0;
        // debug_clocks (profiling aid, scripts/tc_phase_clocks.py): clock64() sums over the T steps of the first tile, per phase,
        // for thread 0 (the MMA issuer) in slots 0..7 and thread 32 (a plain worker) in slots 8..15 of this CTA's row
        const bool prof = a.dbg != nullptr && tile == blockIdx.x && (tid == 0 || tid == 32);
        long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pt = 0;
#define TC_PROF(slot)                          \
    if (prof) {                                \
        const long long now_ = clock64();      \
        pc[slot] += now_ - pt;                 \
        pt = now_;                             \
    }
        unsigned long long gt_loop0 = 0;
        if (prof) {
            pt = clock64();
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_loop0));
        }
        for (int t = 0; t < T; ++t) {
            real v[NU] = {(real)0}, eps[NU] = {(real)0};
            real u = (real)0;
            if (roller) {
                if (active) {
                    action_at<real, VARIANT, NU>(a, sm, kg, t, v);
                    noise_at<real, VARIANT, NU>(a, sm, t, v, eps);
                }
                u = O::mul(nm.u_scale, v[0]);
                const real uc = clamp<real>(u, -mp.max_torque, mp.max_torque);
                *reinterpret_cast<float4*>(sX + 4 * row) = make_float4(x[0], x[1], uc, 0.0f);
            }
            TC_PROF(0)      // state of the previous step + layer-1 input
            __syncthreads();
            TC_PROF(1)      // barrier
            float hv[16];
            {   // layer 1 on the FP32 pipe (exact fp32): 16 units x 3 FMAs -> tanh -> this thread's half of the layer-2 operand row
                const float4 xin = *reinterpret_cast<const float4*>(sX + 4 * row);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    float acc = mp.b1[hb + i];
                    acc = fmaf(mp.W1[0 * H + hb + i], xin.x, acc);
                    acc = fmaf(mp.W1[1 * H + hb + i], xin.y, acc);
                    acc = fmaf(mp.W1[2 * H + hb + i], xin.z, acc);
                    hv[i] = acc;
                }
#pragma unroll
                for (int i = 0; i < 16; i += 4) Model::tanh4_(hv + i, FAST);
                tc::write_a_half<SPLIT, CHUNKS>(sA2, row, half, hv);
                TC_PROF(5)  // layer 1 + tanh + pack + store
                tc::fence_async_smem();
                tc::fence_before();
                TC_PROF(6)  // proxy fence
            }
            __syncthreads();
            TC_PROF(1)
            if (warp == 0 && tc::elect_one()) {
                tc::fence_after();
#pragma unroll
                for (int s = 0; s < NSTEP; ++s) tc::mma_f16(tmem + C2, dA2 + s * KSTEP, dB2 + s * KSTEP, I32, s > 0 ? 1u : 0u);
                if (SPLIT) {
#pragma unroll
                    for (int s = 0; s < 2; ++s) tc::mma_f16(tmem + C2, dA2 + s * KSTEP, dB2lo + s * KSTEP, I32, 1u);
                }
                tc::mma_commit(&s_mma_bar);
            }
            TC_PROF(2)      // MMA issue (thread 0)
            // in the shadow of the layer-2 MMA: the running cost of the state the PREVIOUS step produced (x is x_t, the
            // state step t-1 led to) and this step's action cost — same values and summation order as the plain loop
            if (active) {
                if (t > 0) roll = O::add(roll, Model::template cost<real>(mp, x, &u_prev));   // mppi.py:318-319 (step t-1)
                pert = O::add(pert, action_cost_term<real, NU>(nm, eps, sm.Us + t * NU));
                if (VARIANT == V_SMPPI) {
                    if (t > 0) {
                        const real d = O::mul(nm.u_scale, O::sub(v[0], vprev));
                        smooth = O::add(smooth, O::mul(d, d));
                    }
                    vprev = v[0];
                }
            }
            u_prev = u;
            TC_PROF(7)      // deferred cost
            {   // layer 2 -> tanh -> half row of the layer-3 operand
                tc::mbar_wait_bounded(&s_mma_bar, mma_phase);
                TC_PROF(3)  // commit -> mbarrier
                tc::fence_after();
                tc::tmem_ld16_nowait(my_lane + C2 + 16 * half, hv);
                tc::tmem_wait_ld();
                TC_PROF(4)  // TMEM load
#pragma unroll
                for (int i = 0; i < 16; i += 4) Model::tanh4_(hv + i, FAST);
                tc::write_a_half<SPLIT, CHUNKS>(sA2, row, half, hv);     // MMA 2 has completed (barrier): its operand tile is free
                TC_PROF(5)
                tc::fence_async_smem();
                tc::fence_before();
                TC_PROF(6)
            }
            mma_phase ^= 1u;
            __syncthreads();
            TC_PROF(1)
            if (warp == 0 && tc::elect_one()) {
                tc::fence_after();
#pragma unroll
                for (int s = 0; s < NSTEP; ++s) tc::mma_f16(tmem + C3, dA2 + s * KSTEP, dB3 + s * KSTEP, I16, s > 0 ? 1u : 0u);
                if (SPLIT) {
#pragma unroll
                    for (int s = 0; s < 2; ++s) tc::mma_f16(tmem + C3, dA2 + s * KSTEP, dB3lo + s * KSTEP, I16, 1u);
                }
                tc::mma_commit(&s_mma_bar);
            }
            TC_PROF(2)
            tc::mbar_wait_bounded(&s_mma_bar, mma_phase);
            TC_PROF(3)
            tc::fence_after();
            if (roller) {
                float o0, o1;
                tc::tmem_ld2(my_lane + C3, o0, o1);
                const real th = O::add(x[0], o0);
                x[0] = O::sub(remainder<real>(O::add(th, mp.pi), mp.two_pi), mp.pi);    // pendulum_approximate.py:65
                x[1] = O::add(x[1], o1);
            }
            TC_PROF(4)
            // the next step's MMAs overwrite these accumulators: order the reads before the barrier that releases them
            tc::fence_before();
            mma_phase ^= 1u;
        }
        if (active) roll = O::add(roll, Model::template cost<real>(mp, x, &u_prev));              // step T-1
        if (prof) {
            if (tid == 0) {
#pragma unroll
                for (int i = 0; i < 8; ++i) a.dbg[(size_t)blockIdx.x * 16 + i] = (unsigned long long)pc[i];
            } else {     // the worker: its waiting / loading / tanh / cost sums, then wall-clock stamps of the rollout loop
                a.dbg[(size_t)blockIdx.x * 16 + 8] = (unsigned long long)pc[3];
                a.dbg[(size_t)blockIdx.x * 16 + 9] = (unsigned long long)pc[4];
                a.dbg[(size_t)blockIdx.x * 16 + 10] = (unsigned long long)pc[5];
                a.dbg[(size_t)blockIdx.x * 16 + 11] = (unsigned long long)(pc[0] + pc[1] + pc[2] + pc[6] + pc[7]);
                a.dbg[(size_t)blockIdx.x * 16 + 13] = gt_loop0;
                unsigned long long gt1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
                a.dbg[(size_t)blockIdx.x * 16 + 14] = gt1;
            }
        }
#undef TC_PROF
        real c_tot = O::inf();
        if (active) {
            c_tot = O::add(roll, pert);
            if (VARIANT == V_SMPPI) c_tot = O::add(c_tot, O::mul(smooth, nm.w_smooth));
            a.cost_total[k] = c_tot;
        }
        // the rollout warps (one sample per thread) fold the tile; the rows were ordered by the rollout's barriers
        if (roller) warp_fold<real, VARIANT, FOLD_ROWS>(a, sm, c_tot, active, nvalid);
        if (tile == blockIdx.x) TC_STAMP(4)     // tile folded
        if (tile + (int)gridDim.x < a.n_tiles) __syncthreads();      // the tile is refilled by the next pass
    }
    if (!staged) stage_finish<real, VARIANT, NU>(a, sm);
    tc::fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TMEM_COLS) : "memory");
    }
    TC_STAMP(5)         // TMEM released
    warp_tail<real, VARIANT, NU>(a, sm);
    if (a.dbg != nullptr && tid == 32) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        a.dbg[(size_t)blockIdx.x * 16 + 15] = gt;
    }
#undef TC_STAMP
}

#endif  // __CUDACC__

}  // namespace mppi
