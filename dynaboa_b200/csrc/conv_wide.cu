// Fused forward convolution, second generation ("wide" CTA): BOTH operands arrive through TMA, and the GroupNorm / residual /
// ReLU transform of the activation operand plus the TF32x3 hi/lo split of both operands are ONE elementwise pass over the
// landed shared-memory tiles, spread over 16 warps.
//
//      y = conv( T(x), W )   and   per (sample, group) statistics of y         (interface: FusedConv, kernels.h)
//
// Why (measured, profiles/r02_summary.md): at batch 1 a backbone layer is a ~10 us problem and the time of a CTA is
// the number of instructions on its critical warp times ~15 cycles (few warps, dependent chains: ncu "one instruction every
// 13..31 cycles per warp").  The first fused kernel of this round (not kept) used the register path of conv_tc.cu for activations --
// per k-block and thread ~300 instructions of address arithmetic, loads, transform and split -- and a per-CTA merge of
// partial statistics; it ran SLOWER than the unfused plan.  Here:
//   * activations: 4-D TMA boxes (32 channels x W x rows x 1 sample) with the filter tap as a coordinate offset and
//     hardware zero fill for the padding: no address arithmetic, no bounds logic, any prefetch depth without registers;
//   * the transform pass handles a tile with 512 threads: 2 float4 of activations + 1 float4 of weights per thread and
//     k-block (~85 instructions), writing hi in place and lo to a second tile at the same (swizzled) offsets;
//   * GroupNorm statistics leave the epilogue as TWO 64-bit fixed-point atomics per (tile, group) (sum, sum of squares
//     scaled by 2^24: integer addition is associative, so the result is exact and order independent, hence deterministic);
//     the consumer reads 8 integers instead of merging hundreds of partial triples;
//   * output tiles are whole image rows (W x rows <= 128 pixels), so a tile is a rectangle the TMA box can address.
// Stride 1 and 2 (1x1, 3x3): for stride 2 the tensor map itself samples every second pixel (TMA element strides).
#include <cooperative_groups.h>
#include <cuda.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace dboa {
namespace wz {

constexpr int BM = 128, BN = 64, BK = 32;
constexpr int NTW = 16, NTT = NTW * 32;              // transform warps / threads
constexpr int W_MMA = 16, W_TMA = 17, NT = 576;
constexpr int DMAX = 4;                               // raw-tile ring depth
constexpr int NACC = 4;                               // TMEM accumulators a reduction chain rotates over (see the MMA issuer)
constexpr uint32_t A_TILE = BM * BK * 4, B_TILE = BN * BK * 4;
constexpr int RED_LD = BN + 4;
constexpr float GN_EPS = 1e-5f;
constexpr double FIX = 16777216.0;                    // 2^24 fixed-point scale of the statistics accumulators

struct Problem {
    const float* res_dummy;      // unused (kept for layout clarity)
    float* a_out;                // materialised transformed operand [B][Hi][Wi][Cin] or NULL
    float* stats_out;            // (mean, rstd) [B][4][2] of the operand's GroupNorm or NULL
    float* stats2_out;
    const long long* acc_in;     // modes 1-3: fixed-point (sum, sum of squares) [B][4][2] of x
    const long long* acc2_in;    // mode 3: of res
    const float* gamma; const float* beta; const float* gamma2; const float* beta2;
    float* y;                    // output [B][Ho][Wo][Cout]
    unsigned long long* acc_out; // [B][4][2]
    int Hi, Wi, Cin, Ho, Wo, Cout, k, pad, stride;
    int bh, tps, ntiles, nclusters;
};
struct Launch {
    Problem p[2];
    int nprob, nz, per, D, tabc;
    const float* next_w;         // weights of the NEXT launch: prefetched into L2 by this one
    unsigned long long next_bytes;
    // chain dependency (see chain_wait): counter every CTA of the PREVIOUS fused launch increments when its outputs are stored,
    // the value it reaches, and this launch's own counter; NULL = ordinary programmatic dependency (griddepcontrol.wait)
    const unsigned* dep_flag;
    unsigned dep_expect;
    unsigned* done_flag;
    int launch_id;
};

// Diagnostic build (-DDBOA_TIMELINE, scripts/fused_timeline.py): %globaltimer stamps of thread 0 of the first 256 CTAs of every
// launch at the phase boundaries, g_ftl[launch][cta][16], and per-k-block stamps of CTA 0; compiled out of the product library.
#ifdef DBOA_TIMELINE
__device__ unsigned long long* g_ftl = nullptr;
__device__ int g_knobs = 0;          // diagnostic knobs (results are WRONG with any of them set): 1 no MMAs, 2 no transform body, 4 no cluster reduction
#define KNOB(b) ((g_knobs & (b)) != 0)
#define FTL(i)                                                                                          \
    do {                                                                                                \
        if (threadIdx.x == 0 && g_ftl != nullptr && blockIdx.x < 256 && L.launch_id < 128) {           \
            unsigned long long t_;                                                                      \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                      \
            g_ftl[((size_t)L.launch_id * 256 + blockIdx.x) * 16 + (i)] = t_;                            \
        }                                                                                               \
    } while (0)
#define FTI(it, j)                                                                                      \
    do {                                                                                                \
        if (g_ftl != nullptr && blockIdx.x == 0 && L.launch_id < 128 && (it) < 16) {                    \
            unsigned long long t_;                                                                      \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                      \
            g_ftl[(size_t)128 * 256 * 16 + ((size_t)L.launch_id * 16 + (it)) * 8 + (j)] = t_;           \
        }                                                                                               \
    } while (0)
#else
#define FTL(i)
#define FTI(it, j)
#define KNOB(b) false
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// K-major, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor, layout_type 2)
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)((1024 >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand read from tensor memory (lane = tile row, one 32-bit column per TF32 element): the tensor core fetches only B from
// shared memory
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 8 consecutive 32-bit columns of this thread's TMEM lane (lane = 32 * (warp % 4) + lane id)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float4 a, const float4 b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(__float_as_uint(a.x)),
                 "r"(__float_as_uint(a.y)), "r"(__float_as_uint(a.z)), "r"(__float_as_uint(a.w)), "r"(__float_as_uint(b.x)), "r"(__float_as_uint(b.y)),
                 "r"(__float_as_uint(b.z)), "r"(__float_as_uint(b.w))
                 : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded wait: a protocol error traps (the launch fails) instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0, addr = smem_u32(bar);
    long long t0 = 0;
    while (true) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (t0 == 0) t0 = clock64();
        else if (clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
                 : "memory");
}
// shared memory through 32-bit shared-window addresses (the carve-up below goes through integer arithmetic, which makes the
// compiler fall back to generic LD/ST with 64-bit address arithmetic otherwise)
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 ldc128(uint32_t a, uint32_t cta) {      // the same offset in the shared memory of CTA `cta` of the cluster
    uint32_t ra;
    float4 v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(cta));
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ra) : "memory");
    return v;
}
// one lane of a converged warp (elect.sync): the compiler knows the guarded region runs on a single thread and keeps tcgen05
// instructions on the uniform datapath without its per-thread ELECT / BRA.U.ANY wrapper loops
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
// Dependency of a fused launch on the previous fused launch of the same forward WITHOUT waiting for that grid to complete:
// griddepcontrol.wait returns only when every CTA of the producer has exited and its memory is flushed, which puts the producer's
// exit barrier (cluster.sync: peers still read this CTA's shared memory), its tear-down and the completion signalling (~1.5 us) on
// the critical path of every layer.  Here every producer CTA increments a counter right after its last global store / atomic
// (fence + atomic = release), and the consumer's two readers of producer data -- the thread that issues the activation TMA loads
// and the threads that read the statistics accumulators -- spin on it with acquire loads.  No deadlock: a dependent grid is only
// launched once every CTA of its predecessor has executed griddepcontrol.launch_dependents, i.e. is resident, so a spinning
// consumer never holds an SM that its producer still needs.  Bounded: a protocol error traps instead of hanging the device.
__device__ __forceinline__ void chain_wait(const unsigned* flag, unsigned expect) {
    long long t0 = 0;
    while (true) {
        unsigned v;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v >= expect) break;
        if (t0 == 0) t0 = clock64();
        else if (clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

#define PW(field) (second ? L.p[1].field : L.p[0].field)

// tensor maps: tmx = operand x of problem 0 / 1, tmr = second operand (modes 2, 3), tmw = weights
// ATM: the transformed activation operand (hi and lo parts) lives in tensor memory instead of shared memory (see the transform warps)
template <int MODE, bool ATM>
__global__ void __launch_bounds__(NT, 1) conv_wide_kernel(const __grid_constant__ Launch L, const __grid_constant__ CUtensorMap tmx0,
                                                          const __grid_constant__ CUtensorMap tmx1, const __grid_constant__ CUtensorMap tmr0,
                                                          const __grid_constant__ CUtensorMap tmr1, const __grid_constant__ CUtensorMap tmw0,
                                                          const __grid_constant__ CUtensorMap tmw1) {
    extern __shared__ uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nz = L.nz, D = L.D;
    FTL(0);
    const int cidx = blockIdx.x / nz, rank = blockIdx.x - cidx * nz;
    const bool second = L.nprob > 1 && cidx >= L.p[0].nclusters;
    const int tix = second ? cidx - L.p[0].nclusters : cidx;
    const CUtensorMap* tmx = second ? &tmx1 : &tmx0;
    const CUtensorMap* tmw = second ? &tmw1 : &tmw0;
    const CUtensorMap* tmr = second ? &tmr1 : &tmr0;
    const int Hi = PW(Hi), Wi = PW(Wi), Cin = PW(Cin), Ho = PW(Ho), Wo = PW(Wo), Cout = PW(Cout), ks = PW(k), pad = PW(pad), stride = PW(stride);
    const int bh = PW(bh), tps = PW(tps), ntiles = PW(ntiles);
    const int nt = tix % ntiles, bm = tix / ntiles, mt = bm % tps, b = bm / tps;
    const int h0 = mt * bh, n0 = nt * BN;
    const int rows_valid = min(bh, Ho - h0) * Wo;          // output pixels of this tile (whole image rows)
    const int m0 = h0 * Wo;                                // first output pixel of the tile inside the sample
    const int nkb_total = (ks * ks * Cin) / BK;
    const int kb_begin = rank * L.per;
    const int nkb = max(0, min(L.per, nkb_total - kb_begin));
    constexpr bool HAS_RES = MODE >= 2;
    const uint32_t slot_bytes = A_TILE * (HAS_RES ? 2 : 1) + B_TILE;
    const uint32_t a_bytes = (uint32_t)(bh * Wo) * 128u;   // bytes one activation box delivers

    // ---- shared memory (1024-byte aligned): D raw slots {A [, R], B}, 2 lo sets {A, B}, tables, barriers
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* slots = base;
    uint8_t* lo_a = slots + (size_t)D * slot_bytes;        // 2 x 16 KB
    uint8_t* lo_b = lo_a + 2 * A_TILE;                     // 2 x 8 KB
    float* tab = reinterpret_cast<float*>(lo_b + 2 * B_TILE);                 // gamma | beta [| gamma2 | beta2], tabc floats each
    uint64_t* bars = reinterpret_cast<uint64_t*>(tab + (MODE == 3 ? 4 : (MODE >= 1 ? 2 : 0)) * (size_t)L.tabc);
    uint64_t* s_full = bars;               // [DMAX] TMA -> transform warps
    uint64_t* s_empty = bars + DMAX;       // [DMAX] tcgen05.commit -> TMA warp
    uint64_t* l_full = bars + 2 * DMAX;    // [2] transform warps -> MMA issuer
    uint64_t* l_empty = l_full + 2;        // [2] tcgen05.commit -> transform warps
    uint64_t* done = l_empty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    float4* wpart = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(bars) + 128);     // [NTW][4]
    float* sstat = reinterpret_cast<float*>(wpart + NTW * 4);                                // [16]
    float* red = reinterpret_cast<float*>(lo_a);           // 128 x RED_LD fp32 partial tile over the lo sets after the last MMA (34 KB <= 48 KB)

    if (tid == 0) {
        for (int s = 0; s < DMAX; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&l_full[s], ATM ? NTW / 2 : NTW); mbar_init(&l_empty[s], 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(ATM ? 512 : BN * NACC) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    const int tc0 = ks == 1 ? kb_begin * BK : 0, tcn = ks == 1 ? nkb * BK : Cin;
    if (MODE >= 1) {
        const float* ga = PW(gamma); const float* be = PW(beta);
        for (int i = tid; i < tcn; i += NT) { tab[i] = __ldg(ga + tc0 + i); tab[L.tabc + i] = __ldg(be + tc0 + i); }
        if (MODE == 3) {
            const float* ga2 = PW(gamma2); const float* be2 = PW(beta2);
            for (int i = tid; i < tcn; i += NT) { tab[2 * L.tabc + i] = __ldg(ga2 + tc0 + i); tab[3 * L.tabc + i] = __ldg(be2 + tc0 + i); }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;
    FTL(1);

    // reduction cursor of k-block kb: filter tap (r, s) and channel offset
    auto tap_of = [&](int kb, int& r, int& s, int& c) {
        const int k0 = kb * BK, tap = k0 / Cin;
        c = k0 - tap * Cin; r = tap / ks; s = tap - r * ks;
    };

    if (warp == W_TMA) {
        // =====================================================================================
        // operand feed (one thread): weight boxes before the dependency wait, activation boxes after it
        // =====================================================================================
        if (lane == 0 && nkb > 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmw)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmx)) : "memory");
            const int npre = min(nkb, D);
            for (int it = 0; it < npre; ++it) {
                mbar_expect_tx(&s_full[it], a_bytes * (HAS_RES ? 2 : 1) + B_TILE);
                tma_load_2d(smem_u32(slots + (size_t)it * slot_bytes + A_TILE * (HAS_RES ? 2 : 1)), tmw, (kb_begin + it) * BK, n0, &s_full[it]);
            }
            if (L.dep_flag != nullptr) {
                pdl_trigger();
                chain_wait(L.dep_flag, L.dep_expect);
                asm volatile("fence.proxy.async;" ::: "memory");        // the producer's generic-proxy stores before this thread's TMA reads
            } else {
                pdl_wait();
                pdl_trigger();
            }
            for (int it = 0; it < nkb; ++it) {
                const int sl = it % D;
                uint8_t* slot = slots + (size_t)sl * slot_bytes;
                if (it >= D) {
                    mbar_wait(&s_empty[sl], (uint32_t)(((it / D) - 1) & 1));
                    mbar_expect_tx(&s_full[sl], a_bytes * (HAS_RES ? 2 : 1) + B_TILE);
                    tma_load_2d(smem_u32(slot + A_TILE * (HAS_RES ? 2 : 1)), tmw, (kb_begin + it) * BK, n0, &s_full[sl]);
                }
                int r, s, c;
                tap_of(kb_begin + it, r, s, c);
                // box origin in INPUT coordinates; the tensor map samples every `stride`-th pixel (element strides)
                tma_load_4d(smem_u32(slot), tmx, c, s - pad, h0 * stride + r - pad, b, &s_full[sl]);
                FTI(it, 7);
                if (HAS_RES) tma_load_4d(smem_u32(slot + A_TILE), tmr, c, s - pad, h0 * stride + r - pad, b, &s_full[sl]);
            }
        } else {
            // lanes 1..31: the NEXT layer's weights DRAM -> L2 while this layer computes (each CTA takes a slice; weights are
            // never written by a convolution launch, so no dependency wait is needed)
            if (L.next_w != nullptr && lane > 0) {
                const unsigned long long chunk = ((L.next_bytes / gridDim.x) + 1023) & ~1023ull;
                const unsigned long long beg = chunk * blockIdx.x;
                for (unsigned long long o = beg + (unsigned long long)(lane - 1) * 1024; o < beg + chunk && o + 1024 <= L.next_bytes; o += 31 * 1024)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], 1024;" ::"l"(reinterpret_cast<const char*>(L.next_w) + o) : "memory");
            }
            if (L.dep_flag == nullptr) pdl_wait();
            pdl_trigger();
        }
    } else if (warp == W_MMA) {
        // =====================================================================================
        // MMA issuer: 12 x tcgen05.mma per k-block (4 k-steps of 8 x {Ah*Bh, Ah*Bl, Al*Bh}).
        // The tensor core adds into the fp32 accumulator with truncation: a chain of n accumulations shrinks the result by
        // ~n * 2^-25 (measured: 2e-5 after 72 k-blocks).  k-block `it` therefore goes to accumulator it % 4 (4 x 64 TMEM
        // columns); the epilogue adds the four in fp32 with round-to-nearest.
        // =====================================================================================
        // The whole warp runs the loop (warp-uniform control flow keeps the descriptor arithmetic on the uniform datapath: under a
        // divergent `if (lane == 0)` every tcgen05.mma paid four R2UR moves with their latency); lane 0 issues.
        if (nkb > 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint64_t dslot = desc_sw128(smem_u32(slots)), dloa = desc_sw128(smem_u32(lo_a)), dlob = desc_sw128(smem_u32(lo_b));
            constexpr uint64_t KSTEP = 32 >> 4;
            const uint32_t slot16 = slot_bytes >> 4, wofs16 = (A_TILE * (HAS_RES ? 2 : 1)) >> 4;
            int sl = 0;
#pragma unroll 1
            for (int it = 0; it < nkb; ++it) {
                const int ls = it & 1;
                mbar_wait(&l_full[ls], (uint32_t)((it >> 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                FTI(it, 5);
                const uint64_t dah = dslot + (uint64_t)(sl * slot16);
                const uint64_t dbh = dah + (uint64_t)wofs16;
                const uint64_t dal = dloa + (uint64_t)(ls * (A_TILE >> 4)), dbl = dlob + (uint64_t)(ls * (B_TILE >> 4));
                const uint32_t dacc = tmem_d + (uint32_t)((it & (NACC - 1)) * BN);
                const uint32_t first = it >= NACC ? 1u : 0u;
                if (elect_one()) {
                    if (KNOB(1)) {
                    } else if constexpr (ATM) {
                        // A hi / lo of stage ls: TMEM columns ACOL + 64 ls + {0..31, 32..63}, 8 columns per k-step
                        const uint32_t tah = tmem_d + (uint32_t)(BN * NACC + ls * 2 * BK), tal = tah + (uint32_t)BK;
#pragma unroll
                        for (int kk = 0; kk < BK / 8; ++kk) {
                            mma_tf32_ts(dacc, tah + kk * 8, dbh + kk * KSTEP, idesc, kk > 0 ? 1u : first);
                            mma_tf32_ts(dacc, tah + kk * 8, dbl + kk * KSTEP, idesc, 1u);
                            mma_tf32_ts(dacc, tal + kk * 8, dbh + kk * KSTEP, idesc, 1u);
                        }
                    } else {
#pragma unroll
                        for (int kk = 0; kk < BK / 8; ++kk) {
                            mma_tf32(dacc, dah + kk * KSTEP, dbh + kk * KSTEP, idesc, kk > 0 ? 1u : first);
                            mma_tf32(dacc, dah + kk * KSTEP, dbl + kk * KSTEP, idesc, 1u);
                            mma_tf32(dacc, dal + kk * KSTEP, dbh + kk * KSTEP, idesc, 1u);
                        }
                    }
                    umma_commit(&l_empty[ls]);
                    umma_commit(&s_empty[sl]);
                }
                __syncwarp();
                FTI(it, 6);
                if (++sl == D) sl = 0;
            }
            if (elect_one()) umma_commit(done);
        }
        if (L.dep_flag == nullptr) pdl_wait();
        pdl_trigger();
    } else {
        // =====================================================================================
        // transform warps: thread t owns float4 t and t + 512 of the activation tile (rows r0 = t >> 3 and r0 + 64, the same
        // physical 16-byte chunk pc = t & 7, hence the same logical chunk lc = pc ^ (r0 & 7)) and float4 t of the weight tile
        // =====================================================================================
        // ATM: thread = tile row (= its TMEM lane: 32 * (warp % 4) + lane) x 16 channels kh * 16 .. + 15 of every second k-block; only
        // entry 0 of the per-row arrays is used
        const int r0 = ATM ? (warp & 3) * 32 + lane : tid >> 3, pc = tid & 7, lc = pc ^ (r0 & 7), kh = (warp >> 2) & 1, grp = warp >> 3;
        // per-thread invariants of the two activation rows: input coordinates of tap (0, 0), validity, tape pointer of tap (0, 0)
        float* ab = (MODE >= 1 && PW(a_out) != nullptr && nt == 0) ? PW(a_out) + (size_t)b * Hi * Wi * Cin : nullptr;
        int hq[2], wq[2];
        bool rowok[2];
        float* abq[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int i = r0 + 64 * q, oh = i / Wo, ow = i - oh * Wo;
            hq[q] = (h0 + oh) * stride - pad; wq[q] = ow * stride - pad; rowok[q] = i < rows_valid;
            abq[q] = ab + ((long long)hq[q] * Wi + wq[q]) * Cin + (ATM ? kh * 16 : lc * 4);      // only dereferenced for in-bounds taps
        }
        int lgw = 0;
        while ((4 << lgw) < Cin) ++lgw;
        // everything that does not depend on the producing kernel happens before the dependency wait (double-precision
        // divisions included: 1 / (N * 2^24) turns the fixed-point sums into means with one multiplication each)
        const double inv_nfix = 1.0 / ((double)Hi * Wi * (Cin >> 2) * FIX);
        int r, s, c;
        tap_of(kb_begin, r, s, c);
        if (L.dep_flag != nullptr) {
            // only the threads that read the statistics accumulators wait; the barrier after them orders everybody else
            pdl_trigger();
            if (MODE == 0 || tid < (MODE == 3 ? 8 : 4)) chain_wait(L.dep_flag, L.dep_expect);
        } else {
            pdl_wait();
            pdl_trigger();
        }
        FTL(2);
        if (MODE >= 1) {
            // statistics of the operand's GroupNorm(s): 8 fixed-point sums per sample -> (mean, rstd)
            if (tid < (MODE == 3 ? 8 : 4)) {
                const long long* acc = (tid < 4 ? PW(acc_in) : PW(acc2_in)) + ((size_t)b * 4 + (tid & 3)) * 2;
                const double mu = (double)__ldcg(acc) * inv_nfix, var = fmax((double)__ldcg(acc + 1) * inv_nfix - mu * mu, 0.0);
                sstat[(tid >> 2) * 8 + (tid & 3)] = (float)mu;
                sstat[(tid >> 2) * 8 + 4 + (tid & 3)] = 1.0f / sqrtf((float)var + GN_EPS);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(NTT) : "memory");
            if (mt == 0 && nt == 0 && rank == 0 && tid < 8) {
                float* so = PW(stats_out);
                if (so != nullptr) so[(b * 4 + (tid & 3)) * 2 + (tid >> 2)] = sstat[tid];
                if (MODE == 3) {
                    float* so2 = PW(stats2_out);
                    if (so2 != nullptr) so2[(b * 4 + (tid & 3)) * 2 + (tid >> 2)] = sstat[8 + tid];
                }
            }
            // per-channel affine of the normalisation, folded once per CTA: a = x * sc + sh with sc = gamma * rstd,
            // sh = beta - mean * sc (mode 3: the second operand's shift is folded into sh as well)
            for (int i = tid; i < tcn; i += NTT) {
                const int g = (tc0 + i) >> lgw;
                const float sc = tab[i] * sstat[4 + g];
                float sh = tab[L.tabc + i] - sstat[g] * sc;
                if (MODE == 3) {
                    const float sc2 = tab[2 * L.tabc + i] * sstat[12 + g];
                    sh += tab[3 * L.tabc + i] - sstat[8 + g] * sc2;
                    tab[2 * L.tabc + i] = sc2;
                }
                tab[i] = sc; tab[L.tabc + i] = sh;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(NTT) : "memory");
        }
        int sl = 0;
        uint32_t ph_full = 0;
        const uint32_t slots32 = smem_u32(slots), tab32 = smem_u32(tab), tabc4 = (uint32_t)L.tabc * 4u;
        const uint32_t offA = (uint32_t)tid * 16u;
        const uint32_t lo_a32 = smem_u32(lo_a) + offA, lo_b32 = smem_u32(lo_b) + offA;
        const uint32_t wofs = A_TILE * (HAS_RES ? 2 : 1);
        uint32_t slot = slots32 + offA;                                  // this thread's first chunk inside the current slot
        if constexpr (ATM) {
            // The transformed activation tile goes to TENSOR memory (tcgen05.st, thread = row) and the MMAs read it from there: per
            // k-block the shared-memory pipe carries 24 KB of raw reads + 16 KB of weight hi / lo writes + 24 KB of tensor-core B
            // reads instead of 24 + 48 + 72 KB.  Row r's logical 16-byte chunk j sits at physical chunk j ^ (r & 7) (128-byte
            // swizzle of the TMA box): a quarter warp reads 8 different physical chunks -> conflict-free.
            // TWO GROUPS of 8 warps alternate k-blocks (group g: k-blocks g, g + 2, ...; stage g of the TMEM operand and of the
            // weight lo tile): one k-block is a dependent chain  barrier wait -> LDS -> FMA -> STTM / STS -> wait::st -> proxy
            // fence -> arrive  of ~600 cycles that 16 warps in lock step cannot hide (stall samples of the one-group loop: LDS
            // scoreboard, FENCE.VIEW.ASYNC and the barrier polls); with two groups the chains of consecutive k-blocks overlap.
            // Thread = row r0 x 16 channels (logical chunks 4 kh .. 4 kh + 3) + float4 tg and tg + 256 of the weight tile.
            const uint32_t rowofs = (uint32_t)r0 * 128u, sw = (uint32_t)(r0 & 7);
            uint32_t pa[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pa[j] = rowofs + (((uint32_t)(4 * kh + j) ^ sw) << 4);
            const uint32_t ta = tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(BN * NACC + grp * 2 * BK + kh * 16);
            const uint32_t offW = (uint32_t)((warp & 7) * 32 + lane) * 16u;
            const uint32_t lob = smem_u32(lo_b) + (uint32_t)grp * B_TILE + offW;
            auto step = [&]() { c += BK; if (c >= Cin) { c = 0; if (++s == ks) { s = 0; ++r; } } };
            if (grp == 1) step();
            int sl = grp % D;
            uint32_t ph_full = (uint32_t)((grp / D) & 1);
            uint32_t sbase = slots32 + (uint32_t)sl * slot_bytes;
#pragma unroll 1
            for (int it = grp; it < nkb; it += 2) {
                const uint32_t ti = tab32 + (uint32_t)(c - tc0 + kh * 16) * 4u;   // this warp's 16 channels inside the channel table (broadcast reads)
                const bool desig = ab != nullptr && (ks == 1 ? stride == 1 : (stride == 1 ? (r == 1 && s == 1) : (r >= 1 && s >= 1)));
                const int tapoff = (r * Wi + s) * Cin + c;
                const bool in0 = rowok[0] && (unsigned)(hq[0] + r) < (unsigned)Hi && (unsigned)(wq[0] + s) < (unsigned)Wi;
                if ((tid & 255) == 0) FTI(it, 0);
                mbar_wait(&s_full[sl], ph_full);
                if ((tid & 255) == 0) FTI(it, 1);
                float4 v[4], q[4];
                if (KNOB(2)) {
                    if (it >= 2) mbar_wait(&l_empty[grp], (uint32_t)(((it >> 1) - 1) & 1));
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&l_full[grp]);
                    sl += 2;
                    while (sl >= D) { sl -= D; ph_full ^= 1u; }
                    sbase = slots32 + (uint32_t)sl * slot_bytes;
                    step(); step();
                    continue;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = lds128(sbase + pa[j]);
                if (MODE >= 2) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) q[j] = lds128(sbase + A_TILE + pa[j]);
                }
                const float4 w0 = lds128(sbase + wofs + offW), w1 = lds128(sbase + wofs + offW + 4096u);
                if (MODE >= 1) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 sc = lds128(ti + 16 * j), sh = lds128(ti + tabc4 + 16 * j);
                        v[j].x = fmaf(v[j].x, sc.x, sh.x); v[j].y = fmaf(v[j].y, sc.y, sh.y); v[j].z = fmaf(v[j].z, sc.z, sh.z); v[j].w = fmaf(v[j].w, sc.w, sh.w);
                        if (MODE == 2) {
                            v[j].x += q[j].x; v[j].y += q[j].y; v[j].z += q[j].z; v[j].w += q[j].w;
                        } else if (MODE == 3) {
                            const float4 s2 = lds128(ti + 2 * tabc4 + 16 * j);
                            v[j].x = fmaf(q[j].x, s2.x, v[j].x); v[j].y = fmaf(q[j].y, s2.y, v[j].y); v[j].z = fmaf(q[j].z, s2.z, v[j].z); v[j].w = fmaf(q[j].w, s2.w, v[j].w);
                        }
                        // padding is zero in the ACTIVATION domain
                        v[j].x = in0 ? fmaxf(v[j].x, 0.f) : 0.f; v[j].y = in0 ? fmaxf(v[j].y, 0.f) : 0.f;
                        v[j].z = in0 ? fmaxf(v[j].z, 0.f) : 0.f; v[j].w = in0 ? fmaxf(v[j].w, 0.f) : 0.f;
                    }
                    if (desig && in0) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(abq[0] + tapoff + 4 * j) = v[j];
                    }
                } else if (!rowok[0]) {
                    // rows the box did not deliver hold stale shared memory: keep them finite
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                float4 h[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    h[j] = make_float4(tf32_hi(v[j].x), tf32_hi(v[j].y), tf32_hi(v[j].z), tf32_hi(v[j].w));
                    v[j] = make_float4(v[j].x - h[j].x, v[j].y - h[j].y, v[j].z - h[j].z, v[j].w - h[j].w);
                }
                const float4 hw0 = make_float4(tf32_hi(w0.x), tf32_hi(w0.y), tf32_hi(w0.z), tf32_hi(w0.w));
                const float4 hw1 = make_float4(tf32_hi(w1.x), tf32_hi(w1.y), tf32_hi(w1.z), tf32_hi(w1.w));
                // the MMAs of k-block it - 2 (the previous user of this group's TMEM / lo stage) must have completed
                if ((tid & 255) == 0) FTI(it, 2);
                if (it >= 2) mbar_wait(&l_empty[grp], (uint32_t)(((it >> 1) - 1) & 1));
                if ((tid & 255) == 0) FTI(it, 4);
                tmem_st8(ta, h[0], h[1]);
                tmem_st8(ta + 8, h[2], h[3]);
                tmem_st8(ta + BK, v[0], v[1]);
                tmem_st8(ta + BK + 8, v[2], v[3]);
                sts128(sbase + wofs + offW, hw0);
                sts128(sbase + wofs + offW + 4096u, hw1);
                sts128(lob, make_float4(w0.x - hw0.x, w0.y - hw0.y, w0.z - hw0.z, w0.w - hw0.w));
                sts128(lob + 4096u, make_float4(w1.x - hw1.x, w1.y - hw1.y, w1.z - hw1.z, w1.w - hw1.w));
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&l_full[grp]);
                if ((tid & 255) == 0) FTI(it, 3);
                if (it == 0) FTL(3);
                // this group's next k-block: two steps of the slot ring and of the reduction cursor
                sl += 2;
                while (sl >= D) { sl -= D; ph_full ^= 1u; }
                sbase = slots32 + (uint32_t)sl * slot_bytes;
                step(); step();
            }
        } else {
#pragma unroll 1
        for (int it = 0; it < nkb; ++it) {
            const int ls = it & 1;
            const uint32_t ti = tab32 + (uint32_t)(c - tc0 + lc * 4) * 4u;   // this thread's chunk inside the channel table
            float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f), sc2 = sc;
            if (MODE >= 1) {
                sc = lds128(ti); sh = lds128(ti + tabc4);
                if (MODE == 3) sc2 = lds128(ti + 2 * tabc4);
            }
            // taps that together visit every input pixel exactly once (stride 2, 3x3: the four taps (1..2, 1..2))
            const bool desig = ab != nullptr && (ks == 1 ? stride == 1 : (stride == 1 ? (r == 1 && s == 1) : (r >= 1 && s >= 1)));
            const int tapoff = (r * Wi + s) * Cin + c;
            if (tid == 0) FTI(it, 0);
            mbar_wait(&s_full[sl], ph_full);
            if (tid == 0) FTI(it, 1);
            if (it >= 2) mbar_wait(&l_empty[ls], (uint32_t)(((it >> 1) - 1) & 1));
            if (tid == 0) FTI(it, 2);
            float4 v0 = lds128(slot), v1 = lds128(slot + NTT * 16u);
            const float4 vw = lds128(slot + wofs);
            if (MODE >= 1) {
                float4 q0, q1;
                if (MODE >= 2) { q0 = lds128(slot + A_TILE); q1 = lds128(slot + A_TILE + NTT * 16u); }
                const bool in0 = rowok[0] && (unsigned)(hq[0] + r) < (unsigned)Hi && (unsigned)(wq[0] + s) < (unsigned)Wi;
                const bool in1 = rowok[1] && (unsigned)(hq[1] + r) < (unsigned)Hi && (unsigned)(wq[1] + s) < (unsigned)Wi;
                v0.x = fmaf(v0.x, sc.x, sh.x); v0.y = fmaf(v0.y, sc.y, sh.y); v0.z = fmaf(v0.z, sc.z, sh.z); v0.w = fmaf(v0.w, sc.w, sh.w);
                v1.x = fmaf(v1.x, sc.x, sh.x); v1.y = fmaf(v1.y, sc.y, sh.y); v1.z = fmaf(v1.z, sc.z, sh.z); v1.w = fmaf(v1.w, sc.w, sh.w);
                if (MODE == 2) {
                    v0.x += q0.x; v0.y += q0.y; v0.z += q0.z; v0.w += q0.w;
                    v1.x += q1.x; v1.y += q1.y; v1.z += q1.z; v1.w += q1.w;
                } else if (MODE == 3) {
                    v0.x = fmaf(q0.x, sc2.x, v0.x); v0.y = fmaf(q0.y, sc2.y, v0.y); v0.z = fmaf(q0.z, sc2.z, v0.z); v0.w = fmaf(q0.w, sc2.w, v0.w);
                    v1.x = fmaf(q1.x, sc2.x, v1.x); v1.y = fmaf(q1.y, sc2.y, v1.y); v1.z = fmaf(q1.z, sc2.z, v1.z); v1.w = fmaf(q1.w, sc2.w, v1.w);
                }
                // padding is zero in the ACTIVATION domain
                v0.x = in0 ? fmaxf(v0.x, 0.f) : 0.f; v0.y = in0 ? fmaxf(v0.y, 0.f) : 0.f; v0.z = in0 ? fmaxf(v0.z, 0.f) : 0.f; v0.w = in0 ? fmaxf(v0.w, 0.f) : 0.f;
                v1.x = in1 ? fmaxf(v1.x, 0.f) : 0.f; v1.y = in1 ? fmaxf(v1.y, 0.f) : 0.f; v1.z = in1 ? fmaxf(v1.z, 0.f) : 0.f; v1.w = in1 ? fmaxf(v1.w, 0.f) : 0.f;
                if (desig) {
                    if (in0) *reinterpret_cast<float4*>(abq[0] + tapoff) = v0;
                    if (in1) *reinterpret_cast<float4*>(abq[1] + tapoff) = v1;
                }
            }
            const float4 h0v = make_float4(tf32_hi(v0.x), tf32_hi(v0.y), tf32_hi(v0.z), tf32_hi(v0.w));
            const float4 h1v = make_float4(tf32_hi(v1.x), tf32_hi(v1.y), tf32_hi(v1.z), tf32_hi(v1.w));
            const float4 hw = make_float4(tf32_hi(vw.x), tf32_hi(vw.y), tf32_hi(vw.z), tf32_hi(vw.w));
            sts128(slot, h0v);
            sts128(slot + NTT * 16u, h1v);
            sts128(slot + wofs, hw);
            sts128(lo_a32 + ls * A_TILE, make_float4(v0.x - h0v.x, v0.y - h0v.y, v0.z - h0v.z, v0.w - h0v.w));
            sts128(lo_a32 + ls * A_TILE + NTT * 16u, make_float4(v1.x - h1v.x, v1.y - h1v.y, v1.z - h1v.z, v1.w - h1v.w));
            sts128(lo_b32 + ls * B_TILE, make_float4(vw.x - hw.x, vw.y - hw.y, vw.z - hw.z, vw.w - hw.w));
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&l_full[ls]);
            if (tid == 0) FTI(it, 3);
            if (it == 0) FTL(3);
            // next k-block: slot ring and reduction cursor (no divisions in the loop)
            slot += slot_bytes;
            if (++sl == D) { sl = 0; slot = slots32 + offA; ph_full ^= 1u; }
            c += BK;
            if (c >= Cin) { c = 0; if (++s == ks) { s = 0; ++r; } }
        }
        }
    }
    FTL(4);
    if (nkb > 0) mbar_wait(done, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    FTL(5);

    // ---- epilogue: TMEM -> shared memory (thread = row), split-K reduction over the cluster, output + statistics
    const uint32_t red32 = smem_u32(red);
    if (warp < NTW) {
        const int q4 = warp & 3, cgp = warp >> 2;               // lane quadrant, 16-column group
        float facc[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) facc[q] = 0.f;
        const int nacc = nkb < NACC ? nkb : NACC;
#pragma unroll 1
        for (int a = 0; a < nacc; a += 2) {
            uint32_t r[32];
            const uint32_t taddr = tmem_d + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(a * BN + cgp * 16);
            const bool two = a + 1 < nacc;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                  "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                : "r"(taddr)
                : "memory");
            if (two)
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                    : "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                      "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr + (uint32_t)BN)
                    : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int q = 0; q < 16; ++q) facc[q] += __uint_as_float(r[q]);
            if (two) {
#pragma unroll
                for (int q = 0; q < 16; ++q) facc[q] += __uint_as_float(r[16 + q]);
            }
        }
        const uint32_t dst = red32 + (uint32_t)((q4 * 32 + lane) * RED_LD + cgp * 16) * 4u;
#pragma unroll
        for (int q = 0; q < 4; ++q) sts128(dst + q * 16, make_float4(facc[q * 4], facc[q * 4 + 1], facc[q * 4 + 2], facc[q * 4 + 3]));
    }
    FTL(9);
    cg::cluster_group cluster = cg::this_cluster();
    if (nz == 1) __syncthreads(); else cluster.sync();
    FTL(6);

    // rows [rank * rows_per, +rows_per) of the tile belong to this CTA: thread -> float4 column c4 of rows row0, row0 + 32, ...
    const int rows_per = BM / nz;
    const int gw = Cout >> 2;                               // channels per GroupNorm group of the OUTPUT
    const int lg_lpg = gw >= BN ? 4 : (gw == 32 ? 3 : 2);   // lanes (float4 columns) per group inside the 64-column tile: 16, 8, 4
    const int gpt = 16 >> lg_lpg;                           // groups per tile: 1, 2, 4
    // statistics of the band: every thread turns its own (count, mean, M2) -- exact about a thread-local pivot -- into 64-bit
    // fixed-point contributions to (sum x, sum x^2); from there on everything is integer addition (warp shuffles, one shared
    // slot per warp and group, two global atomics per group and CTA): associative, so the result does not depend on any order.
    unsigned long long* wsum = reinterpret_cast<unsigned long long*>(wpart);      // [NTW][4 groups][2]
    if (warp < NTW) {
        const int c4 = (tid & 15) * 4, row0 = tid >> 4;
        int lr = rank * rows_per + row0;
        float* Yp = PW(y) + ((size_t)b * Ho * Wo + m0 + lr) * Cout + n0 + c4;
        const size_t ystep = (size_t)32 * Cout;
        uint32_t ra = red32 + (uint32_t)(lr * RED_LD + c4) * 4u;
        float pv = 0.f, s1 = 0.f, s2 = 0.f;
        int cnt = 0;
#pragma unroll 1
        for (int k = row0; k < rows_per; k += 32, lr += 32, ra += 32 * RED_LD * 4, Yp += ystep) {
            if (lr < rows_valid) {
                float4 acc;
                if (nz == 1 || KNOB(4)) {
                    acc = lds128(ra);
                } else {
                    // four DSMEM loads in flight per round (one remote-latency round per four K-slices); the additions keep the
                    // order of the slices
                    acc = ldc128(ra, 0);
                    const float4 q1 = ldc128(ra, 1);
                    if (nz >= 4) {
                        const float4 q2 = ldc128(ra, 2), q3 = ldc128(ra, 3);
                        acc.x += q1.x; acc.y += q1.y; acc.z += q1.z; acc.w += q1.w;
                        acc.x += q2.x; acc.y += q2.y; acc.z += q2.z; acc.w += q2.w;
                        acc.x += q3.x; acc.y += q3.y; acc.z += q3.z; acc.w += q3.w;
#pragma unroll 1
                        for (int z = 4; z < nz; z += 4) {
                            const float4 qa = ldc128(ra, z), qb = ldc128(ra, z + 1), qc = ldc128(ra, z + 2), qd = ldc128(ra, z + 3);
                            acc.x += qa.x; acc.y += qa.y; acc.z += qa.z; acc.w += qa.w;
                            acc.x += qb.x; acc.y += qb.y; acc.z += qb.z; acc.w += qb.w;
                            acc.x += qc.x; acc.y += qc.y; acc.z += qc.z; acc.w += qc.w;
                            acc.x += qd.x; acc.y += qd.y; acc.z += qd.z; acc.w += qd.w;
                        }
                    } else {
                        acc.x += q1.x; acc.y += q1.y; acc.z += q1.z; acc.w += q1.w;
                    }
                }
                *reinterpret_cast<float4*>(Yp) = acc;
                if (cnt == 0) pv = acc.x;
                const float d0 = acc.x - pv, d1 = acc.y - pv, d2 = acc.z - pv, d3 = acc.w - pv;
                s1 += (d0 + d1) + (d2 + d3);
                s2 += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
                cnt += 4;
            }
        }
        FTL(10);
        // sum x = n p + s1;  sum x^2 = s2 + 2 p s1 + n p^2   (double: exact to 2^-24 absolute after the scaling)
        const double dn = (double)cnt, dp = (double)pv, d1 = (double)s1;
        long long q1 = __double2ll_rn((dn * dp + d1) * FIX), q2 = __double2ll_rn(((double)s2 + 2.0 * dp * d1 + dn * dp * dp) * FIX);
        // lanes of one group: the 16 >> lg(gpt) float4 columns of both rows a warp covers per step
        q1 += __shfl_xor_sync(0xffffffffu, q1, 16); q2 += __shfl_xor_sync(0xffffffffu, q2, 16);
        if (lg_lpg > 3) { q1 += __shfl_xor_sync(0xffffffffu, q1, 8); q2 += __shfl_xor_sync(0xffffffffu, q2, 8); }
        if (lg_lpg > 2) { q1 += __shfl_xor_sync(0xffffffffu, q1, 4); q2 += __shfl_xor_sync(0xffffffffu, q2, 4); }
        q1 += __shfl_xor_sync(0xffffffffu, q1, 2); q2 += __shfl_xor_sync(0xffffffffu, q2, 2);
        q1 += __shfl_xor_sync(0xffffffffu, q1, 1); q2 += __shfl_xor_sync(0xffffffffu, q2, 1);
        FTL(11);
        if (lane < 16 && (lane & ((1 << lg_lpg) - 1)) == 0) {
            unsigned long long* w = wsum + (warp * 4 + (lane >> lg_lpg)) * 2;
            w[0] = (unsigned long long)q1; w[1] = (unsigned long long)q2;
        }
    }
    __syncthreads();
    FTL(12);
    if (tid < 2 * gpt) {
        const int gi = tid >> 1, g = gw >= BN ? (nt * BN) / gw : nt * gpt + gi;
        unsigned long long t = 0ull;
#pragma unroll
        for (int w = 0; w < NTW; ++w) t += wsum[(w * 4 + gi) * 2 + (tid & 1)];
        atomicAdd(PW(acc_out) + ((size_t)b * 4 + g) * 2 + (tid & 1), t);
    }
    if (L.done_flag != nullptr && warp == 0) {
        // outputs (stored before the barrier above), tape writes and the statistics atomics of this CTA are complete: release
        __syncwarp();
        if (lane == 0) {
            __threadfence();
            atomicAdd(L.done_flag, 1u);
        }
    }
    FTL(7);
    if (nz > 1) cluster.sync();
    FTL(8);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(ATM ? 512 : BN * NACC) : "memory");
}

// -------------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
struct alignas(64) TmHolder { CUtensorMap tm; };

// Bounded cache of tensor maps with POINTER-STABLE eviction.  Tapes come and go with the allocator, so the activation maps must be
// bounded; but a launch collects up to six map pointers before it dereferences them, and an eviction between two of those lookups
// must not free the earlier ones (the allocator reuses the first bytes of a freed holder at once: a corrupted tensor map, i.e. TMA
// loads from a wild address -- seen in round 2 as one core dump in five suite runs).  Eviction therefore works in two generations:
// holders evicted now are freed at the NEXT eviction, more than `bound` insertions later.  Checked on the CPU by
// dboa_selftest_map_cache (tests/test_cabi.py).
template <class Key>
struct MapCache {
    std::map<Key, TmHolder*> live;
    std::vector<TmHolder*> retired;
    size_t bound;
    explicit MapCache(size_t b) : bound(b) {}
    TmHolder* find(const Key& k) const {
        auto it = live.find(k);
        return it == live.end() ? nullptr : it->second;
    }
    TmHolder* insert(const Key& k) {                 // the caller fills the holder (or calls drop on failure)
        if (live.size() > bound) {
            for (TmHolder* h : retired) delete h;
            retired.clear();
            for (auto& kv : live) retired.push_back(kv.second);
            live.clear();
        }
        TmHolder* h = new TmHolder;
        live[k] = h;
        return h;
    }
    void drop(const Key& k) {
        auto it = live.find(k);
        if (it != live.end()) { delete it->second; live.erase(it); }
    }
};

static const CUtensorMap* weight_map(const float* w, int K, int Cout) {
    static std::map<std::tuple<const float*, int, int>, TmHolder*> cache;
    auto key = std::make_tuple(w, K, Cout);
    auto it = cache.find(key);
    if (it != cache.end()) return &it->second->tm;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return nullptr;
    TmHolder* h = new TmHolder;
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Cout};
    const cuuint64_t strides[1] = {(cuuint64_t)K * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BN};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&h->tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { delete h; return nullptr; }
    cache[key] = h;
    return &h->tm;
}
// weight matrix [Cout][K] read TRANSPOSED (data gradient: B[n = ci][k = co]): boxes of 32 input channels (contiguous) x 32 output
// channels with the 32-byte-atom swizzle = the MN-major TF32 operand layout of tcgen05
static const CUtensorMap* weight_map_mn(const float* w, int K, int Cout) {
    static std::map<std::tuple<const float*, int, int>, TmHolder*> cache;
    auto key = std::make_tuple(w, K, Cout);
    auto it = cache.find(key);
    if (it != cache.end()) return &it->second->tm;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return nullptr;
    TmHolder* h = new TmHolder;
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Cout};
    const cuuint64_t strides[1] = {(cuuint64_t)K * sizeof(float)};
    const cuuint32_t box[2] = {32, 32};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&h->tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { delete h; return nullptr; }
    cache[key] = h;
    return &h->tm;
}
// activation [B][H][W][C] as a 4-D tensor (C, W, H, B); box = 32 channels x W x bh rows x 1 sample, zero fill outside
// atom32: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B (32-byte chunks swizzled with the row index mod 4): the only shared-memory layout
// tcgen05 accepts for MN-major TF32 operands (UMMA layout type SWIZZLE_128B_BASE32B)
// stride: the box delivers bw x bh pixels sampled every `stride`-th pixel (boxDim = N * elementStride, as cuTensorMapEncodeTiled
// specifies for element strides other than one)
static const CUtensorMap* act_map(const float* x, int B, int H, int W, int C, int bw, int bh, bool atom32 = false, int stride = 1) {
    // 32768 maps = ~10 MB of host memory: a stream in steady state re-uses a few thousand (address, shape) pairs; with a bound of 4096
    // the one eviction while the allocator's addresses were still settling cost a 1.4 - 4.6 ms host stall around frame 16
    // (bench.py --frame-times)
    static MapCache<std::tuple<const float*, int, int, int, int, int, int, bool, int>> cache(32768);
    const auto key = std::make_tuple(x, B, H, W, C, bw, bh, atom32, stride);
    if (TmHolder* hit = cache.find(key)) return &hit->tm;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return nullptr;
    TmHolder* h = cache.insert(key);
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
    const cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(bw * stride), (cuuint32_t)(bh * stride), 1};
    const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    if (enc(&h->tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { cache.drop(key); return nullptr; }
    return &h->tm;
}

static int num_sms() {
    static int n = [] { int dev = 0, v = 148; if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); return v > 0 ? v : 148; }();
    return n;
}
static int rows_of(int Ho) { return Ho * Ho <= BM ? Ho : BM / Ho; }          // image rows per output tile (square images)

}  // namespace wz

// Host-only self test of the eviction rule (no CUDA call): `n` insertions into a cache of bound `bound`; like a launch, the caller
// keeps the pointers of its last `window` lookups and requires that they still carry the signature written into their first bytes
// (exactly the bytes a freed chunk loses to the allocator).  Returns 0, or 1 + the index of the first insertion after which a kept
// pointer was found corrupted.
int map_cache_selftest(int bound, int n, int window) {
    if (bound < 1 || n < 1 || window < 1 || window > 16 || window > bound) return -1;
    wz::MapCache<int> cache((size_t)bound);
    wz::TmHolder* kept[16];
    for (int i = 0; i < n; ++i) {
        wz::TmHolder* h = cache.insert(i);
        unsigned long long sig[2] = {0xD0B0A5EED0000000ull + (unsigned long long)i, ~(unsigned long long)i};
        memcpy(&h->tm, sig, sizeof sig);
        kept[i % window] = h;
        for (int j = 0; j < window && j <= i; ++j) {
            const int k = i - j;
            unsigned long long got[2];
            memcpy(got, &kept[k % window]->tm, sizeof got);
            if (got[0] != 0xD0B0A5EED0000000ull + (unsigned long long)k || got[1] != ~(unsigned long long)k) return 1 + i;
        }
        if (cache.find(i) != h) return 1 + i;
    }
    for (auto& kv : cache.live) delete kv.second;
    for (wz::TmHolder* h : cache.retired) delete h;
    return 0;
}

// shared with conv_wgrad_wide.cu / dgrad_wide.cu
const void* tma_weight_map_mn(const float* w, int K, int Cout) { return wz::weight_map_mn(w, K, Cout); }
const void* tma_act_map(const float* x, int B, int H, int W, int C, int bw, int bh, bool atom32, int stride) { return wz::act_map(x, B, H, W, C, bw, bh, atom32, stride); }

bool conv_wide_ok(const FusedConv& d) {
    return d.Cin % 64 == 0 && d.Cout % 64 == 0 && (d.k == 1 || d.k == 3) && (d.stride == 1 || d.stride == 2) && d.pad == d.k / 2 && d.mode >= 0 &&
           d.mode <= 3 && d.Ho <= wz::BM && d.Hi == d.Ho * d.stride && !(d.a_out != nullptr && d.k == 1 && d.stride == 2);
}

// cluster size (K-slices): largest power of two <= 16 that keeps the launch inside one wave of one CTA per SM (thread-block
// clusters of 4 can use 132 SMs, of 8 / 16 only 128: B300_MICROARCH.md) with at least `min_kb` k-blocks per slice
// CTA budget of a launch (default: every SM).  Two forwards that run side by side on different streams (student / teacher,
// output forward next to the following frame's adaptation) are given half the SMs each: a launch owns its SMs (one CTA of
// ~150-200 KB shared memory per SM), so two full-width launches would simply alternate.
// Measured (bench.py, C2, 1 x B200): 143.3 frames/s with all 148 SMs per launch, 151.8 with 96, 151.2 with 74, 148.1 with 64; the
// isolated forward is also slightly faster with fewer K-slices (0.831 vs 0.855 ms).  Default 96; DBOA_FUSED_MAX_CTAS overrides.
// activation operand of the fused kernels in tensor memory (DBOA_OPERAND_TMEM=0 / dboa_set_operand_tmem(0): all-shared-memory variant)
static bool g_operand_tmem = [] { const char* e = getenv("DBOA_OPERAND_TMEM"); return e ? e[0] != '0' : true; }();
void conv_wide_set_operand_tmem(bool on) { g_operand_tmem = on; }
bool conv_wide_operand_tmem() { return g_operand_tmem; }
static int fused_cta_budget_default() { const char* e = getenv("DBOA_FUSED_MAX_CTAS"); return e ? atoi(e) : 96; }
static int fused_min_kb_default() { const char* e = getenv("DBOA_FUSED_MINKB"); return e ? atoi(e) : 2; }
static int fused_max_nz_default() { const char* e = getenv("DBOA_FUSED_MAX_NZ"); return e ? atoi(e) : 16; }
static int g_cta_budget = fused_cta_budget_default();
static int g_min_kb = clamp_split(fused_min_kb_default(), 1, 1 << 30);     // k-blocks a K-slice must at least hold
static int g_max_nz = clamp_split(fused_max_nz_default(), 1, 16);           // largest cluster (K-slices of one tile)
void conv_wide_set_cta_budget(int n) { g_cta_budget = n; }
void conv_wide_set_limits(int max_ctas, int max_nz, int min_kb) {
    g_cta_budget = max_ctas < 0 ? fused_cta_budget_default() : max_ctas;
    g_max_nz = clamp_split(max_nz < 0 ? fused_max_nz_default() : max_nz, 1, 16);
    g_min_kb = clamp_split(min_kb < 0 ? fused_min_kb_default() : min_kb, 1, 1 << 30);
}
int conv_wide_plan(const FusedConv* d, int nprob, int B) {
    int tiles = 0;
    for (int i = 0; i < nprob; ++i) tiles += B * ceil_div(d[i].Ho, wz::rows_of(d[i].Ho)) * (d[i].Cout / wz::BN);
    const int nkb = d[0].k * d[0].k * d[0].Cin / wz::BK;
    int nz = 1;
    // the budget limits how far a launch with FEW tiles is split; a launch whose tiles alone exceed it (large batches) may still
    // split up to the hardware wave, which halves its accumulation chains
    auto cap = [tiles](int c) {
        const int hw = c <= 2 ? wz::num_sms() : (c == 4 ? (wz::num_sms() * 132) / 148 : (wz::num_sms() * 128) / 148);
        const int soft = g_cta_budget > 2 * tiles ? g_cta_budget : 2 * tiles;
        return g_cta_budget > 0 && soft < hw ? soft : hw;
    };
    while (nz < g_max_nz && tiles * nz * 2 <= cap(nz * 2) && nkb / (nz * 2) >= g_min_kb) nz *= 2;
    while (nz > 1 && (nz - 1) * ceil_div(nkb, nz) >= nkb) nz >>= 1;
    return nz;
}

// split-K plan of the most recent launch of each wide kernel (dboa_last_wide_plan): one host store per launch
static WidePlan g_last_plan[3];
void wide_plan_note(int kernel, int nz, int per, int D, int grid, int nkb) {
    g_last_plan[kernel] = WidePlan{nz, per, D, grid, nkb - (nz - 1) * per};
}
bool wide_plan_last(int kernel, long long out[5]) {
    if (kernel < 0 || kernel > 2) return false;
    const WidePlan& p = g_last_plan[kernel];
    out[0] = p.nz; out[1] = p.per; out[2] = p.D; out[3] = p.grid; out[4] = p.last;
    return true;
}

#ifdef DBOA_TIMELINE
static int g_wide_launch_id = 0;
extern "C" int dboa_debug_set_fused_knobs(int knobs) { return cudaMemcpyToSymbol(wz::g_knobs, &knobs, sizeof(knobs)) == cudaSuccess ? 0 : -3; }
extern "C" int dboa_debug_set_fused_timeline(unsigned long long* buf) {
    g_wide_launch_id = 0;
    return cudaMemcpyToSymbol(wz::g_ftl, &buf, sizeof(buf)) == cudaSuccess ? 0 : -3;
}
#endif

int conv_wide_launch(const FusedConv* d, int nprob, int B, int nz, const float* next_w, size_t next_bytes, cudaStream_t st, bool pdl,
                     const ChainDep* dep) {
    if (nprob < 1 || nprob > 2 || B < 1) return DBOA_ERR_ARG;
    wz::Launch L;
    memset(&L, 0, sizeof L);
    const CUtensorMap *tmx[2] = {nullptr, nullptr}, *tmw[2] = {nullptr, nullptr}, *tmr[2] = {nullptr, nullptr};
    const int K0 = d[0].k * d[0].k * d[0].Cin;
    const int nkb = K0 / wz::BK, per = ceil_div(nkb, nz);
    if (nz < 1 || nz > 16 || (nz & (nz - 1)) || (nz - 1) * per >= nkb) return DBOA_ERR_ARG;
    int total = 0, tabc = 0;
    for (int i = 0; i < nprob; ++i) {
        const FusedConv& c = d[i];
        if (!conv_wide_ok(c) || c.mode != d[0].mode || c.k * c.k * c.Cin != K0) return DBOA_ERR_UNSUPPORTED;
        if (i == 1 && (c.x != d[0].x || c.res != d[0].res || c.Hi != d[0].Hi || c.Cin != d[0].Cin)) return DBOA_ERR_UNSUPPORTED;    // one `res` map
        wz::Problem& p = L.p[i];
        p.a_out = c.a_out; p.stats_out = c.stats_out; p.stats2_out = c.stats2_out;
        p.acc_in = reinterpret_cast<const long long*>(c.part_in); p.acc2_in = reinterpret_cast<const long long*>(c.part2_in);
        p.gamma = c.gamma; p.beta = c.beta; p.gamma2 = c.gamma2; p.beta2 = c.beta2;
        p.y = c.y; p.acc_out = reinterpret_cast<unsigned long long*>(c.part_out);
        p.Hi = c.Hi; p.Wi = c.Hi; p.Cin = c.Cin; p.Ho = c.Ho; p.Wo = c.Ho; p.Cout = c.Cout; p.k = c.k; p.pad = c.pad; p.stride = c.stride;
        p.bh = wz::rows_of(c.Ho); p.tps = ceil_div(c.Ho, p.bh); p.ntiles = c.Cout / wz::BN; p.nclusters = B * p.tps * p.ntiles;
        total += p.nclusters;
        const int tcn = c.k == 1 ? per * wz::BK : c.Cin;
        if (c.mode >= 1 && tcn > tabc) tabc = tcn;
        tmw[i] = wz::weight_map(c.w, K0, c.Cout);
        tmx[i] = wz::act_map(c.x, B, c.Hi, c.Hi, c.Cin, c.Ho, p.bh, false, c.stride);
        tmr[i] = c.mode >= 2 ? wz::act_map(c.res, B, c.Hi, c.Hi, c.Cin, c.Ho, p.bh, false, c.stride) : tmx[i];
        if (tmw[i] == nullptr || tmx[i] == nullptr || tmr[i] == nullptr) return DBOA_ERR_CUDA;
    }
    if (nprob == 1) { tmx[1] = tmx[0]; tmw[1] = tmw[0]; tmr[1] = tmr[0]; }
    L.nprob = nprob; L.nz = nz; L.per = per; L.tabc = tabc;
    L.next_w = next_w; L.next_bytes = (unsigned long long)next_bytes;
#ifdef DBOA_TIMELINE
    L.launch_id = g_wide_launch_id++;
#endif
    const int ntab = d[0].mode == 3 ? 4 : (d[0].mode >= 1 ? 2 : 0);
    const size_t slot = (size_t)wz::A_TILE * (d[0].mode >= 2 ? 2 : 1) + wz::B_TILE;
    const size_t fixed = 2 * (size_t)(wz::A_TILE + wz::B_TILE) + (size_t)ntab * tabc * sizeof(float) + 2048 + 1024;     // + barriers / scratch + alignment slack
    int D = per < wz::DMAX ? per : wz::DMAX;
    while (D > 1 && fixed + (size_t)D * slot > 227 * 1024) --D;
    L.D = D;
    const size_t smem = fixed + (size_t)D * slot;
    if (smem > 227 * 1024) return DBOA_ERR_SHAPE;
    const dim3 grid(total * nz), block(wz::NT), cl(nz, 1, 1);
    wide_plan_note(0, nz, per, D, (int)grid.x, nkb);
    if (dep != nullptr) {
        // mode 0 has no statistics barrier behind which the other transform threads could be ordered: every thread waits there
        L.dep_flag = pdl ? dep->wait_flag : nullptr; L.dep_expect = dep->wait_count; L.done_flag = dep->signal_flag;
        if (dep->signal_count != nullptr) *dep->signal_count = grid.x;
    }
#define DBOA_WIDE_LAUNCH(M)                                                                                                                          \
    (g_operand_tmem ? launch_ex(wz::conv_wide_kernel<M, true>, grid, block, smem, st, cl, pdl, L, *tmx[0], *tmx[1], *tmr[0], *tmr[1], *tmw[0], *tmw[1]) \
                    : launch_ex(wz::conv_wide_kernel<M, false>, grid, block, smem, st, cl, pdl, L, *tmx[0], *tmx[1], *tmr[0], *tmr[1], *tmw[0], *tmw[1]))
    switch (d[0].mode) {
        case 0: return DBOA_WIDE_LAUNCH(0);
        case 1: return DBOA_WIDE_LAUNCH(1);
        case 2: return DBOA_WIDE_LAUNCH(2);
        default: return DBOA_WIDE_LAUNCH(3);
    }
#undef DBOA_WIDE_LAUNCH
}

// -------------------------------------------------------------------------------------------------
// GroupNorm apply from the fixed-point statistics (+ residual, ReLU) fused with the 7x7 average pool: the last layer of the
// backbone (reference model/hmr.py:57-60 of layer4.2, :156-157).  grid (C / 128, B), 256 threads.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gn_acc_res_avgpool_kernel(const float* __restrict__ y, const float* __restrict__ res, const long long* __restrict__ acc,
                                                                  const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                  float* __restrict__ a_out, float* __restrict__ stats_out, float* __restrict__ out, int HW,
                                                                  int C, int ld, int ncopy, size_t copy_stride) {
    __shared__ float4 part[8][32];
    __shared__ float sst[8];
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 4) {
        const long long* a = acc + ((size_t)b * 4 + threadIdx.x) * 2;
        const double N = (double)HW * (C >> 2);
        const double s1 = (double)__ldcg(a) / wz::FIX, s2 = (double)__ldcg(a + 1) / wz::FIX;
        const double mu = s1 / N, var = fmax(s2 / N - mu * mu, 0.0);
        sst[threadIdx.x] = (float)mu;
        sst[4 + threadIdx.x] = 1.0f / sqrtf((float)var + wz::GN_EPS);
    }
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x < 8 && stats_out != nullptr) stats_out[(b * 4 + (threadIdx.x & 3)) * 2 + (threadIdx.x >> 2)] = sst[threadIdx.x];
    const int c = blockIdx.x * 128 + lane * 4, g = c / (C >> 2);
    const float mu = sst[g], rs = sst[4 + g];
    const float4 ga = ldg4(gamma + c), be = ldg4(beta + c);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = warp; p < HW; p += 8) {
        const size_t off = ((size_t)b * HW + p) * C + c;
        const float4 v = ldg4(y + off), r = ldg4(res + off);
        float4 o;
        o.x = (v.x - mu) * (rs * ga.x) + be.x; o.y = (v.y - mu) * (rs * ga.y) + be.y;
        o.z = (v.z - mu) * (rs * ga.z) + be.z; o.w = (v.w - mu) * (rs * ga.w) + be.w;
        o.x = fmaxf(o.x + r.x, 0.f); o.y = fmaxf(o.y + r.y, 0.f); o.z = fmaxf(o.z + r.z, 0.f); o.w = fmaxf(o.w + r.w, 0.f);
        *reinterpret_cast<float4*>(a_out + off) = o;
        s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
    }
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0) {
        float4 t = part[0][lane];
        for (int w = 1; w < 8; ++w) { const float4 q = part[w][lane]; t.x += q.x; t.y += q.y; t.z += q.z; t.w += q.w; }
        const float hw = (float)HW;
        t.x /= hw; t.y /= hw; t.z /= hw; t.w /= hw;
        for (int k = 0; k < ncopy; ++k) *reinterpret_cast<float4*>(out + k * copy_stride + (size_t)b * ld + c) = t;
    }
}
int gn_acc_res_avgpool(const float* y, const float* res, const float* acc, const float* gamma, const float* beta, float* a_out, float* stats_out,
                       float* out, int B, int HW, int C, int ld, int ncopy, size_t copy_stride, cudaStream_t st) {
    if (C % 128 != 0 || ld % 4 != 0 || copy_stride % 4 != 0) return DBOA_ERR_SHAPE;
    return launch_ex(gn_acc_res_avgpool_kernel, dim3(C / 128, B), dim3(256), 0, st, dim3(1, 1, 1), true, y, res, reinterpret_cast<const long long*>(acc), gamma,
                     beta, a_out, stats_out, out, HW, C, ld, ncopy, copy_stride);
}

// statistics of a materialised-elsewhere tensor are not available in fixed point: (sum, sum of squares) of y [B][HW][C] per
// (sample, group) for a layer that ran on the unfused kernels -- not needed (those layers hand over a materialised activation)

}  // namespace dboa
