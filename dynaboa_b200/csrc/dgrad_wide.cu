// Fused data gradient of a stride-1 backbone convolution on tcgen05 tensor cores (the backward mirror of conv_wide.cu):
//
//      dy   = GroupNorm_c backward of dz          (on load: dy = rstd (dz gamma - m1 - x^ m2), x^ = (y - mean) rstd)
//      dX   = conv_c^T(dy)  [+ addend]            (implicit GEMM: rows = input pixels, K = (tap, co), flipped taps)
//      dz_p = dX * (a_p > 0)                      (epilogue: ReLU mask of the producing layer p)
//      sums of GroupNorm_p's backward            (epilogue: sum q, sum q x^ per (sample, group); d gamma, d beta per channel)
//
// Replaces, per layer, the launches  gn_bwd_fused -> conv dgrad (-> relu_mask)  of round 1 (reference: the autograd backward of
// nn.GroupNorm / ReLU / nn.Conv2d / the residual add in Bottleneck.forward, model/hmr.py:40-60, under MAML.adapt / loss.backward(),
// dynaboa_benchmark.py:140,150): GroupNorm backward needs two group-wide sums before it can produce dy, so round 1 ran it as its
// own cluster kernel (53 launches of ~10 us on the critical chain of every backward).  Here those sums are produced by the
// epilogue of the kernel that creates dz (this kernel, one layer later in the chain), as 64-bit fixed-point atomics (exact, order
// independent -> deterministic), and GroupNorm backward itself happens while the operand tile is in shared memory.
//   * A operand (dz and y of layer c): two 4-D TMA boxes per k-block, K-major 128B swizzle; one designated tap also writes dy to
//     memory, because the weight-gradient kernel (side stream) reads it;
//   * B operand (W_c^T): W[co][tap][ci] is ci-contiguous, i.e. MN-major for this GEMM; TMA boxes of 32 ci x 32 co with the
//     128B / 32-byte-atom swizzle feed tcgen05 directly (instruction descriptor b_major = MN) -- no transposing store;
//   * TF32x3 split and GroupNorm-backward transform: one elementwise pass over the landed tiles (16 warps);
//   * split-K over a thread-block cluster, DSMEM reduction (as conv_wide.cu).
// Stride-2 layers stay on conv_tc.cu + groupnorm.cu (hmr_plan.cu stitches the two worlds with gn_bwd_prep below).
#include <cooperative_groups.h>
#include <cuda.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace dboa {
const void* tma_act_map(const float* x, int B, int H, int W, int C, int bw, int bh, bool atom32, int stride);      // conv_wide.cu
const void* tma_weight_map_mn(const float* w, int K, int Cout);                                         // conv_wide.cu

namespace dz {

constexpr int BM = 128, BN = 64, BK = 32;
constexpr int NTW = 16, NTT = NTW * 32, W_MMA = 16, W_TMA = 17, NT = 576;
constexpr int DMAX = 3;
constexpr int NACC = 4;                                  // TMEM accumulators a reduction chain rotates over (see conv_wide.cu)
constexpr uint32_t A_TILE = BM * BK * 4, B_TILE = BN * BK * 4;          // 16 KB, 8 KB (2 atoms of 32 ci x 32 co)
constexpr uint32_t SLOT = 2 * A_TILE + B_TILE;                          // dz tile, y tile, weight tile
constexpr int RED_LD = BN + 4;
constexpr double FIX = 268435456.0;                                     // 2^28 fixed point of the backward sums

struct Prep {                      // GroupNorm whose backward the epilogue prepares (layer p = producer of this conv's input)
    const float* y;                // raw output of layer p [B][H][W][C]
    const float* stats;            // (mean, rstd) [B][4][2]
    const float* gamma;
    unsigned long long* sums;      // [B][4][2]: sum q, sum q x^
    unsigned long long* dgb;       // [C][2]: d gamma, d beta
};
struct Launch {
    // GroupNorm_c backward on load
    const float* stats_c; const long long* sums_c; const float* gamma_c;
    float* dy_out;                 // materialised dy_c [B][H][W][Cout] (weight gradient operand) or NULL
    // output side
    const float* addend;           // [B][H][W][Cin] or NULL
    float* out;                    // plain mode: dX; prep mode: dz_p
    const float* mask;             // prep mode: a_p (post-activation output of layer p); NULL = plain mode
    Prep p[2];
    int nprep;
    int H, W, Cin, Cout, k, pad, B;
    int bh, tps, ntiles, nz, per, D, tabc, accumulate;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) {       // K-major, 128B swizzle (activations)
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)((1024 >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// MN-major TF32 (weights): SWIZZLE_128B_BASE32B, LBO = 4096 B between the two 32-channel atoms, SBO = 512 B between 4-row groups
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((4096 >> 4) & 0x3FFF) << 16) | ((uint64_t)((512 >> 4) & 0x3FFF) << 32) | (1ull << 46) |
           (1ull << 61);
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
// A operand from tensor memory, 8-column tensor-memory store of a thread's lane (see conv_wide.cu)
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
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
        else if (clock64() - t0 > 4000000000ll) __trap();       // a protocol error fails the launch instead of hanging the device
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
// shared memory through 32-bit shared-window addresses (see conv_wide.cu: the integer carve-up would otherwise cost generic LD/ST)
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, const float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
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
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
__device__ __forceinline__ long long to_fix(float v) { return __double2ll_rn((double)v * FIX); }

// ATM: the transformed operand dy (hi and lo parts) lives in tensor memory instead of shared memory (conv_wide.cu explains why)
template <bool ATM>
__global__ void __launch_bounds__(NT, 1) dgrad_wide_kernel(const __grid_constant__ Launch L, const __grid_constant__ CUtensorMap tmdz,
                                                           const __grid_constant__ CUtensorMap tmy, const __grid_constant__ CUtensorMap tmw) {
    extern __shared__ uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nz = L.nz, D = L.D;
    const int cidx = blockIdx.x / nz, rank = blockIdx.x - cidx * nz;
    const int H = L.H, W = L.W, Cin = L.Cin, Cout = L.Cout, ks = L.k, pad = L.pad, bh = L.bh;
    const int nt = cidx % L.ntiles, bm = cidx / L.ntiles, mt = bm % L.tps, b = bm / L.tps;
    const int h0 = mt * bh, n0 = nt * BN;
    const int rows_valid = min(bh, H - h0) * W, m0 = h0 * W;
    const int nkb_total = (ks * ks * Cout) / BK;
    const int kb_begin = rank * L.per;
    const int nkb = max(0, min(L.per, nkb_total - kb_begin));
    const uint32_t a_bytes = (uint32_t)(bh * W) * 128u;

    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* slots = base;                                  // D x {dz 16 KB, y 16 KB, W^T 8 KB}
    uint8_t* lo_a = slots + (size_t)D * SLOT;               // 2 x 16 KB
    uint8_t* lo_b = lo_a + 2 * A_TILE;                      // 2 x 8 KB
    float* tab = reinterpret_cast<float*>(lo_b + 2 * B_TILE);          // gamma_c of this CTA's channel range
    uint64_t* bars = reinterpret_cast<uint64_t*>(tab + L.tabc);
    uint64_t* s_full = bars;               // [DMAX]
    uint64_t* s_empty = bars + DMAX;       // [DMAX]
    uint64_t* l_full = bars + 2 * DMAX;    // [2]
    uint64_t* l_empty = l_full + 2;        // [2]
    uint64_t* done = l_empty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    float* sstat = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 128);                     // [16]: mean, rstd, m1, m2 per group
    float* red = reinterpret_cast<float*>(lo_a);

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
    // gamma of layer c for the output channels this CTA reduces over (parameters: no dependency on the previous kernel)
    const int tc0 = ks == 1 ? kb_begin * BK : 0, tcn = ks == 1 ? nkb * BK : Cout;
    for (int i = tid; i < tcn; i += NT) tab[i] = __ldg(L.gamma_c + tc0 + i);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    // k-block kb: filter tap (r, s) and output-channel offset c
    auto tap_of = [&](int kb, int& r, int& s, int& c) {
        const int k0 = kb * BK, tap = k0 / Cout;
        c = k0 - tap * Cout; r = tap / ks; s = tap - r * ks;
    };

    if (warp == W_TMA) {
        if (lane == 0 && nkb > 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmw)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmdz)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmy)) : "memory");
            auto load_w = [&](int it, int sl) {             // W^T tile: 2 boxes of 32 ci x 32 co at (tap * Cin + n0 + 32 j, co)
                int r, s, c;
                tap_of(kb_begin + it, r, s, c);
                uint8_t* wt = slots + (size_t)sl * SLOT + 2 * A_TILE;
                tma_load_2d(smem_u32(wt), &tmw, (r * ks + s) * Cin + n0, c, &s_full[sl]);
                tma_load_2d(smem_u32(wt + 4096), &tmw, (r * ks + s) * Cin + n0 + 32, c, &s_full[sl]);
            };
            const int npre = min(nkb, D);
            for (int it = 0; it < npre; ++it) {
                mbar_expect_tx(&s_full[it], 2 * a_bytes + B_TILE);
                load_w(it, it);
            }
            pdl_wait();
            pdl_trigger();
            for (int it = 0; it < nkb; ++it) {
                const int sl = it % D;
                uint8_t* slot = slots + (size_t)sl * SLOT;
                if (it >= D) {
                    mbar_wait(&s_empty[sl], (uint32_t)(((it / D) - 1) & 1));
                    mbar_expect_tx(&s_full[sl], 2 * a_bytes + B_TILE);
                    load_w(it, sl);
                }
                int r, s, c;
                tap_of(kb_begin + it, r, s, c);
                // dX[hi][wi] += dy[hi + pad - r][wi + pad - s] W[co][r][s][ci]: the box starts at (pad - s, h0 + pad - r)
                tma_load_4d(smem_u32(slot), &tmdz, c, pad - s, h0 + pad - r, b, &s_full[sl]);
                tma_load_4d(smem_u32(slot + A_TILE), &tmy, c, pad - s, h0 + pad - r, b, &s_full[sl]);
            }
        } else {
            pdl_wait();
            pdl_trigger();
        }
    } else if (warp == W_MMA) {
        // warp-uniform loop, one elected lane issues (see conv_wide.cu)
        if (nkb > 0) {
            // D = F32, A = B = TF32, A K-major, B MN-major (bit 16), N >> 3, M >> 4
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint64_t dslot = desc_sw128(smem_u32(slots)), dloa = desc_sw128(smem_u32(lo_a));
            const uint64_t dwslot = desc_mn(smem_u32(slots + 2 * A_TILE)), dlob = desc_mn(smem_u32(lo_b));
            constexpr uint64_t KSTEP_A = 32 >> 4;            // 8 channels = 32 bytes inside the 128-byte row
            constexpr uint64_t KSTEP_B = 1024 >> 4;          // 8 output channels = 8 rows of the MN-major tile
            int sl = 0;
#pragma unroll 1
            for (int it = 0; it < nkb; ++it) {
                const int ls = it & 1;
                mbar_wait(&l_full[ls], (uint32_t)((it >> 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t so = (uint64_t)(sl * (SLOT >> 4));
                const uint64_t dah = dslot + so, dbh = dwslot + so;
                const uint64_t dal = dloa + (uint64_t)(ls * (A_TILE >> 4)), dbl = dlob + (uint64_t)(ls * (B_TILE >> 4));
                const uint32_t dacc = tmem_d + (uint32_t)((it & (NACC - 1)) * BN);      // truncating accumulation: short chains
                const uint32_t first = it >= NACC ? 1u : 0u;
                if (elect_one()) {
                    if constexpr (ATM) {
                        const uint32_t tah = tmem_d + (uint32_t)(BN * NACC + ls * 2 * BK), tal = tah + (uint32_t)BK;
#pragma unroll
                        for (int kk = 0; kk < BK / 8; ++kk) {
                            mma_tf32_ts(dacc, tah + kk * 8, dbh + kk * KSTEP_B, idesc, kk > 0 ? 1u : first);
                            mma_tf32_ts(dacc, tah + kk * 8, dbl + kk * KSTEP_B, idesc, 1u);
                            mma_tf32_ts(dacc, tal + kk * 8, dbh + kk * KSTEP_B, idesc, 1u);
                        }
                    } else {
#pragma unroll
                        for (int kk = 0; kk < BK / 8; ++kk) {
                            mma_tf32(dacc, dah + kk * KSTEP_A, dbh + kk * KSTEP_B, idesc, kk > 0 ? 1u : first);
                            mma_tf32(dacc, dah + kk * KSTEP_A, dbl + kk * KSTEP_B, idesc, 1u);
                            mma_tf32(dacc, dal + kk * KSTEP_A, dbh + kk * KSTEP_B, idesc, 1u);
                        }
                    }
                    umma_commit(&l_empty[ls]);
                    umma_commit(&s_empty[sl]);
                }
                __syncwarp();
                if (++sl == D) sl = 0;
            }
            if (elect_one()) umma_commit(done);
        }
        pdl_wait();
        pdl_trigger();
    } else {
        // ---- transform warps: GroupNorm_c backward + TF32 split of (dz, y) -> dy hi / lo; split of the weight tile
        // ATM: thread = tile row (= its TMEM lane) x 16 channels kh * 16 .. + 15 of every second k-block; only entry 0 of the per-row arrays is used
        const int r0 = ATM ? (warp & 3) * 32 + lane : tid >> 3, pc = tid & 7, lc = pc ^ (r0 & 7), kh = (warp >> 2) & 1, grp = warp >> 3;
        float* dyb = (L.dy_out != nullptr && nt == 0) ? L.dy_out + (size_t)b * H * W * Cout : nullptr;
        int hq[2], wq[2];                                   // pixel of layer c's output the two rows read at tap (0, 0)
        bool rowok[2];
        float* dyq[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int i = r0 + 64 * q, oh = i / W, ow = i - oh * W;
            hq[q] = h0 + oh + pad; wq[q] = ow + pad; rowok[q] = i < rows_valid;
            dyq[q] = dyb + ((long long)hq[q] * W + wq[q]) * Cout + (ATM ? kh * 16 : lc * 4);       // only dereferenced for in-bounds taps
        }
        int lgw = 0;
        while ((4 << lgw) < Cout) ++lgw;
        const double inv_nfix = 1.0 / ((double)H * W * (Cout >> 2) * FIX);      // before the wait: no division after it
        int r, s, c;
        tap_of(kb_begin, r, s, c);
        pdl_wait();
        pdl_trigger();
        // dy = rstd (dz gamma - m1 - x^ m2) = dz * A_c - (y - mean) * B_g + C_g  with A_c = gamma_c rstd, B_g = rstd^2 m2, C_g = -rstd m1
        if (tid < 4) {
            const float* st = L.stats_c + ((size_t)b * 4 + tid) * 2;
            const long long* sm = L.sums_c + ((size_t)b * 4 + tid) * 2;
            const float mu = __ldcg(st), rs = __ldcg(st + 1);
            const float m1 = (float)((double)__ldcg(sm) * inv_nfix), m2 = (float)((double)__ldcg(sm + 1) * inv_nfix);
            sstat[tid] = mu; sstat[4 + tid] = rs * rs * m2; sstat[8 + tid] = -rs * m1; sstat[12 + tid] = rs;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NTT) : "memory");
        for (int i = tid; i < tcn; i += NTT) tab[i] *= sstat[12 + ((tc0 + i) >> lgw)];
        asm volatile("bar.sync 1, %0;" ::"n"(NTT) : "memory");
        int sl = 0;
        uint32_t ph_full = 0;
        const uint32_t offA = (uint32_t)tid * 16u;
        const uint32_t slots32 = smem_u32(slots) + offA, tab32 = smem_u32(tab), st32 = smem_u32(sstat);
        const uint32_t lo_a32 = smem_u32(lo_a) + offA, lo_b32 = smem_u32(lo_b) + offA;
        uint32_t slot = slots32;
        if constexpr (ATM) {
            // two groups of 8 warps alternate k-blocks (conv_wide.cu): thread = row r0 x 16 channels (logical chunks 4 kh .. 4 kh + 3)
            // + float4 tg and tg + 256 of the weight tile; group g owns stage g of the TMEM operand and of the weight lo tile
            const uint32_t rowofs = (uint32_t)r0 * 128u, sw = (uint32_t)(r0 & 7);
            uint32_t pa[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pa[j] = rowofs + (((uint32_t)(4 * kh + j) ^ sw) << 4);
            const uint32_t ta = tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(BN * NACC + grp * 2 * BK + kh * 16);
            const uint32_t offW = (uint32_t)((warp & 7) * 32 + lane) * 16u;
            const uint32_t lob = smem_u32(lo_b) + (uint32_t)grp * B_TILE + offW;
            const uint32_t sl0 = smem_u32(slots);
            auto step = [&]() { c += BK; if (c >= Cout) { c = 0; if (++s == ks) { s = 0; ++r; } } };
            if (grp == 1) step();
            int sl = grp % D;
            uint32_t ph_full = (uint32_t)((grp / D) & 1);
            uint32_t sbase = sl0 + (uint32_t)sl * SLOT;
#pragma unroll 1
            for (int it = grp; it < nkb; it += 2) {
                const int cch = c + kh * 16;                     // 16 channels of one GroupNorm group (groups are >= 16 channels wide)
                const uint32_t sg = st32 + (uint32_t)(cch >> lgw) * 4u;
                const uint32_t tg = tab32 + (uint32_t)(cch - tc0) * 4u;
                const float mu = lds32(sg), gb = lds32(sg + 16), gc = lds32(sg + 32);
                const bool desig = dyb != nullptr && (ks == 1 || (r == 1 && s == 1));
                const int tapoff = c - (r * W + s) * Cout;
                const bool in0 = rowok[0] && (unsigned)(hq[0] - r) < (unsigned)H && (unsigned)(wq[0] - s) < (unsigned)W;
                mbar_wait(&s_full[sl], ph_full);
                float4 d[4], y[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) d[j] = lds128(sbase + pa[j]);
#pragma unroll
                for (int j = 0; j < 4; ++j) y[j] = lds128(sbase + A_TILE + pa[j]);
                const float4 w0 = lds128(sbase + 2 * A_TILE + offW), w1 = lds128(sbase + 2 * A_TILE + offW + 4096u);
                float4 h[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 ga = lds128(tg + 16 * j);
                    float4 o;
                    o.x = fmaf(mu - y[j].x, gb, fmaf(d[j].x, ga.x, gc)); o.y = fmaf(mu - y[j].y, gb, fmaf(d[j].y, ga.y, gc));
                    o.z = fmaf(mu - y[j].z, gb, fmaf(d[j].z, ga.z, gc)); o.w = fmaf(mu - y[j].w, gb, fmaf(d[j].w, ga.w, gc));
                    if (!in0) o = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (desig && in0) *reinterpret_cast<float4*>(dyq[0] + tapoff + 4 * j) = o;
                    h[j] = make_float4(tf32_hi(o.x), tf32_hi(o.y), tf32_hi(o.z), tf32_hi(o.w));
                    d[j] = make_float4(o.x - h[j].x, o.y - h[j].y, o.z - h[j].z, o.w - h[j].w);
                }
                const float4 hw0 = make_float4(tf32_hi(w0.x), tf32_hi(w0.y), tf32_hi(w0.z), tf32_hi(w0.w));
                const float4 hw1 = make_float4(tf32_hi(w1.x), tf32_hi(w1.y), tf32_hi(w1.z), tf32_hi(w1.w));
                // the MMAs of k-block it - 2 (the previous user of this group's TMEM / lo stage) must have completed
                if (it >= 2) mbar_wait(&l_empty[grp], (uint32_t)(((it >> 1) - 1) & 1));
                tmem_st8(ta, h[0], h[1]);
                tmem_st8(ta + 8, h[2], h[3]);
                tmem_st8(ta + BK, d[0], d[1]);
                tmem_st8(ta + BK + 8, d[2], d[3]);
                sts128(sbase + 2 * A_TILE + offW, hw0);
                sts128(sbase + 2 * A_TILE + offW + 4096u, hw1);
                sts128(lob, make_float4(w0.x - hw0.x, w0.y - hw0.y, w0.z - hw0.z, w0.w - hw0.w));
                sts128(lob + 4096u, make_float4(w1.x - hw1.x, w1.y - hw1.y, w1.z - hw1.z, w1.w - hw1.w));
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&l_full[grp]);
                sl += 2;
                while (sl >= D) { sl -= D; ph_full ^= 1u; }
                sbase = sl0 + (uint32_t)sl * SLOT;
                step(); step();
            }
        } else {
#pragma unroll 1
        for (int it = 0; it < nkb; ++it) {
            const int ls = it & 1;
            const int cch = c + lc * 4;
            const uint32_t sg = st32 + (uint32_t)(cch >> lgw) * 4u;
            const float4 ga = lds128(tab32 + (uint32_t)(cch - tc0) * 4u);
            const float mu = lds32(sg), gb = lds32(sg + 16), gc = lds32(sg + 32);
            const bool desig = dyb != nullptr && (ks == 1 || (r == 1 && s == 1));
            const int tapoff = c - (r * W + s) * Cout;
            mbar_wait(&s_full[sl], ph_full);
            if (it >= 2) mbar_wait(&l_empty[ls], (uint32_t)(((it >> 1) - 1) & 1));
            const float4 d0 = lds128(slot), d1 = lds128(slot + NTT * 16u);
            const float4 y0 = lds128(slot + A_TILE), y1 = lds128(slot + A_TILE + NTT * 16u);
            const float4 vw = lds128(slot + 2 * A_TILE);
            const bool in0 = rowok[0] && (unsigned)(hq[0] - r) < (unsigned)H && (unsigned)(wq[0] - s) < (unsigned)W;
            const bool in1 = rowok[1] && (unsigned)(hq[1] - r) < (unsigned)H && (unsigned)(wq[1] - s) < (unsigned)W;
            float4 o0, o1;
            o0.x = fmaf(mu - y0.x, gb, fmaf(d0.x, ga.x, gc)); o0.y = fmaf(mu - y0.y, gb, fmaf(d0.y, ga.y, gc));
            o0.z = fmaf(mu - y0.z, gb, fmaf(d0.z, ga.z, gc)); o0.w = fmaf(mu - y0.w, gb, fmaf(d0.w, ga.w, gc));
            o1.x = fmaf(mu - y1.x, gb, fmaf(d1.x, ga.x, gc)); o1.y = fmaf(mu - y1.y, gb, fmaf(d1.y, ga.y, gc));
            o1.z = fmaf(mu - y1.z, gb, fmaf(d1.z, ga.z, gc)); o1.w = fmaf(mu - y1.w, gb, fmaf(d1.w, ga.w, gc));
            if (!in0) o0 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!in1) o1 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (desig) {
                if (in0) *reinterpret_cast<float4*>(dyq[0] + tapoff) = o0;
                if (in1) *reinterpret_cast<float4*>(dyq[1] + tapoff) = o1;
            }
            const float4 h0v = make_float4(tf32_hi(o0.x), tf32_hi(o0.y), tf32_hi(o0.z), tf32_hi(o0.w));
            const float4 h1v = make_float4(tf32_hi(o1.x), tf32_hi(o1.y), tf32_hi(o1.z), tf32_hi(o1.w));
            const float4 hw = make_float4(tf32_hi(vw.x), tf32_hi(vw.y), tf32_hi(vw.z), tf32_hi(vw.w));
            sts128(slot, h0v);
            sts128(slot + NTT * 16u, h1v);
            sts128(slot + 2 * A_TILE, hw);
            sts128(lo_a32 + ls * A_TILE, make_float4(o0.x - h0v.x, o0.y - h0v.y, o0.z - h0v.z, o0.w - h0v.w));
            sts128(lo_a32 + ls * A_TILE + NTT * 16u, make_float4(o1.x - h1v.x, o1.y - h1v.y, o1.z - h1v.z, o1.w - h1v.w));
            sts128(lo_b32 + ls * B_TILE, make_float4(vw.x - hw.x, vw.y - hw.y, vw.z - hw.z, vw.w - hw.w));
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&l_full[ls]);
            slot += SLOT;
            if (++sl == D) { sl = 0; slot = slots32; ph_full ^= 1u; }
            c += BK;
            if (c >= Cout) { c = 0; if (++s == ks) { s = 0; ++r; } }
        }
        }
    }
    if (nkb > 0) mbar_wait(done, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: TMEM -> shared memory, cluster reduction, [+ addend], ReLU mask, stores, GroupNorm_p backward sums
    if (warp < NTW) {
        const int q4 = warp & 3, cgp = warp >> 2;
        float facc[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) facc[q] = 0.f;
        const int nacc = nkb < NACC ? nkb : NACC;
#pragma unroll 1
        for (int a = 0; a < nacc; ++a) {
            uint32_t v[16];
            const uint32_t taddr = tmem_d + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(a * BN + cgp * 16);
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                  "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                : "r"(taddr)
                : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int q = 0; q < 16; ++q) facc[q] += __uint_as_float(v[q]);
        }
        const uint32_t dst = smem_u32(red) + (uint32_t)((q4 * 32 + lane) * RED_LD + cgp * 16) * 4u;
#pragma unroll
        for (int q = 0; q < 4; ++q) sts128(dst + q * 16, make_float4(facc[q * 4], facc[q * 4 + 1], facc[q * 4 + 2], facc[q * 4 + 3]));
    }
    cg::cluster_group cluster = cg::this_cluster();
    if (nz == 1) __syncthreads(); else cluster.sync();

    // rows [rank * rows_per, +rows_per) of the tile belong to this CTA: thread -> float4 column c4 of rows row0, row0 + 32, ...
    const int rows_per = BM / nz;
    const int gw = Cin >> 2;
    const int lg_lpg = gw >= BN ? 4 : (gw == 32 ? 3 : 2), gpt = 16 >> lg_lpg;       // float4 columns per group inside the tile; groups per tile
    const bool prep = L.mask != nullptr;
    // per-warp partial sums (plain stores, summed in a fixed order below): the operand slots are free after the last MMA
    float* wsq = reinterpret_cast<float*>(slots);           // [NTW][2 GN][4 groups][2]: sum q, sum q x^
    float* wdg = wsq + NTW * 16;                            // [NTW][2 GN][64]: d gamma
    float* wdb = wdg + NTW * 128;                           // [NTW][64]: d beta
    if (warp < NTW) {
        const int c4 = (tid & 15) * 4, cabs = n0 + c4, g = cabs / gw, row0 = tid >> 4;     // this thread's 4 channels: fixed over the loop
        int lr = rank * rows_per + row0;
        size_t e = ((size_t)b * H * W + m0 + lr) * Cin + cabs;
        const size_t estep = (size_t)32 * Cin;
        uint32_t ra = smem_u32(red) + (uint32_t)(lr * RED_LD + c4) * 4u;
        float4 sdg[2], sdb = make_float4(0.f, 0.f, 0.f, 0.f);
        sdg[0] = sdg[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        float sq[2] = {0.f, 0.f}, sqx[2] = {0.f, 0.f};
        float4 gam[2];
        float pmu[2] = {0.f, 0.f}, prs[2] = {1.f, 1.f};
        if (prep) {
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (j < L.nprep) {
                    gam[j] = ldg4(L.p[j].gamma + cabs);
                    pmu[j] = __ldg(L.p[j].stats + ((size_t)b * 4 + g) * 2); prs[j] = __ldg(L.p[j].stats + ((size_t)b * 4 + g) * 2 + 1);
                }
        }
#pragma unroll 1
        for (int k = row0; k < rows_per; k += 32, lr += 32, ra += 32 * RED_LD * 4, e += estep) {
            if (lr < rows_valid) {
                float4 acc;
                if (nz == 1) {
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
                if (L.addend != nullptr) { const float4 a = __ldcg(reinterpret_cast<const float4*>(L.addend + e)); acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w; }
                if (prep) {
                    const float4 m = __ldcg(reinterpret_cast<const float4*>(L.mask + e));
                    acc.x = m.x > 0.f ? acc.x : 0.f; acc.y = m.y > 0.f ? acc.y : 0.f; acc.z = m.z > 0.f ? acc.z : 0.f; acc.w = m.w > 0.f ? acc.w : 0.f;
                    sdb.x += acc.x; sdb.y += acc.y; sdb.z += acc.z; sdb.w += acc.w;
#pragma unroll
                    for (int j = 0; j < 2; ++j)
                        if (j < L.nprep) {
                            const float4 yv = __ldcg(reinterpret_cast<const float4*>(L.p[j].y + e));
                            const float x0 = (yv.x - pmu[j]) * prs[j], x1 = (yv.y - pmu[j]) * prs[j], x2 = (yv.z - pmu[j]) * prs[j], x3 = (yv.w - pmu[j]) * prs[j];
                            const float q0 = acc.x * gam[j].x, q1 = acc.y * gam[j].y, q2 = acc.z * gam[j].z, q3 = acc.w * gam[j].w;
                            sdg[j].x += acc.x * x0; sdg[j].y += acc.y * x1; sdg[j].z += acc.z * x2; sdg[j].w += acc.w * x3;
                            sq[j] += (q0 + q1) + (q2 + q3);
                            sqx[j] += (q0 * x0 + q1 * x1) + (q2 * x2 + q3 * x3);
                        }
                } else if (L.accumulate) {
                    const float4 a = *reinterpret_cast<const float4*>(L.out + e);
                    acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
                }
                *reinterpret_cast<float4*>(L.out + e) = acc;
            }
        }
        if (prep) {
            // fixed-order reductions: warp butterflies, then one plain shared slot per warp; the cross-CTA step is integer (below)
            const uint32_t wsq32 = smem_u32(wsq), wdg32 = smem_u32(wdg), wdb32 = smem_u32(wdb);
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (j < L.nprep) {
                    float a = sq[j], c = sqx[j];
                    a += __shfl_xor_sync(0xffffffffu, a, 16); c += __shfl_xor_sync(0xffffffffu, c, 16);
                    if (lg_lpg > 3) { a += __shfl_xor_sync(0xffffffffu, a, 8); c += __shfl_xor_sync(0xffffffffu, c, 8); }
                    if (lg_lpg > 2) { a += __shfl_xor_sync(0xffffffffu, a, 4); c += __shfl_xor_sync(0xffffffffu, c, 4); }
                    a += __shfl_xor_sync(0xffffffffu, a, 2); c += __shfl_xor_sync(0xffffffffu, c, 2);
                    a += __shfl_xor_sync(0xffffffffu, a, 1); c += __shfl_xor_sync(0xffffffffu, c, 1);
                    if (lane < 16 && (lane & ((1 << lg_lpg) - 1)) == 0) {
                        const uint32_t w = wsq32 + (uint32_t)(((warp * 2 + j) * 4 + (lane >> lg_lpg)) * 2) * 4u;
                        sts32(w, a); sts32(w + 4, c);
                    }
                    // per-channel d gamma: rows of lanes l and l + 16
                    float4 dg = sdg[j];
                    dg.x += __shfl_xor_sync(0xffffffffu, dg.x, 16); dg.y += __shfl_xor_sync(0xffffffffu, dg.y, 16);
                    dg.z += __shfl_xor_sync(0xffffffffu, dg.z, 16); dg.w += __shfl_xor_sync(0xffffffffu, dg.w, 16);
                    if (lane < 16) sts128(wdg32 + (uint32_t)((warp * 2 + j) * 64 + c4) * 4u, dg);
                }
            float4 db = sdb;                                 // d beta: the same for both GroupNorms
            db.x += __shfl_xor_sync(0xffffffffu, db.x, 16); db.y += __shfl_xor_sync(0xffffffffu, db.y, 16);
            db.z += __shfl_xor_sync(0xffffffffu, db.z, 16); db.w += __shfl_xor_sync(0xffffffffu, db.w, 16);
            if (lane < 16) sts128(wdb32 + (uint32_t)(warp * 64 + c4) * 4u, db);
        }
    }
    __syncthreads();
    if (prep) {
        // per CTA and quantity: 16 warp partials added in warp order, then ONE 64-bit fixed-point atomic (exact, order independent)
        if (tid < 16 * L.nprep) {
            const int j = tid >> 4, i = tid & 15, gi = i >> 1;
            if (gi < gpt) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < NTW; ++w) t += wsq[((w * 2 + j) * 4 + gi) * 2 + (i & 1)];
                const int g = gw >= BN ? (nt * BN) / gw : nt * gpt + gi;
                atomicAdd(L.p[j].sums + ((size_t)b * 4 + g) * 2 + (i & 1), (unsigned long long)to_fix(t));
            }
        } else if (tid >= 64 && tid < 64 + 128 * L.nprep) {
            const int j = (tid - 64) >> 7, i = (tid - 64) & 127, ch = i >> 1;
            float t = 0.f;
            if (i & 1) {
#pragma unroll
                for (int w = 0; w < NTW; ++w) t += wdb[w * 64 + ch];
            } else {
#pragma unroll
                for (int w = 0; w < NTW; ++w) t += wdg[(w * 2 + j) * 64 + ch];
            }
            atomicAdd(L.p[j].dgb + (size_t)(n0 + ch) * 2 + (i & 1), (unsigned long long)to_fix(t));
        }
    }
    if (nz > 1) cluster.sync();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(ATM ? 512 : BN * NACC) : "memory");
}

// Stand-alone version of the epilogue above for the seams with the unfused kernels (after avgpool_bwd; after a stride-2 block):
// dz = dA * (a > 0) -> out; sums / d gamma / d beta of GroupNorm_p.  grid (ceil(HW / rows_per_cta), B), 256 threads: a thread keeps
// its channel vector(s) over the (few) rows of the CTA, all loads of a row group in flight together; the two group sums go
// through a warp butterfly before they touch shared memory (a warp's 32 channel vectors lie in one group for C >= 512; for
// narrower layers the segments are 16 / 8 lanes), so the shared 64-bit adds see at most 8 contenders instead of 256.
__global__ void __launch_bounds__(256) gn_bwd_prep_kernel(const float* __restrict__ dA, const float* __restrict__ mask, float* __restrict__ out,
                                                          Prep p, int HW, int C, int rows_per_cta) {
    __shared__ unsigned long long sacc[8];
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y, C4 = C >> 2, gw = C >> 2, lane = threadIdx.x & 31;
    const int cvg = C4 >> 2;                                 // channel vectors per group (a power of two >= 4 for the backbone widths)
    const int seg = cvg >= 32 ? 32 : cvg;                    // lanes of a warp that share a group
    if (threadIdx.x < 8) sacc[threadIdx.x] = 0ull;
    __syncthreads();
    const int r_begin = blockIdx.x * rows_per_cta, r_end = min(HW, r_begin + rows_per_cta);
    for (int cv0 = 0; cv0 < C4; cv0 += 256) {                // uniform trip count: every lane takes part in the butterflies
        const int cv = cv0 + threadIdx.x;
        const bool live = cv < C4;
        const int c = live ? cv * 4 : 0, g = c / gw;
        float4 sdg = make_float4(0.f, 0.f, 0.f, 0.f), sdb = sdg;
        float sq = 0.f, sqx = 0.f;
        if (live) {
            const float4 ga = ldg4(p.gamma + c);
            const float mu = __ldg(p.stats + ((size_t)b * 4 + g) * 2), rs = __ldg(p.stats + ((size_t)b * 4 + g) * 2 + 1);
#pragma unroll 4
            for (int r = r_begin; r < r_end; ++r) {
                const size_t e = ((size_t)b * HW + r) * C + c;
                float4 d = __ldcg(reinterpret_cast<const float4*>(dA + e));
                const float4 m = __ldcg(reinterpret_cast<const float4*>(mask + e)), yv = __ldcg(reinterpret_cast<const float4*>(p.y + e));
                d.x = m.x > 0.f ? d.x : 0.f; d.y = m.y > 0.f ? d.y : 0.f; d.z = m.z > 0.f ? d.z : 0.f; d.w = m.w > 0.f ? d.w : 0.f;
                *reinterpret_cast<float4*>(out + e) = d;
                const float x0 = (yv.x - mu) * rs, x1 = (yv.y - mu) * rs, x2 = (yv.z - mu) * rs, x3 = (yv.w - mu) * rs;
                const float q0 = d.x * ga.x, q1 = d.y * ga.y, q2 = d.z * ga.z, q3 = d.w * ga.w;
                sdg.x += d.x * x0; sdg.y += d.y * x1; sdg.z += d.z * x2; sdg.w += d.w * x3;
                sdb.x += d.x; sdb.y += d.y; sdb.z += d.z; sdb.w += d.w;
                sq += (q0 + q1) + (q2 + q3);
                sqx += (q0 * x0 + q1 * x1) + (q2 * x2 + q3 * x3);
            }
        }
        long long a1 = to_fix(sq), a2 = to_fix(sqx);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1)
            if (o < seg) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
        if (live && (lane & (seg - 1)) == 0) {
            atomicAdd(&sacc[g * 2], (unsigned long long)a1);
            atomicAdd(&sacc[g * 2 + 1], (unsigned long long)a2);
        }
        if (live) {
            const float dgv[4] = {sdg.x, sdg.y, sdg.z, sdg.w}, dbv[4] = {sdb.x, sdb.y, sdb.z, sdb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                atomicAdd(p.dgb + (size_t)(c + e) * 2, (unsigned long long)to_fix(dgv[e]));
                atomicAdd(p.dgb + (size_t)(c + e) * 2 + 1, (unsigned long long)to_fix(dbv[e]));
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < 8) atomicAdd(p.sums + (size_t)b * 8 + threadIdx.x, sacc[threadIdx.x]);
}

// G[g_off + c] += d gamma, G[b_off + c] += d beta from the fixed-point accumulators of every GroupNorm (one launch per backward)
__global__ void __launch_bounds__(256) gn_dgb_finish_kernel(const GnFinishItem* __restrict__ items, const long long* __restrict__ dgb, float* __restrict__ G) {
    pdl_wait();
    pdl_trigger();
    const GnFinishItem it = items[blockIdx.x];
    const long long* a = dgb + 2 * it.cum_channels;
    for (int c = threadIdx.x; c < it.C; c += 256) {
        const long long vg = a[2 * c], vb = a[2 * c + 1];
        if (vg != 0) G[it.g_off + c] += (float)((double)vg / FIX);
        if (vb != 0) G[it.b_off + c] += (float)((double)vb / FIX);
    }
}

}  // namespace dz

bool dgrad_wide_ok(const ConvDims& d) {
    return d.stride == 1 && d.Ho == d.Hi && d.Wo == d.Wi && d.Hi == d.Wi && d.Cin % 64 == 0 && d.Cout % 64 == 0 && (d.kh == 1 || d.kh == 3) && d.kh == d.kw &&
           d.pad == d.kh / 2 && d.Kpitch == d.kh * d.kw * d.Cin && d.Hi <= 128;
}

// split-K limits: CTA budget (DBOA_DGRAD_MAX_CTAS; a budget that does not exceed twice the tiles means 2 x tiles, at most 128),
// largest cluster (DBOA_DGRAD_MAX_NZ) and the fewest k-blocks a K-slice may hold
static int dgrad_budget_default() { const char* e = getenv("DBOA_DGRAD_MAX_CTAS"); return e ? atoi(e) : 64; }
static int dgrad_max_nz_default() { const char* e = getenv("DBOA_DGRAD_MAX_NZ"); return clamp_split(e ? atoi(e) : 16, 1, 16); }
static int g_dgrad_budget = dgrad_budget_default();
static int g_dgrad_max_nz = dgrad_max_nz_default();
static int g_dgrad_min_kb = 2;
void dgrad_wide_set_limits(int max_ctas, int max_nz, int min_kb) {
    g_dgrad_budget = max_ctas < 0 ? dgrad_budget_default() : max_ctas;
    g_dgrad_max_nz = max_nz < 0 ? dgrad_max_nz_default() : clamp_split(max_nz, 1, 16);
    g_dgrad_min_kb = min_kb < 0 ? 2 : clamp_split(min_kb, 1, 1 << 30);
}

int dgrad_wide(const DgradFused& f, const ConvDims& d, cudaStream_t st, bool pdl) {
    if (!dgrad_wide_ok(d)) return DBOA_ERR_UNSUPPORTED;
    dz::Launch L;
    memset(&L, 0, sizeof L);
    L.stats_c = f.stats_c; L.sums_c = reinterpret_cast<const long long*>(f.sums_c); L.gamma_c = f.gamma_c; L.dy_out = f.dy_out;
    L.addend = f.addend; L.out = f.out; L.mask = f.mask; L.nprep = f.mask ? f.nprep : 0; L.accumulate = f.accumulate;
    for (int j = 0; j < 2; ++j) {
        L.p[j].y = f.prep[j].y; L.p[j].stats = f.prep[j].stats; L.p[j].gamma = f.prep[j].gamma;
        L.p[j].sums = reinterpret_cast<unsigned long long*>(f.prep[j].sums); L.p[j].dgb = reinterpret_cast<unsigned long long*>(f.prep[j].dgb);
    }
    L.H = d.Hi; L.W = d.Wi; L.Cin = d.Cin; L.Cout = d.Cout; L.k = d.kh; L.pad = d.pad; L.B = d.B;
    L.bh = d.Hi * d.Hi <= dz::BM ? d.Hi : dz::BM / d.Hi;
    L.tps = ceil_div(d.Hi, L.bh); L.ntiles = d.Cin / dz::BN;
    const int tiles = d.B * L.tps * L.ntiles, nkb = d.kh * d.kw * d.Cout / dz::BK;
    const int budget = g_dgrad_budget;
    int nz = 1;
    while (nz < g_dgrad_max_nz && tiles * nz * 2 <= (budget > 2 * tiles ? budget : (2 * tiles < 128 ? 2 * tiles : 128)) && nkb / (nz * 2) >= g_dgrad_min_kb)
        nz *= 2;
    while (nz > 1 && (nz - 1) * ceil_div(nkb, nz) >= nkb) nz >>= 1;
    L.nz = nz; L.per = ceil_div(nkb, nz);
    L.tabc = d.kh == 1 ? L.per * dz::BK : d.Cout;
    const size_t fixed = 2 * (size_t)(dz::A_TILE + dz::B_TILE) + (size_t)L.tabc * sizeof(float) + 4096 + 1024;
    int D = L.per < dz::DMAX ? L.per : dz::DMAX;
    while (D > 1 && fixed + (size_t)D * dz::SLOT > 227 * 1024) --D;
    L.D = D;
    const size_t smem = fixed + (size_t)D * dz::SLOT;
    const CUtensorMap* tmdz = static_cast<const CUtensorMap*>(tma_act_map(f.dz, d.B, d.Hi, d.Wi, d.Cout, d.Wi, L.bh, false, 1));
    const CUtensorMap* tmy = static_cast<const CUtensorMap*>(tma_act_map(f.y_c, d.B, d.Hi, d.Wi, d.Cout, d.Wi, L.bh, false, 1));
    const CUtensorMap* tmw = static_cast<const CUtensorMap*>(tma_weight_map_mn(f.w, d.kh * d.kw * d.Cin, d.Cout));
    if (!tmdz || !tmy || !tmw) return DBOA_ERR_CUDA;
    wide_plan_note(1, nz, L.per, D, tiles * nz, nkb);
    return conv_wide_operand_tmem() ? launch_ex(dz::dgrad_wide_kernel<true>, dim3(tiles * nz), dim3(dz::NT), smem, st, dim3(nz, 1, 1), pdl, L, *tmdz, *tmy, *tmw)
                                    : launch_ex(dz::dgrad_wide_kernel<false>, dim3(tiles * nz), dim3(dz::NT), smem, st, dim3(nz, 1, 1), pdl, L, *tmdz, *tmy, *tmw);
}

int gn_bwd_prep(const float* dA, const float* mask, float* out, const DgradPrep& p, int B, int HW, int C, cudaStream_t st) {
    if (C % 4 != 0 || C / 4 > 512) return DBOA_ERR_SHAPE;
    dz::Prep pp;
    pp.y = p.y; pp.stats = p.stats; pp.gamma = p.gamma; pp.sums = reinterpret_cast<unsigned long long*>(p.sums); pp.dgb = reinterpret_cast<unsigned long long*>(p.dgb);
    // enough CTAs to cover the GPU with SHORT row loops (the kernel is a latency chain: a row is one memory round trip)
    int rows_per = 1;
    while (rows_per < 8 && ceil_div(HW, rows_per * 2) * B >= 148) rows_per *= 2;
    return launch_ex(dz::gn_bwd_prep_kernel, dim3(ceil_div(HW, rows_per), B), dim3(256), 0, st, dim3(1, 1, 1), true, dA, mask, out, pp, HW, C, rows_per);
}

int gn_dgb_finish(const GnFinishItem* items_dev, int n_items, const float* dgb, float* G, cudaStream_t st) {
    return launch_ex(dz::gn_dgb_finish_kernel, dim3(n_items), dim3(256), 0, st, dim3(1, 1, 1), true, items_dev, reinterpret_cast<const long long*>(dgb), G);
}

}  // namespace dboa
