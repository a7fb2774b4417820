// Weight gradient of a stride-1 convolution on tcgen05 tensor cores, both operands through TMA, no transposing stores:
//
//      dW[co][tap][ci] += sum_{pixels} dY[pix][co] * X[pix + tap - pad][ci]
//
// Replaces the autograd weight gradient of nn.Conv2d (reference model/hmr.py:29-34 under loss.backward(), dynaboa_benchmark.py:
// 140,150).  Round 1 ran it on CUDA cores (conv.cu: conv_wgrad_kernel<4>, 18 % of the kernel time of a frame) because in the
// K-major layouts conv_tc.cu uses BOTH operands of this GEMM need a transposing shared-memory store: the reduction index is the
// pixel, and memory is channel-contiguous.  tcgen05 takes MN-major operands directly (instruction descriptor bits 15 / 16,
// cute::UMMA::InstrDescriptor a_major_ / b_major_, valid for TF32), and the MN-major 128-byte-swizzle canonical layout
//      ((4, 8, m), (8, k)) : ((1, 4, LBO), (32, SBO))   in floats  (cute/atom/mma_traits_sm100.hpp, "Major-MN")
// -- for TF32 its 32-byte-atom variant (SWIZZLE_128B_BASE32B, 4-pixel groups 512 B apart) -- is exactly what a TMA box of
// 32 channels x (pixels) with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B writes: one 128-byte row per pixel, one box per 32-channel
// block, LBO apart.  (With the plain 128-byte swizzle and layout type 2 the MN-major TF32 MMA silently produces zeros.)  So:
//   * GEMM: M = 128 output channels (4 boxes of dY), N = 64 input channels (2 boxes of X, shifted by the filter tap, zero fill
//     at the image border by TMA), K = 56 pixels per k-block (whole image rows: 1 x 56, 2 x 28, 4 x 14 or the 7 x 7 image padded
//     by one out-of-bounds row), 7 k-steps of 8;
//   * TF32x3: one elementwise shared-memory pass turns the landed raw tiles into (hi in place, lo in a second tile) -- the same
//     pass as conv_wide.cu, layout agnostic;
//   * split-K over thread-block clusters (pixels), deterministic DSMEM reduction, then dW += tile (single writer per element).
// Stride 2: the X tensor map samples every second pixel (TMA element strides).  Layers with Cout < 128 (stem, layer1's
// 64-channel outputs) stay on conv.cu.
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

namespace wg {

constexpr int BM = 128, BN = 64, KB = 56;
constexpr int NTW = 16, NTT = NTW * 32, W_MMA = 16, W_TMA = 17, NT = 576;
constexpr uint32_t ATOM = KB * 128;                     // one box: 56 pixels x 32 channels (7168 B = 7 x 1024)
constexpr uint32_t A_BYTES = 4 * ATOM, B_BYTES = 2 * ATOM, STAGE = A_BYTES + B_BYTES;        // 43008 B raw per stage (+ the same for lo)
constexpr int RED_LD = BN + 4;
constexpr int NACC = 4;                                 // TMEM accumulators a reduction chain rotates over (see conv_wide.cu)

struct Launch {
    float* dw;
    int Cin, Cout, k, pad, stride, H, W, bh, kps, nkb_total;     // kps: k-blocks per sample; nkb_total = B * kps
    int ntn, taps, nz, per;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// MN-major TF32: the only layout tcgen05 takes is SWIZZLE_128B_BASE32B (layout type 1: 32-byte chunks XOR (row & 3), atoms of
// 32 channels x 4 pixels; cutlass sm100_common.inl: "for mn-major tf32 operands, SW128_32B is the only available smem layout").
// LBO = byte distance between 32-channel blocks, SBO = byte distance between 4-pixel groups (512 B: rows are stacked densely).
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((ATOM >> 4) & 0x3FFF) << 16) | ((uint64_t)((512 >> 4) & 0x3FFF) << 32) | (1ull << 46) |
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
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

__global__ void __launch_bounds__(NT, 1) conv_wgrad_wide_kernel(const __grid_constant__ Launch L, const __grid_constant__ CUtensorMap tmdy,
                                                                const __grid_constant__ CUtensorMap tmx) {
    extern __shared__ uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nz = L.nz;
    const int cidx = blockIdx.x / nz, rank = blockIdx.x - cidx * nz;
    // tile: cidx = (mt * ntn + nt) * taps + tap
    const int tap = cidx % L.taps, mn = cidx / L.taps, nt = mn % L.ntn, mt = mn / L.ntn;
    const int r = tap / L.k, s = tap - r * L.k;
    const int m0 = mt * BM, n0 = nt * BN;
    const int kb_begin = rank * L.per;
    const int nkb = max(0, min(L.per, L.nkb_total - kb_begin));

    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* raw = base;                          // 2 stages x {A: 4 atoms, B: 2 atoms}
    uint8_t* lo = raw + 2 * STAGE;                // same shape
    uint64_t* bars = reinterpret_cast<uint64_t*>(lo + 2 * STAGE);
    uint64_t* s_full = bars;                      // [2] TMA -> split pass
    uint64_t* l_full = bars + 2;                  // [2] split pass -> MMA issuer
    uint64_t* s_empty = bars + 4;                 // [2] tcgen05.commit -> TMA warp
    uint64_t* done = bars + 6;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
    float* red = reinterpret_cast<float*>(raw);   // 128 x RED_LD fp32 partial tile over the raw stages after the last MMA

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&l_full[i], NTW); mbar_init(&s_empty[i], 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(BN * NACC) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;
    pdl_wait();
    pdl_trigger();

    if (warp == W_TMA) {
        if (lane == 0) {
            for (int it = 0; it < nkb; ++it) {
                const int st = it & 1;
                if (it >= 2) mbar_wait(&s_empty[st], (uint32_t)(((it >> 1) - 1) & 1));
                const int kb = kb_begin + it, b = kb / L.kps, h0 = (kb - b * L.kps) * L.bh;
                uint8_t* a = raw + (size_t)st * STAGE;
                mbar_expect_tx(&s_full[st], STAGE);
#pragma unroll
                for (int j = 0; j < 4; ++j) tma_load_4d(smem_u32(a + j * ATOM), &tmdy, m0 + 32 * j, 0, h0, b, &s_full[st]);
#pragma unroll
                for (int j = 0; j < 2; ++j) tma_load_4d(smem_u32(a + A_BYTES + j * ATOM), &tmx, n0 + 32 * j, s - L.pad, h0 * L.stride + r - L.pad, b, &s_full[st]);
            }
        }
    } else if (warp == W_MMA) {
        // warp-uniform loop, one elected lane issues (see conv_wide.cu)
        if (nkb > 0) {
            // D = F32, A = B = TF32, both MN-major (bits 15, 16), N >> 3, M >> 4
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint64_t draw = desc_mn(smem_u32(raw)), dlo = desc_mn(smem_u32(lo));
            constexpr uint64_t KSTEP = 1024 >> 4;                  // 8 pixels = one 8-row group
#pragma unroll 1
            for (int it = 0; it < nkb; ++it) {
                const int st = it & 1;
                mbar_wait(&l_full[st], (uint32_t)((it >> 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t so = (uint64_t)(st * (STAGE >> 4));
                const uint64_t dah = draw + so, dbh = dah + (A_BYTES >> 4), dal = dlo + so, dbl = dal + (A_BYTES >> 4);
                // the tensor core accumulates with truncation: k-block `it` goes to accumulator it % NACC, which keeps each chain
                // short (one chain of 112 k-blocks was 5e-5 off an fp64 reference on a B200); the epilogue adds the accumulators in fp32
                const uint32_t dacc = tmem_d + (uint32_t)((it & (NACC - 1)) * BN);
                const uint32_t first = it >= NACC ? 1u : 0u;
                if (elect_one()) {
#pragma unroll
                    for (int kk = 0; kk < KB / 8; ++kk) {
                        mma_tf32(dacc, dah + kk * KSTEP, dbh + kk * KSTEP, idesc, kk > 0 ? 1u : first);
                        mma_tf32(dacc, dah + kk * KSTEP, dbl + kk * KSTEP, idesc, 1u);
                        mma_tf32(dacc, dal + kk * KSTEP, dbh + kk * KSTEP, idesc, 1u);
                    }
                    umma_commit(&s_empty[st]);
                }
                __syncwarp();
            }
            if (elect_one()) umma_commit(done);
        }
    } else {
        // split pass: raw -> (hi in place, lo) at the same offsets; 2688 float4 per stage over 512 threads
        const uint32_t raw32 = smem_u32(raw) + (uint32_t)tid * 16u;
        constexpr uint32_t LO_OFS = 2 * STAGE, NV = STAGE / 16;
#pragma unroll 1
        for (int it = 0; it < nkb; ++it) {
            const int st = it & 1;
            mbar_wait(&s_full[st], (uint32_t)((it >> 1) & 1));
            const uint32_t rp = raw32 + (uint32_t)st * STAGE;
            float4 v[6];
#pragma unroll
            for (int j = 0; j < 6; ++j)
                if (j < 5 || tid + 5 * NTT < (int)NV) v[j] = lds128(rp + (uint32_t)j * NTT * 16u);
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                if (j < 5 || tid + 5 * NTT < (int)NV) {
                    const float4 h = make_float4(tf32_hi(v[j].x), tf32_hi(v[j].y), tf32_hi(v[j].z), tf32_hi(v[j].w));
                    sts128(rp + (uint32_t)j * NTT * 16u, h);
                    sts128(rp + LO_OFS + (uint32_t)j * NTT * 16u, make_float4(v[j].x - h.x, v[j].y - h.y, v[j].z - h.z, v[j].w - h.w));
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&l_full[st]);
        }
    }
    if (nkb > 0) mbar_wait(done, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: TMEM (lane = output channel, column = input channel) -> shared memory -> cluster reduction -> dW +=
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
    if (warp < NTW) {
        // rows [rank * rows_per, +rows_per) of the tile belong to this CTA: thread -> float4 column c4 of rows row0, row0 + 32, ...
        const int rows_per = BM / nz, Kfull = L.k * L.k * L.Cin;
        const int c4 = (tid & 15) * 4, row0 = tid >> 4;
        int lr = rank * rows_per + row0;
        float* dp = L.dw + (size_t)(m0 + lr) * Kfull + (size_t)tap * L.Cin + n0 + c4;
        const size_t dstep = (size_t)32 * Kfull;
        uint32_t ra = smem_u32(red) + (uint32_t)(lr * RED_LD + c4) * 4u;
#pragma unroll 1
        for (int k = row0; k < rows_per; k += 32, ra += 32 * RED_LD * 4, dp += dstep) {
            float4 cur = *reinterpret_cast<const float4*>(dp);
            float4 acc;
            if (nz == 1) {
                acc = lds128(ra);
            } else {
                acc = ldc128(ra, 0);
                const float4 q1 = ldc128(ra, 1);
                acc.x += q1.x; acc.y += q1.y; acc.z += q1.z; acc.w += q1.w;
#pragma unroll 1
                for (int z = 2; z < nz; z += 2) {
                    const float4 qa = ldc128(ra, z), qb = ldc128(ra, z + 1);
                    acc.x += qa.x; acc.y += qa.y; acc.z += qa.z; acc.w += qa.w;
                    acc.x += qb.x; acc.y += qb.y; acc.z += qb.z; acc.w += qb.w;
                }
            }
            cur.x += acc.x; cur.y += acc.y; cur.z += acc.z; cur.w += acc.w;
            *reinterpret_cast<float4*>(dp) = cur;
        }
    }
    if (nz > 1) cluster.sync();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(BN * NACC) : "memory");
}

}  // namespace wg

bool conv_wgrad_wide_ok(const ConvDims& d) {
    const int W = d.Wo;
    return (d.stride == 1 || d.stride == 2) && d.Hi == d.Ho * d.stride && d.Wi == d.Wo * d.stride && d.Ho == d.Wo && d.Cout % 128 == 0 && d.Cin % 64 == 0 && (d.kh == 1 || d.kh == 3) && d.kh == d.kw &&
           d.pad == d.kh / 2 && d.Kpitch == d.kh * d.kw * d.Cin && (W == 56 || W == 28 || W == 14 || W == 7);
}

// Split-K limits.  Weight gradients run on side streams NEXT to the data-gradient chain: a launch owns its SMs (one CTA of 170 KB
// each), so its K-slices are limited to a CTA budget that leaves room for the chain (DBOA_WGRAD_MAX_CTAS, at least 1).
// DBOA_WGRAD_MAX_NZ: largest cluster (K-slices of one tile).  A cluster needs that many free SMs inside ONE GPC, so large
// clusters cannot start next to another stream's kernel that has CTAs in every GPC.
static int wgrad_budget_default() { const char* e = getenv("DBOA_WGRAD_MAX_CTAS"); return clamp_split(e ? atoi(e) : 128, 1, 1 << 30); }
static int wgrad_max_nz_default() { const char* e = getenv("DBOA_WGRAD_MAX_NZ"); return clamp_split(e ? atoi(e) : 16, 1, 16); }
static int g_wgrad_budget = wgrad_budget_default();
static int g_wgrad_max_nz = wgrad_max_nz_default();
static int g_wgrad_min_kb = 1;
void conv_wgrad_wide_set_limits(int max_ctas, int max_nz, int min_kb) {
    g_wgrad_budget = max_ctas < 0 ? wgrad_budget_default() : clamp_split(max_ctas, 1, 1 << 30);
    g_wgrad_max_nz = max_nz < 0 ? wgrad_max_nz_default() : clamp_split(max_nz, 1, 16);
    g_wgrad_min_kb = min_kb < 0 ? 1 : clamp_split(min_kb, 1, 1 << 30);
}

int conv_wgrad_wide(const float* dy, const float* x, float* dw, const ConvDims& d, cudaStream_t st, bool pdl) {
    if (!conv_wgrad_wide_ok(d)) return DBOA_ERR_UNSUPPORTED;
    wg::Launch L;
    memset(&L, 0, sizeof L);
    const int W = d.Wo, bh = W == 7 ? 8 : wg::KB / W;
    L.dw = dw; L.Cin = d.Cin; L.Cout = d.Cout; L.k = d.kh; L.pad = d.pad; L.stride = d.stride; L.H = d.Ho; L.W = W; L.bh = bh;
    L.kps = ceil_div(d.Ho, bh); L.nkb_total = d.B * L.kps;
    L.ntn = d.Cin / wg::BN; L.taps = d.kh * d.kw;
    const int tiles = (d.Cout / wg::BM) * L.ntn * L.taps;
    int nz = 1;
    while (nz < g_wgrad_max_nz && tiles * nz * 2 <= g_wgrad_budget && L.nkb_total / (nz * 2) >= g_wgrad_min_kb) nz *= 2;
    while (nz > 1 && (nz - 1) * ceil_div(L.nkb_total, nz) >= L.nkb_total) nz >>= 1;
    L.nz = nz; L.per = ceil_div(L.nkb_total, nz);
    const CUtensorMap* tmdy = static_cast<const CUtensorMap*>(tma_act_map(dy, d.B, d.Ho, d.Wo, d.Cout, W, bh, true, 1));
    const CUtensorMap* tmx = static_cast<const CUtensorMap*>(tma_act_map(x, d.B, d.Hi, d.Wi, d.Cin, W, bh, true, d.stride));
    if (tmdy == nullptr || tmx == nullptr) return DBOA_ERR_CUDA;
    wide_plan_note(2, nz, L.per, 2, tiles * nz, L.nkb_total);      // two operand stages
    const size_t smem = 4 * (size_t)wg::STAGE + 1024 + 1024;
    return launch_ex(wg::conv_wgrad_wide_kernel, dim3(tiles * nz), dim3(wg::NT), smem, st, dim3(nz, 1, 1), pdl, L, *tmdy, *tmx);
}

}  // namespace dboa
