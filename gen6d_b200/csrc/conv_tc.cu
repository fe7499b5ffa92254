// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05), fp32-faithful through a
// three-term operand split:  A*B ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi, x_hi = round(x) to an 11-bit
// significand, x_lo = x - x_hi (exact in fp32).  The dropped A_lo*B_lo term is O(2^-22) relative, so
// index selections (detection cell, viewpoint) stay bit-exact against the fp32 reference while the
// contraction runs on the tensor pipe instead of the FFMA pipe.  Two operand kinds share every kernel:
//
//   G6D_TC_TF32  hi/lo are tf32 (fp32 containers, 8-bit exponent): any fp32 range, kind::tf32 MMAs
//                (K = 8 per instruction, 32 K-elements per 128-byte swizzle row);
//   G6D_TC_F16   hi = fp16(x), lo = fp16((x - hi) * 2^11): the same 11 + 11 significand bits, but
//                kind::f16 MMAs issue K = 16 per instruction at the same cycle cost and every operand
//                byte (shared-memory tile, TMA weight stream, operand re-read) carries twice the K:
//                2x the tensor ceiling and half the shared-memory traffic per flop.  The lo halves are
//                pre-scaled by 2^11 so that they live in the same exponent range as the hi halves (no
//                fp16 subnormals); both cross terms accumulate in their own TMEM accumulator, which the
//                epilogue folds in with an exact 2^-11.  Range contract: |x| <= 65504 for activations
//                and weights (saturating conversion beyond that), full relative accuracy for |x| >=
//                6.1e-5, absolute error <= ~2^-36 below.  Inside this network every tensor-core operand
//                is a BN-folded weight, a post-ReLU / InstanceNorm-ed / L2-normalised activation or a
//                VGG feature, all O(1e-3 .. 1e3).  G6D_CONV_KIND=tf32 selects the wide-range kind.
//
// GEMM view (same as conv_ffma.cu): M = B*Do*Ho*Wo, N = Cout, K = taps*Cin, channels-last.
// One CTA computes 128 x BLOCK_N output tiles (UMMA M=128, cta_group::1, accumulators in TMEM).
//
// conv_tc2_kernel (general strides / shapes): persistent, one CTA per SM loops over (M tile, N tile,
// K split) work items.  14 warps:
//   warps 0-7   A producers: gather the im2col rows of the K-block from global memory (coalesced
//               128-bit loads, register prefetch ring), apply the folded InstanceNorm(+ReLU) /
//               selector q(.)ref prologue to in-bounds elements, split into hi/lo and st.shared both
//               tiles in the canonical K-major SWIZZLE_128B layout the UMMA descriptor expects;
//   warp 8      B producer: one lane issues TMA (cp.async.bulk.tensor.2d, 128B swizzle) loads of the
//               pre-split weight tiles W_hi / W_lo [Cout, K] (K-major) + an L2 prefetch running ahead;
//   warp 9      MMA issuer (+ TMEM owner): 12 tcgen05.mma per K-block (4 K-steps x 3 split terms);
//               tcgen05.commit releases the stage; two TMEM accumulator buffers so that
//   warps 10-13 the epilogue (tcgen05.ld -> bias/activation -> global, or split-K partials) of tile i
//               overlaps the MMAs of tile i+1.
// conv_tcflat_kernel (stride-1 multi-tap convolutions whose halo fits in shared memory): A-operand
// reuse across taps, see below.
#include <stdlib.h>
#include <string.h>

#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace g6d {

constexpr int TC_BM = 128;       // rows per tile (UMMA M)
constexpr int TC_PRODUCER_WARPS = 8;
constexpr int TC_THREADS = (TC_PRODUCER_WARPS + 2) * 32;   // flat kernel: producers double as epilogue
constexpr int TC_MAX_K_PER_CHAIN = 2048;                   // longest accumulate chain per CTA (see fill_tc_params)

template <int KIND> struct KindCfg;
template <> struct KindCfg<G6D_TC_TF32> {
    static constexpr int BK = 32;          // K elements per 128-byte swizzle row
    static constexpr int NV = 1;           // float4 loads per (thread, row) chunk of 16 smem bytes
    static constexpr int RING = 3;         // register prefetch ring (K-blocks)
    static constexpr float CROSS = 1.f;    // scale of the cross-term accumulator
};
template <> struct KindCfg<G6D_TC_F16> {
    static constexpr int BK = 64;
    static constexpr int NV = 2;
    static constexpr int RING = 2;
    static constexpr float CROSS = 1.f / 2048.f;
};
constexpr float F16_LO_SCALE = 2048.f;
// K order inside a 64-element fp16 K-block.  A producer thread fills one 16-byte shared-memory chunk
// (8 halves) of a tile row from two 128-bit global loads; to keep BOTH loads of a warp fully coalesced
// (8 lanes x 16 B = one 128-byte line per row) lane c reads channels [4c, 4c+4) and [32+4c, 32+4c+4), so
// chunk c holds those eight channels.  The contraction does not care about the order of K as long as the
// weight operand uses the same one: the pack / split kernels write K position p from source channel
// f16_k_source(p).  (ncu, round 2: with adjacent channels per lane every gather touched 8 lines per
// instruction instead of 4 -- twice the L1 tag requests and L2 sectors of the ideal.)
__host__ __device__ __forceinline__ int f16_k_source(int p) {      // p in [0, 64)
    const int c = p >> 3, i = p & 7;
    return i < 4 ? 4 * c + i : 32 + 4 * c + (i - 4);
}

struct ConvTcP {
    const float* x; const float* bias; const float* ps; const float* pb;
    float* y; float* ws;
    int B, D, H, W, Cin, ics, ico, Cout, kd, kh, kw, stride, pd, ph, pw, Do, Ho, Wo, ocs, oco, pro, act;
    long long group_rows;
    int in_items;                             // input items: output item b reads input item b % in_items
    int M, K, kblocks, splits, kb_per_split;
    double* stats; long long stats_rows;      // fused InstanceNorm statistics of the OUTPUT (see epilogue_stats)
};

// ------------------------------------------------------------------------------------------ operand split
// fp16 pair (element 0 in the low half, as laid out in memory), saturating instead of overflowing to inf
__device__ __forceinline__ uint32_t cvt_f16x2_sat(float e0, float e1) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));
    return r;
}
__device__ __forceinline__ void split_f16x2(float e0, float e1, uint32_t& hi, uint32_t& lo) {
    hi = cvt_f16x2_sat(e0, e1);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    // (x - hi) is exact in fp32 and so is the power-of-two scaling
    lo = cvt_f16x2_sat((e0 - hf.x) * F16_LO_SCALE, (e1 - hf.y) * F16_LO_SCALE);
}
// tf32: hi = round-to-nearest (ties away) of the fp32 significand to 10 bits with integer ops (same
// as cvt.rna.tf32.f32 for finite values), lo = v - hi (exact; the tensor core ignores its low 13 bits)
__device__ __forceinline__ void split_tf32x4(const float4 v, float4& hi, float4& lo) {
    hi.x = __uint_as_float((__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u);
    hi.y = __uint_as_float((__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u);
    hi.z = __uint_as_float((__float_as_uint(v.z) + 0x1000u) & 0xFFFFE000u);
    hi.w = __uint_as_float((__float_as_uint(v.w) + 0x1000u) & 0xFFFFE000u);
    lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// one 16-byte chunk of a tile row: NV float4 of fp32 input -> hi and lo tiles
template <int KIND>
__device__ __forceinline__ void split_store(uint32_t hi_addr, uint32_t lo_addr, const float4 (&v)[KindCfg<KIND>::NV]) {
    if constexpr (KIND == G6D_TC_TF32) {
        float4 hi, lo;
        split_tf32x4(v[0], hi, lo);
        st_shared_v4(hi_addr, __float_as_uint(hi.x), __float_as_uint(hi.y), __float_as_uint(hi.z), __float_as_uint(hi.w));
        st_shared_v4(lo_addr, __float_as_uint(lo.x), __float_as_uint(lo.y), __float_as_uint(lo.z), __float_as_uint(lo.w));
    } else {
        uint32_t h[4], l[4];
        split_f16x2(v[0].x, v[0].y, h[0], l[0]);
        split_f16x2(v[0].z, v[0].w, h[1], l[1]);
        split_f16x2(v[1].x, v[1].y, h[2], l[2]);
        split_f16x2(v[1].z, v[1].w, h[3], l[3]);
        st_shared_v4(hi_addr, h[0], h[1], h[2], h[3]);
        st_shared_v4(lo_addr, l[0], l[1], l[2], l[3]);
    }
}
__device__ __forceinline__ float4 affine4(float4 x, const float4 sc, const float4 sh, bool relu) {
    x.x = fmaf(x.x, sc.x, sh.x); x.y = fmaf(x.y, sc.y, sh.y); x.z = fmaf(x.z, sc.z, sh.z); x.w = fmaf(x.w, sc.w, sh.w);
    if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
    return x;
}

// ------------------------------------------------------------------------------------------ MMA
// cute::UMMA::InstrDescriptor, fp32 accumulate, both operands K-major: c_format F32 (1) at [4,6);
// a_format / b_format at [7,10) / [10,13): TF32 = 2 for kind::tf32, F16 = 0 for kind::f16;
// n_dim = N>>3 at [17,23); m_dim = M>>4 at [24,29).
template <int KIND>
__device__ __forceinline__ uint32_t umma_idesc(int M, int N) {
    constexpr uint32_t fmt = KIND == G6D_TC_TF32 ? 2u : 0u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
template <int KIND>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (KIND == G6D_TC_TF32) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    }
}
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
#define G6D_TMEM_LD16(r, taddr)                                                                                       \
    asm volatile(                                                                                                     \
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"      \
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),             \
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])        \
        : "r"(taddr))

// Fused InstanceNorm statistics of the convolution's OUTPUT (the reference normalises the raw conv
// result and the next layer's loader applies it): each epilogue warp holds 32 output rows x 16 channels
// of final values; a transposing butterfly (8+4+2+1+1 shuffles per quantity) leaves the 32-row sums of
// channel (lane >> 1) in lanes 2c / 2c+1; even lanes add sum(y), odd lanes sum(y^2) to the per
// (group, channel) fp64 accumulators the separate in_stats_partial pass used to produce.  All 32 rows of
// a warp belong to one group (the host only enables this when stats_rows % 32 == 0 / whole planes).
__device__ __forceinline__ void epilogue_stats(float (&v)[16], bool row_valid, double* __restrict__ ws, long long group,
                                               int Cout, int n0, int lane) {
    float q[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { v[j] = row_valid ? v[j] : 0.f; q[j] = v[j] * v[j]; }
#pragma unroll
    for (int half = 8, off = 16; half >= 1; half >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < half; ++j) {
            const float sv = upper ? v[j] : v[j + half], kv = upper ? v[j + half] : v[j];
            const float sq = upper ? q[j] : q[j + half], kq = upper ? q[j + half] : q[j];
            v[j] = kv + __shfl_xor_sync(0xffffffffu, sv, off);
            q[j] = kq + __shfl_xor_sync(0xffffffffu, sq, off);
        }
    }
    const float s1 = v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
    const float s2 = q[0] + __shfl_xor_sync(0xffffffffu, q[0], 1);
    const int n = n0 + (lane >> 1);
    if (n < Cout) atomicAdd(ws + (group * Cout + n) * 2 + (lane & 1), (double)((lane & 1) ? s2 : s1));
}

// ==========================================================================================
// conv_tc2_kernel: persistent implicit-GEMM convolution.
//   * one CTA per SM loops over (M tile, N tile, K split) work items, so there is no wave tail and
//     the per-CTA set-up (TMEM allocation, barrier init, descriptor prefetch) is paid once;
//   * two TMEM accumulator buffers: the MMA warp starts the next tile while four dedicated
//     epilogue warps drain the previous one (tmem_full / tmem_empty barriers);
//   * the eight producer warps keep a register prefetch ring (global loads of the next K-block(s)
//     in flight while K-block it is transformed and stored);
//   * the smem ring never drains between tiles (one global K-block counter).
// TMEM accumulators per buffer: NMAIN round-robin chains for the main (hi*hi) term + one for the
// cross terms.  Each tensor-core accumulate truncates to fp32; spreading the K-blocks over several
// shorter, smaller-magnitude chains (summed in fp32 round-to-nearest by the epilogue) divides the
// resulting bias on same-sign data by ~NMAIN at no cost.
// NPW producer warps + TMA + MMA + 4 epilogue warps.  NPW = 8 is what ships: 16 producer warps (2 tile
// rows per thread, one more K-block of loads in flight) were measured 25-30 % SLOWER on the large layers
// (704 threads cap the kernel at 80 registers: the deeper ring spills into the same L1 data pipe).
constexpr int tc2_threads(int npw) { return (npw + 6) * 32; }
constexpr int TC2_PF_BYTES = 12 * 128;      // weight-tile L2 prefetch distance, in bytes of K per row

template <int BN> struct Tc2Cfg {
    static constexpr int A_BYTES = TC_BM * 128;
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int STAGES = (208 * 1024) / STAGE_BYTES > 6 ? 6 : (208 * 1024) / STAGE_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
    static constexpr int NMAIN = BN == 32 ? 7 : (BN == 64 ? 3 : 1);      // per accumulator buffer
    static constexpr int BUF_COLS = (NMAIN + 1) * BN;                     // 256
    static constexpr int TMEM_COLS = 2 * BUF_COLS;                        // 512: two buffers
};

struct Tc2Work { int m_tiles, n_tiles, total; };

template <int BN, int KIND, int NPW>
__global__ void __launch_bounds__(tc2_threads(NPW), 1)  // 448 threads x 128 registers, or 704 x 80 (warps allocate registers in units of 512)
conv_tc2_kernel(const ConvTcP p, const Tc2Work wk, const __grid_constant__ CUtensorMap map_hi,
                const __grid_constant__ CUtensorMap map_lo) {
    using Cfg = Tc2Cfg<BN>;
    using KC = KindCfg<KIND>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int NMAIN = Cfg::NMAIN;
    constexpr int BK = KC::BK, NV = KC::NV;
    constexpr int ROWS = 32 / NPW;                       // tile rows per producer thread (4 or 2)
    constexpr int RSTEP = NPW * 4;                       // rows r0 + RSTEP*j
    constexpr int RING = KC::RING;                       // register prefetch ring (K-blocks); RING-1 in flight
    constexpr int W_TMA = NPW, W_MMA = NPW + 1;          // warp roles; epilogue = the four warps after W_MMA
    constexpr int PF = TC2_PF_BYTES / 128;     // K-blocks
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bar_base = base + STAGES * Cfg::STAGE_BYTES;
    auto a_hi = [&](int s) { return base + s * Cfg::STAGE_BYTES; };
    auto a_lo = [&](int s) { return base + s * Cfg::STAGE_BYTES + Cfg::A_BYTES; };
    auto b_hi = [&](int s) { return base + s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES; };
    auto b_lo = [&](int s) { return base + s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES + Cfg::B_BYTES; };
    auto full_a = [&](int s) { return bar_base + 8 * s; };
    auto full_b = [&](int s) { return bar_base + 8 * (STAGES + s); };
    auto empty = [&](int s) { return bar_base + 8 * (2 * STAGES + s); };
    auto tmem_full = [&](int b) { return bar_base + 8 * (3 * STAGES + b); };
    auto tmem_empty = [&](int b) { return bar_base + 8 * (3 * STAGES + 2 + b); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base_ptr + STAGES * Cfg::STAGE_BYTES + 8 * (3 * STAGES + 4));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == W_TMA && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_a(s), NPW);        // the producer warps
            mbar_init(full_b(s), 1);
            mbar_init(empty(s), 1);
        }
        for (int b = 0; b < 2; ++b) { mbar_init(tmem_full(b), 1); mbar_init(tmem_empty(b), 4); }
        fence_barrier_init();
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_lo) : "memory");
    }
    if (warp == W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32((const void*)tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;

    // work item -> (m tile, n tile, split); n fastest so neighbouring CTAs share the gathered A rows in L2
    auto decode = [&](int w, int& mt, int& nt, int& sp) {
        nt = w % wk.n_tiles; w /= wk.n_tiles;
        mt = w % wk.m_tiles;
        sp = w / wk.m_tiles;
    };

    if (warp < NPW) {
        // =============================== A producers ===============================
        // All producer warps fill every K-block: ROWS rows x one 16-byte smem chunk (4 or 8 channels) per thread.
        const int chunk = threadIdx.x & 7;
        const int cofs = chunk * 4;                        // this thread's channels inside the K-block: [cofs, cofs+4) (+32 for the 2nd load)
        const int r0 = threadIdx.x >> 3;                   // rows r0 + RSTEP*j, j < ROWS
        int git = 0;                                       // global K-block counter of this CTA
        for (int w = blockIdx.x; w < wk.total; w += gridDim.x) {
            int mt, nt, sp;
            decode(w, mt, nt, sp);
            const int m_base = mt * TC_BM;
            const int kb_begin = sp * p.kb_per_split;
            const int nkb = min(p.kblocks, kb_begin + p.kb_per_split) - kb_begin;
            // Once per tile, so that the K-block loop has no divide: rin = the row's first tap as an input row index
            // (input item * plane + spatial offset); byte j of gd = row j's prologue group minus g0 (bits 0-6; the
            // rows are at most RSTEP * (ROWS - 1) < 128 apart) and its valid flag (bit 7).  The producers sit at the
            // 128-register cap: this is fewer live registers than the (item, spatial offset) pair per row it replaces.
            static_assert(ROWS <= 4 && RSTEP * (ROWS - 1) < 128, "group deltas must fit 7 bits each");
            int rin[ROWS], rc[ROWS];
            int g0 = 0; unsigned gd = 0;
            const long long plane_sz = (long long)p.D * p.H * p.W;
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
                int m = m_base + r0 + RSTEP * j;
                const bool v = m < p.M;
                if (!v) m = 0;
                const int xo = m % p.Wo; m /= p.Wo;
                const int yo = m % p.Ho; m /= p.Ho;
                const int zo = m % p.Do; m /= p.Do;
                const int item = p.in_items == p.B ? m : m % p.in_items;
                const int g = m / (int)p.group_rows;                                  // 32-bit divide (host checks the range)
                if (j == 0) g0 = g;
                if (v) gd |= ((unsigned)(g - g0) | 0x80u) << (8 * j);
                const int z = zo * p.stride - p.pd, y = yo * p.stride - p.ph, x = xo * p.stride - p.pw;
                rin[j] = item * (int)plane_sz + (z * p.H + y) * p.W + x;        // < 2^31 (host checks)
                rc[j] = ((z + 8) << 24) | ((y + 8) << 12) | (x + 8);
            }
            int c0, kx, ky, kz;
            {
                const int k = kb_begin * BK;
                int tap = 0; c0 = k;
                if (p.K != p.Cin) { tap = k / p.Cin; c0 = k - tap * p.Cin; }
                kx = tap % p.kw; const int tq = tap / p.kw; ky = tq % p.kh; kz = tq / p.kh;
            }
            // prefetch ring: slot q holds K-block (it % RING == q)
            float4 v[RING][ROWS][NV];
            unsigned okm[RING]; int kc[RING]; int ksp[RING];
            auto issue_loads = [&](int q) {
                const int tap_sp = (kz * p.H + ky) * p.W + kx;
                okm[q] = 0; kc[q] = c0 + cofs; ksp[q] = tap_sp;
                const float* xb = p.x + p.ico + cofs + c0;
#pragma unroll
                for (int j = 0; j < ROWS; ++j) {
                    const int z = ((rc[j] >> 24) & 0xff) - 8 + kz, y = ((rc[j] >> 12) & 0xfff) - 8 + ky, x = (rc[j] & 0xfff) - 8 + kx;
                    const bool inb = ((gd >> (8 * j + 7)) & 1u) && (unsigned)z < (unsigned)p.D && (unsigned)y < (unsigned)p.H &&
                                     (unsigned)x < (unsigned)p.W;
#pragma unroll
                    for (int e = 0; e < NV; ++e) v[q][j][e] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (inb) {
                        const float4* src = reinterpret_cast<const float4*>(xb + (long long)(rin[j] + tap_sp) * p.ics);
#pragma unroll
                        for (int e = 0; e < NV; ++e) v[q][j][e] = __ldg(src + e * 8);
                        okm[q] |= 1u << j;
                    }
                }
                c0 += BK;
                if (c0 == p.Cin) { c0 = 0; if (++kx == p.kw) { kx = 0; if (++ky == p.kh) { ky = 0; ++kz; } } }
            };
            auto process = [&](int q, int it) {
                const int g_it = git + it;
                const int s = g_it % STAGES;
                const uint32_t n_use = g_it / STAGES;
                if (p.pro != G6D_PRO_NONE) {
                    const bool relu = p.pro == G6D_PRO_AFFINE_RELU;
#pragma unroll
                    for (int j = 0; j < ROWS; ++j) {
                        if (okm[q] & (1u << j)) {
                            const float4* scp; const float4* shp;
                            const int gc = (g0 + (int)((gd >> (8 * j)) & 0x7fu)) * p.Cin;
                            const int sh = gc + kc[q];
                            if (p.pro == G6D_PRO_CORR) {       // scale[g, pos, c]: the spatial offset again from rc
                                const int rsp = ((((rc[j] >> 24) & 0xff) - 8) * p.H + ((rc[j] >> 12) & 0xfff) - 8) * p.W + (rc[j] & 0xfff) - 8;
                                scp = reinterpret_cast<const float4*>(p.ps + (gc * (int)plane_sz + (rsp + ksp[q]) * p.Cin + kc[q]));
                            } else {
                                scp = reinterpret_cast<const float4*>(p.ps + sh);
                            }
                            shp = reinterpret_cast<const float4*>(p.pb + sh);
#pragma unroll
                            for (int e = 0; e < NV; ++e) v[q][j][e] = affine4(v[q][j][e], __ldg(scp + e * 8), __ldg(shp + e * 8), relu);
                        }
                    }
                }
                mbar_wait(empty(s), (n_use & 1) ^ 1, 1, g_it);
#pragma unroll
                for (int j = 0; j < ROWS; ++j) {
                    const int r = r0 + RSTEP * j;
                    const uint32_t so = r * 128 + ((chunk ^ (r & 7)) << 4);        // Swizzle<3,4,3>
                    split_store<KIND>(a_hi(s) + so, a_lo(s) + so, v[q][j]);
                }
                fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) mbar_arrive(full_a(s));
            };
            // software pipeline, unrolled by RING so the ring slots are compile-time register names
#pragma unroll
            for (int q = 0; q < RING - 1; ++q)
                if (q < nkb) issue_loads(q);
            for (int it = 0; it < nkb; it += RING) {
#pragma unroll
                for (int q = 0; q < RING; ++q) {
                    if (it + q < nkb) {
                        if (it + q + RING - 1 < nkb) issue_loads((q + RING - 1) % RING);
                        process(q, it + q);
                    }
                }
            }
            git += nkb;
        }
    } else if (warp == W_TMA) {
        // =============================== B producer (TMA) ===============================
        if (lane == 0) {
            int git = 0;
            for (int w = blockIdx.x; w < wk.total; w += gridDim.x) {
                int mt, nt, sp;
                decode(w, mt, nt, sp);
                const int kb_begin = sp * p.kb_per_split;
                const int nkb = min(p.kblocks, kb_begin + p.kb_per_split) - kb_begin;
                // The weight tiles of a small-M layer are touched once and come from HBM: with only
                // STAGES tiles in flight the ring is latency-bound (measured 5000 cycles per K-block
                // at M = 660).  An L2 prefetch running PF K-blocks ahead costs no shared memory.
                for (int it = 0; it < min(nkb, PF); ++it) {
                    tma_prefetch_2d(&map_hi, (kb_begin + it) * BK, nt * BN);
                    tma_prefetch_2d(&map_lo, (kb_begin + it) * BK, nt * BN);
                }
                for (int it = 0; it < nkb; ++it, ++git) {
                    const int s = git % STAGES;
                    if (it + PF < nkb) {
                        tma_prefetch_2d(&map_hi, (kb_begin + it + PF) * BK, nt * BN);
                        tma_prefetch_2d(&map_lo, (kb_begin + it + PF) * BK, nt * BN);
                    }
                    mbar_wait(empty(s), ((git / STAGES) & 1) ^ 1, 3, git);
                    mbar_expect_tx(full_b(s), 2 * Cfg::B_BYTES);
                    const int k = (kb_begin + it) * BK;
                    tma_load_2d(b_hi(s), &map_hi, full_b(s), k, nt * BN);
                    tma_load_2d(b_lo(s), &map_lo, full_b(s), k, nt * BN);
                }
            }
        }
    } else if (warp == W_MMA) {
        // =============================== MMA issuer ===============================
        if (elect_one_sync()) {
            const uint32_t idesc = umma_idesc<KIND>(TC_BM, BN);
            int git = 0, tile = 0;
            for (int w = blockIdx.x; w < wk.total; w += gridDim.x, ++tile) {
                int mt, nt, sp;
                decode(w, mt, nt, sp);
                const int kb_begin = sp * p.kb_per_split;
                const int nkb = min(p.kblocks, kb_begin + p.kb_per_split) - kb_begin;
                const int buf = tile & 1;
                mbar_wait(tmem_empty(buf), ((tile >> 1) & 1) ^ 1, 6, tile);     // epilogue has drained this buffer
                tc_fence_after();
                const uint32_t acc0 = tmem_acc + (uint32_t)(buf * Cfg::BUF_COLS);
                for (int it = 0; it < nkb; ++it, ++git) {
                    const int s = git % STAGES;
                    mbar_wait(full_a(s), (git / STAGES) & 1, 4, git);
                    mbar_wait(full_b(s), (git / STAGES) & 1, 5, git);
                    tc_fence_after();
                    const uint64_t dah = umma_desc_sw128(a_hi(s)), dal = umma_desc_sw128(a_lo(s));
                    const uint64_t dbh = umma_desc_sw128(b_hi(s)), dbl = umma_desc_sw128(b_lo(s));
                    const uint32_t main_acc = acc0 + (uint32_t)((it % NMAIN) * BN);
                    const uint32_t cross_acc = acc0 + (uint32_t)(NMAIN * BN);
                    if constexpr (BN == 128 && NMAIN == 1) {
                        // B_hi and B_lo sit back to back in the stage (a 256-row K-major tile) and the main and
                        // cross accumulators back to back in TMEM: ONE N = 256 MMA forms A_hi * [B_hi | B_lo],
                        // reading A_hi from shared memory once instead of twice (20 KB of operand reads per
                        // K-step instead of 24; same 192 tensor cycles).  Then cross += A_lo * B_hi.
                        const uint32_t idesc2 = umma_idesc<KIND>(TC_BM, 2 * BN);
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);
                            umma<KIND>(acc0, dah + adv, dbh + adv, idesc2, (it > 0 || ks > 0) ? 1u : 0u);
                            umma<KIND>(cross_acc, dal + adv, dbh + adv, idesc, 1u);
                        }
                    } else {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {                 // 4 x 32 bytes of K per 128-byte row
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);
                            umma<KIND>(cross_acc, dal + adv, dbh + adv, idesc, (it > 0 || ks > 0) ? 1u : 0u);
                            umma<KIND>(cross_acc, dah + adv, dbl + adv, idesc, 1u);
                            umma<KIND>(main_acc, dah + adv, dbh + adv, idesc, (it >= NMAIN || ks > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit(empty(s));
                }
                umma_commit(tmem_full(buf));
            }
        }
    } else {
        // =============================== epilogue (the 4 warps after the MMA warp) ===============================
        const int quad = warp & 3;                     // TMEM lane quadrant = warp id % 4
        int tile = 0;
        for (int w = blockIdx.x; w < wk.total; w += gridDim.x, ++tile) {
            int mt, nt, sp;
            decode(w, mt, nt, sp);
            const int kb_begin = sp * p.kb_per_split;
            const int nkb = min(p.kblocks, kb_begin + p.kb_per_split) - kb_begin;
            const int buf = tile & 1;
            mbar_wait(tmem_full(buf), (tile >> 1) & 1, 2, tile);
            tc_fence_after();
            const int m = mt * TC_BM + quad * 32 + lane;
            const int n_base = nt * BN;
            const bool partial = p.splits > 1;
            // 128-bit stores need 16-byte aligned rows: channel strides / offsets multiples of 4 floats
            const bool vec_ok = partial ? (p.Cout & 3) == 0
                                        : ((p.ocs & 3) == 0 && (p.oco & 3) == 0 && (reinterpret_cast<uintptr_t>(p.y) & 15) == 0 &&
                                           (!p.bias || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0));
            const int n_acc = nkb < NMAIN ? nkb : NMAIN;
            const uint32_t tbase = tmem_acc + (uint32_t)(buf * Cfg::BUF_COLS) + ((uint32_t)(quad * 32) << 16);
#pragma unroll 1
            for (int cc = 0; cc < BN; cc += 16) {
                float accv[16];
                {   // cross terms first (smallest magnitude), scaled back by the lo pre-scale
                    uint32_t r[16];
                    G6D_TMEM_LD16(r, tbase + (uint32_t)(NMAIN * BN + cc));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) accv[j] = __uint_as_float(r[j]) * KC::CROSS;
                }
#pragma unroll
                for (int a = 0; a < NMAIN; ++a) {
                    if (a < n_acc) {
                        uint32_t r[16];
                        G6D_TMEM_LD16(r, tbase + (uint32_t)(a * BN + cc));
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int j = 0; j < 16; ++j) accv[j] += __uint_as_float(r[j]);
                    }
                }
                const int n0 = n_base + cc;
                if (!partial) {
                    if (p.bias) {
                        if (vec_ok && n0 + 16 <= p.Cout) {          // 4 x 128-bit (L1-broadcast) bias loads
#pragma unroll
                            for (int j4 = 0; j4 < 4; ++j4) {
                                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0) + j4);
                                accv[j4 * 4] += bb.x; accv[j4 * 4 + 1] += bb.y; accv[j4 * 4 + 2] += bb.z; accv[j4 * 4 + 3] += bb.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (n0 + j < p.Cout) accv[j] += __ldg(p.bias + n0 + j);
                        }
                    }
                    if (p.act != G6D_ACT_NONE) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) accv[j] = tc_act(accv[j], p.act);
                    }
                }
                if (m < p.M) {
                    float* dst = partial ? p.ws + ((long long)sp * p.M + m) * p.Cout + n0
                                         : p.y + (long long)m * p.ocs + p.oco + n0;
                    if (vec_ok && n0 + 16 <= p.Cout) {      // 4 x 128-bit stores per thread instead of 16 scalar ones
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4)
                            reinterpret_cast<float4*>(dst)[j4] = make_float4(accv[j4 * 4], accv[j4 * 4 + 1], accv[j4 * 4 + 2], accv[j4 * 4 + 3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (n0 + j < p.Cout) dst[j] = accv[j];
                    }
                }
                if (p.stats && !partial)
                    epilogue_stats(accv, m < p.M, p.stats, (long long)(mt * TC_BM + quad * 32) / p.stats_rows, p.Cout, n0, lane);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty(buf));
        }
    }
    __syncthreads();
    if (warp == W_MMA) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "n"(Cfg::TMEM_COLS) : "memory");
    }
}

// Split-K epilogue: y = act(sum_s ws[s] + bias); one thread per output element.
__global__ void conv_tc_reduce_kernel(const float* __restrict__ ws, const float* __restrict__ bias,
                                      float* __restrict__ y, int M, int Cout, int splits, int ocs, int oco, int act) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * Cout) return;
    const int n = (int)(i % Cout);
    const long long m = i / Cout;
    float v = 0.f;
    for (int s = 0; s < splits; ++s) v += ws[(long long)s * M * Cout + i];
    if (bias) v += bias[n];
    y[m * ocs + oco + n] = tc_act(v, act);
}

// The same with the fused InstanceNorm statistics of y: a 256-thread block owns 32 consecutive output
// rows (one group: stats_rows % 32 == 0) x 64 channels; thread = (channel, 8-row slice); the four slices
// are combined in shared memory and one (sum, sum^2) pair per (block, channel) goes to the fp64 accumulators.
__global__ void __launch_bounds__(256) conv_tc_reduce_stats_kernel(const float* __restrict__ ws, const float* __restrict__ bias,
                                                                   float* __restrict__ y, int M, int Cout, int splits, int ocs,
                                                                   int oco, int act, double* __restrict__ stats, long long stats_rows) {
    __shared__ float red[2][4][64];
    const int c = threadIdx.x & 63, rg = threadIdx.x >> 6;
    const int n = blockIdx.y * 64 + c;
    const int m0 = blockIdx.x * 32 + rg * 8;
    const long long slab = (long long)M * Cout;
    float s1 = 0.f, s2 = 0.f;
    if (n < Cout) {
        const float b = bias ? bias[n] : 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int m = m0 + r;
            if (m < M) {
                const long long i = (long long)m * Cout + n;
                float v = 0.f;
                for (int s = 0; s < splits; ++s) v += ws[(long long)s * slab + i];
                v = tc_act(v + b, act);
                y[(long long)m * ocs + oco + n] = v;
                s1 += v; s2 = fmaf(v, v, s2);
            }
        }
    }
    red[0][rg][c] = s1; red[1][rg][c] = s2;
    __syncthreads();
    if (threadIdx.x < 128) {
        const int q = threadIdx.x >> 6;                       // 0: sum, 1: sum of squares
        const float t = red[q][0][c] + red[q][1][c] + red[q][2][c] + red[q][3][c];
        if (n < Cout) atomicAdd(stats + ((long long)((blockIdx.x * 32) / stats_rows) * Cout + n) * 2 + q, (double)t);
    }
}

static void launch_reduce(const float* ws, const float* bias, float* y, int M, int Cout, int splits, int ocs, int oco, int act,
                          double* stats, long long stats_rows, cudaStream_t st) {
    if (stats) {
        dim3 grid(ceil_div(M, 32), ceil_div(Cout, 64));
        conv_tc_reduce_stats_kernel<<<grid, 256, 0, st>>>(ws, bias, y, M, Cout, splits, ocs, oco, act, stats, stats_rows);
    } else {
        const long long n = (long long)M * Cout;
        conv_tc_reduce_kernel<<<ceil_div(n, 256), 256, 0, st>>>(ws, bias, y, M, Cout, splits, ocs, oco, act);
    }
}

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

static int kind_bk(int kind) { return kind == G6D_TC_F16 ? 64 : 32; }
static int kind_esize(int kind) { return kind == G6D_TC_F16 ? 2 : 4; }

// 2-D tensor map over W [rows = Cout_pad, cols = K] (K-major), box = [one 128-byte swizzle row of K, bn rows]
static int make_weight_map(CUtensorMap* map, const void* w, int rows, int K, int bn, int kind) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("g6d_conv_tc: cuTensorMapEncodeTiled unavailable"); return G6D_ECUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K * kind_esize(kind)};
    cuuint32_t box[2] = {(cuuint32_t)kind_bk(kind), (cuuint32_t)bn};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, kind == G6D_TC_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                     const_cast<void*>(w), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("g6d_conv_tc: cuTensorMapEncodeTiled failed (%d)", (int)r); return G6D_ECUDA; }
    return G6D_OK;
}

static int tc_block_n(int Cout) { return Cout > 64 ? 128 : (Cout > 32 ? 64 : 32); }

// the persistent kernel packs (z, y, x) + 8 into 8/12/12 bits and uses 32-bit spatial offsets and group indices
static bool tc2_dims_ok(const g6d_conv_desc* d) {
    return d->D + d->pd + 8 < 256 && d->H + d->ph + 8 < 4096 && d->W + d->pw + 8 < 4096 &&
           (long long)d->D * d->H * d->W < (1ll << 30) && d->group_rows < (1ll << 31) &&
           (long long)(d->in_items > 0 ? d->in_items : d->B) * d->D * d->H * d->W < (1ll << 31);
}

static int fill_tc_params(const g6d_conv_desc* d, int kind, ConvTcP& p) {
    G6D_REQUIRE(d != nullptr, "g6d_conv_tc: null desc");
    G6D_REQUIRE(kind == G6D_TC_TF32 || kind == G6D_TC_F16, "g6d_conv_tc: bad operand kind %d", kind);
    G6D_REQUIRE(d->B > 0 && d->D > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0, "g6d_conv_tc: bad dims");
    G6D_REQUIRE(d->kd > 0 && d->kh > 0 && d->kw > 0 && d->stride > 0, "g6d_conv_tc: bad kernel/stride");
    const int bk = kind_bk(kind);
    G6D_REQUIRE((d->Cin % bk) == 0, "g6d_conv_tc: Cin (%d) must be a multiple of %d", d->Cin, bk);
    G6D_REQUIRE((d->in_cstride & 3) == 0 && (d->in_coff & 3) == 0, "g6d_conv_tc: in_cstride/in_coff must be multiples of 4");
    G6D_REQUIRE(d->in_coff + d->Cin <= d->in_cstride, "g6d_conv_tc: input channel slice out of row");
    G6D_REQUIRE(d->out_coff + d->Cout <= d->out_cstride, "g6d_conv_tc: output channel slice out of row");
    G6D_REQUIRE(in_items_ok(d), "g6d_conv_tc: in_items (%d) must be 0 or divide B (%d)", d->in_items, d->B);
    G6D_REQUIRE(pro_operands_fit(d), "g6d_conv_tc: prologue operands too large");
    G6D_REQUIRE(tc2_dims_ok(d), "g6d_conv_tc: spatial extent too large for the tensor-core kernel");
    const int Do = (d->D + 2 * d->pd - d->kd) / d->stride + 1;
    const int Ho = (d->H + 2 * d->ph - d->kh) / d->stride + 1;
    const int Wo = (d->W + 2 * d->pw - d->kw) / d->stride + 1;
    G6D_REQUIRE(Do == d->Do && Ho == d->Ho && Wo == d->Wo, "g6d_conv_tc: output dims mismatch");
    G6D_REQUIRE(d->prologue >= 0 && d->prologue <= 3 && d->act >= 0 && d->act <= 2, "g6d_conv_tc: bad prologue/act");
    const long long M = (long long)d->B * Do * Ho * Wo;
    const long long K = (long long)d->kd * d->kh * d->kw * d->Cin;
    G6D_REQUIRE(M < (1ll << 31) && K < (1ll << 31), "g6d_conv_tc: problem too large");
    p.B = d->B; p.D = d->D; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.ics = d->in_cstride; p.ico = d->in_coff;
    p.Cout = d->Cout; p.kd = d->kd; p.kh = d->kh; p.kw = d->kw; p.stride = d->stride; p.pd = d->pd; p.ph = d->ph;
    p.pw = d->pw; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.ocs = d->out_cstride; p.oco = d->out_coff; p.pro = d->prologue;
    p.act = d->act; p.group_rows = d->group_rows > 0 ? d->group_rows : 1;
    p.in_items = d->in_items > 0 ? d->in_items : d->B;
    p.M = (int)M; p.K = (int)K; p.kblocks = (int)(K / bk);
    const int bn = tc_block_n(d->Cout);
    const long long ctas = (long long)ceil_div(M, TC_BM) * ceil_div(d->Cout, bn);
    const int min_kb = 256 / bk;                     // never split below 256 K-elements per item
    int splits = 1;
    if (ctas < kNumSMs && p.kblocks >= 2 * min_kb) {
        // as many K splits as still fit in ONE wave of the 148 persistent CTAs (a second, partial wave
        // of long items costs more than the parallelism it adds)
        splits = (int)(kNumSMs / ctas);
        splits = splits > p.kblocks / min_kb ? p.kblocks / min_kb : splits;
        splits = splits < 1 ? 1 : splits;
    }
    // The tensor core adds each K-step into the fp32 accumulator with truncation; over very long
    // K chains of same-sign products (detector correlation: K = 115200 of post-ReLU features)
    // that is a systematic bias of ~4e-5 relative.  For long-K problems (K > 8192) the chain per
    // CTA is bounded to 2048 terms and the partials are summed in fp32 round-to-nearest.
    // d->max_chain_k bounds the K-elements per ACCUMULATOR; a split rotates over NMAIN of them
    const int nmain = bn == 32 ? Tc2Cfg<32>::NMAIN : (bn == 64 ? Tc2Cfg<64>::NMAIN : Tc2Cfg<128>::NMAIN);
    const int chain = d->max_chain_k > 0 ? d->max_chain_k * nmain : (K > 8192 ? TC_MAX_K_PER_CHAIN : 0);
    const int max_kb = chain > bk ? chain / bk : 1;
    const int min_splits = chain > 0 ? (p.kblocks + max_kb - 1) / max_kb : 1;
    splits = splits < min_splits ? min_splits : splits;
    splits = splits > 64 ? 64 : splits;
    p.kb_per_split = (p.kblocks + splits - 1) / splits;
    p.splits = (p.kblocks + p.kb_per_split - 1) / p.kb_per_split;
    return G6D_OK;
}

template <int BN, int KIND, int NPW = 8>
static int launch_tc2(const ConvTcP& p, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
    using Cfg = Tc2Cfg<BN>;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc2_kernel<BN, KIND, NPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
        if (e != cudaSuccess) { set_error("g6d_conv_tc: cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return G6D_ECUDA; }
        configured = true;
    }
    Tc2Work wk;
    wk.m_tiles = ceil_div(p.M, TC_BM); wk.n_tiles = ceil_div(p.Cout, BN);
    const long long total = (long long)wk.m_tiles * wk.n_tiles * p.splits;
    wk.total = (int)total;
    const int grid = total < kNumSMs ? (int)total : kNumSMs;
    conv_tc2_kernel<BN, KIND, NPW><<<grid, tc2_threads(NPW), Cfg::SMEM_BYTES, st>>>(p, wk, mh, ml);
    G6D_CHECK_LAUNCH("g6d_conv_tc");
    return G6D_OK;
}

// elementwise operand split of an fp32 array (detector reference features used as kernels)
__global__ void split_tf32_kernel(const float* __restrict__ in, float* __restrict__ hi, float* __restrict__ lo, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = in[i];
    const float h = to_tf32(v);
    hi[i] = h;
    lo[i] = to_tf32(v - h);
}
__device__ __forceinline__ void split_f16_scalar(float v, __half& h, __half& l) {
    uint32_t hh, ll;
    split_f16x2(v, 0.f, hh, ll);
    h = __ushort_as_half((unsigned short)(hh & 0xffffu));
    l = __ushort_as_half((unsigned short)(ll & 0xffffu));
}
// rows of K-major operands, K a multiple of 64: position p of every 64-block comes from source f16_k_source(p)
__global__ void split_f16_kernel(const float* __restrict__ in, __half* __restrict__ hi, __half* __restrict__ lo, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    split_f16_scalar(in[(i & ~63ll) + f16_k_source((int)(i & 63))], hi[i], lo[i]);
}

// [Cout, Cin, taps] (reference layout) -> hi/lo [rows_pad, taps*Cin_pad], K index = tap*Cin_pad + c
template <int KIND>
__global__ void pack_conv_weight_tc_kernel(const float* __restrict__ w, void* __restrict__ hi, void* __restrict__ lo,
                                           int Cout, int Cin, int Cin_pad, int taps, int rows_pad,
                                           const float* __restrict__ scale) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long K = (long long)taps * Cin_pad;
    if (i >= K * rows_pad) return;
    const int o = (int)(i / K);
    const long long k = i % K;
    const int tap = (int)(k / Cin_pad);
    int c = (int)(k % Cin_pad);
    if constexpr (KIND == G6D_TC_F16) c = (c & ~63) + f16_k_source(c & 63);       // K order of the fp16 K-block
    float v = 0.f;
    if (o < Cout && c < Cin) {
        v = w[((long long)o * Cin + c) * taps + tap];
        if (scale) v *= scale[o];
    }
    if constexpr (KIND == G6D_TC_TF32) {
        const float h = to_tf32(v);
        static_cast<float*>(hi)[i] = h;
        static_cast<float*>(lo)[i] = to_tf32(v - h);
    } else {
        split_f16_scalar(v, static_cast<__half*>(hi)[i], static_cast<__half*>(lo)[i]);
    }
}

// ==========================================================================================
// conv_tcflat_kernel: stride-1 convolutions with A-operand reuse across taps.
//
// The output positions of one image plane are enumerated over the PADDED width Wp = W + 2*pw:
// f = y*Wp + x.  Tap (ky,kx) of output f reads padded-input position f + ky*Wp + kx, so for a
// tile of 128 consecutive f the A operand of EVERY tap is a window of 128 consecutive rows of
// one shared-memory buffer holding padded-input positions [f0, f0 + 127 + (kh-1)*Wp + kw-1]:
// the tap is selected by the UMMA descriptor's start address (+shift*128 B; the 128B swizzle is a
// function of the absolute smem address, verified by g6d_debug_umma_shift).  The producers
// therefore gather (and prologue-transform, and hi/lo split) each input element ONCE per channel
// block instead of once per tap: 9x less producer work / L2 traffic for 3x3 ("FLAT" mode).  When
// the halo (kh-1)*Wp does not fit in shared memory (wide images, 15x15 correlation kernels) the
// buffer holds one kernel row at a time ("ROW" mode: kw-fold reuse).  Columns x >= Wo of the
// padded enumeration are computed and dropped.  B tiles stream by TMA per (channel block, tap).
struct ConvFlatP {
    const float* x; const float* bias; const float* ps; const float* pb; float* y; float* ws;
    int B, D, H, W, Cin, ics, ico, Cout, kd, kh, kw, pd, ph, pw, Do, Ho, Wo, ocs, oco, pro, act;
    long long group_rows;
    int in_items;
    int Wp, tiles_per_plane, mode, nseg, taps_per_seg, seg_rows, rows_pad, ntab, cblocks;
    int a_stages, b_stages, splits, cb_per_split, M;
    double* stats; long long stats_rows;
};

template <int BN> struct FlatCfg {
    static constexpr int NMAIN = BN == 32 ? 7 : (BN == 256 ? 1 : 3);
    static constexpr int TMEM_COLS = (NMAIN + 1) * BN;             // 256 / 256 / 512 columns
};

template <int BN, int KIND>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tcflat_kernel(const ConvFlatP p, const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo) {
    using KC = KindCfg<KIND>;
    constexpr int NMAIN = FlatCfg<BN>::NMAIN;
    constexpr int TMEM_COLS = FlatCfg<BN>::TMEM_COLS;
    constexpr int B_BYTES = BN * 128;
    constexpr int BK = KC::BK, NV = KC::NV;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const int A_TILE = p.rows_pad * 128;                 // one of hi / lo
    const uint32_t a_base = base;
    const uint32_t b_base = base + p.a_stages * 2 * A_TILE;
    const uint32_t bar_base = b_base + p.b_stages * 2 * B_BYTES;
    auto a_hi = [&](int s) { return a_base + s * 2 * A_TILE; };
    auto a_lo = [&](int s) { return a_base + s * 2 * A_TILE + A_TILE; };
    auto b_hi = [&](int s) { return b_base + s * 2 * B_BYTES; };
    auto b_lo = [&](int s) { return b_base + s * 2 * B_BYTES + B_BYTES; };
    auto a_full = [&](int s) { return bar_base + 8 * s; };
    auto a_empty = [&](int s) { return bar_base + 8 * (4 + s); };
    auto b_full = [&](int s) { return bar_base + 8 * (8 + s); };
    auto b_empty = [&](int s) { return bar_base + 8 * (12 + s); };
    const uint32_t tmem_full = bar_base + 8 * 16;
    const uint32_t bar_off = (bar_base - base);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base_ptr + bar_off + 8 * 17);
    int* rowtab = reinterpret_cast<int*>(base_ptr + bar_off + 256);   // [ntab][seg_rows]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int tile = blockIdx.x;
    const int t_in_plane = tile % p.tiles_per_plane; tile /= p.tiles_per_plane;
    const int zo = tile % p.Do;
    const int b = tile / p.Do;
    const int f0 = t_in_plane * TC_BM;
    const int n_base = blockIdx.y * BN;
    const int split = blockIdx.z;
    const int cb_begin = split * p.cb_per_split;
    const int cb_end = min(p.cblocks, cb_begin + p.cb_per_split);
    const int nunits = (cb_end - cb_begin) * p.nseg;

    // ---- setup: row tables (element offset of each gathered row inside its image plane, -1 = zero)
    for (int e = threadIdx.x; e < p.ntab * p.seg_rows; e += blockDim.x) {
        const int tb = e / p.seg_rows, i = e % p.seg_rows;
        const int g = f0 + (p.mode == 1 ? tb * p.Wp : 0) + i;     // padded-input flat position
        const int yy = g / p.Wp - p.ph, xx = g % p.Wp - p.pw;
        rowtab[e] = ((unsigned)yy < (unsigned)p.H && (unsigned)xx < (unsigned)p.W) ? yy * p.W + xx : -1;
    }
    if (warp == TC_PRODUCER_WARPS && lane == 0) {
        for (int s = 0; s < 4; ++s) {
            mbar_init(a_full(s), TC_PRODUCER_WARPS);
            mbar_init(a_empty(s), 1);
            mbar_init(b_full(s), 1);
            mbar_init(b_empty(s), 1);
        }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_lo) : "memory");
    }
    if (warp == TC_PRODUCER_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32((const void*)tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;

    if (warp < TC_PRODUCER_WARPS) {
        // =============================== A producers ===============================
        const int chunk = threadIdx.x & 7;
        const int cofs = chunk * 4;                             // channels [cofs, cofs+4) (+32 for the 2nd load), see f16_k_source
        const int r0 = threadIdx.x >> 3;                        // rows r0 + 32*j
        const long long plane = (long long)p.H * p.W;
        const long long gi = (long long)b / p.group_rows;        // prologue group of the output item
        const int b_in = p.in_items == p.B ? b : b % p.in_items;  // the input item it reads
        const bool relu = p.pro == G6D_PRO_AFFINE_RELU;
        // Software pipeline over (unit, 128-row trip) with a ring of NB register slots: the global loads of
        // the next NB-1 trips (possibly of the next unit: they only touch registers, so they do not wait for
        // the stage to be free) are in flight while a trip is transformed and stored.  Without it every trip
        // paid a full L2 round trip before its first st.shared.
        constexpr int NB = 3;
        const int trips = (p.seg_rows + 127) / 128;
        const int total = nunits * trips;
        float4 v[NB][4][NV]; int off[NB][4];
        auto unit_of = [&](int tt, int& u, int& rbase, int& cb, int& kz, int& tb) {
            u = tt / trips; rbase = (tt - u * trips) * 128;
            cb = cb_begin + u / p.nseg;
            const int seg = u % p.nseg;
            // FLAT: seg = kz, table 0.  ROW: seg = kz*kh + ky, table ky.
            kz = p.mode == 1 ? seg / p.kh : seg;
            tb = p.mode == 1 ? seg % p.kh : 0;
        };
        auto issue = [&](int tt, int q) {
            int u, rbase, cb, kz, tb;
            unit_of(tt, u, rbase, cb, kz, tb);
            const int zz = zo + kz - p.pd;
            const bool zok = (unsigned)zz < (unsigned)p.D;
            const float* xplane = p.x + ((long long)b_in * p.D + (zok ? zz : 0)) * plane * p.ics + p.ico + cb * BK + cofs;
            const int* tab = rowtab + tb * p.seg_rows;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = rbase + r0 + 32 * j;
                off[q][j] = (r < p.seg_rows && zok) ? tab[r] : -1;
#pragma unroll
                for (int e = 0; e < NV; ++e) v[q][j][e] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (off[q][j] >= 0) {
                    const float4* src = reinterpret_cast<const float4*>(xplane + (long long)off[q][j] * p.ics);
#pragma unroll
                    for (int e = 0; e < NV; ++e) v[q][j][e] = __ldg(src + e * 8);
                }
            }
        };
        auto store = [&](int tt, int q) {
            int u, rbase, cb, kz, tb;
            unit_of(tt, u, rbase, cb, kz, tb);
            const int s = u % p.a_stages;
            const int zz = zo + kz - p.pd;
            const int c = cb * BK + cofs;
            if (rbase == 0) mbar_wait(a_empty(s), ((u / p.a_stages) & 1) ^ 1, 1, u);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = rbase + r0 + 32 * j;
                if (r >= p.rows_pad) continue;
                if (p.pro != G6D_PRO_NONE && off[q][j] >= 0) {
                    const float4* scp; const float4* shp;
                    if (p.pro == G6D_PRO_CORR) {
                        const long long sp = (gi * p.D + zz) * plane + off[q][j];
                        scp = reinterpret_cast<const float4*>(p.ps + sp * p.Cin + c);
                        shp = reinterpret_cast<const float4*>(p.pb + gi * p.Cin + c);
                    } else {
                        scp = reinterpret_cast<const float4*>(p.ps + gi * p.Cin + c);
                        shp = reinterpret_cast<const float4*>(p.pb + gi * p.Cin + c);
                    }
#pragma unroll
                    for (int e = 0; e < NV; ++e) v[q][j][e] = affine4(v[q][j][e], __ldg(scp + e * 8), __ldg(shp + e * 8), relu);
                }
                const uint32_t so = r * 128 + ((chunk ^ (r & 7)) << 4);
                split_store<KIND>(a_hi(s) + so, a_lo(s) + so, v[q][j]);
            }
            if (rbase + 128 >= p.seg_rows) {          // last trip of the unit: publish the stage
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full(s));
            }
        };
#pragma unroll
        for (int q = 0; q < NB - 1; ++q)
            if (q < total) issue(q, q);
        for (int tt = 0; tt < total; tt += NB) {
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                if (tt + q < total) {
                    if (tt + q + NB - 1 < total) issue(tt + q + NB - 1, (q + NB - 1) % NB);
                    store(tt + q, q);
                }
            }
        }

        // =============================== epilogue ===============================
        mbar_wait(tmem_full, 0, 2, nunits);
        tc_fence_after();
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        const int f = f0 + row;
        const int yo = f / p.Wp, xo = f % p.Wp;
        const bool valid = yo < p.Ho && xo < p.Wo;
        const long long m = (((long long)b * p.Do + zo) * p.Ho + yo) * p.Wo + xo;
        constexpr int HALF = BN / 2;
        const int col0 = (warp >> 2) * HALF;
        const bool partial = p.splits > 1;
        const bool vec_ok = partial ? (p.Cout & 3) == 0
                                    : ((p.ocs & 3) == 0 && (p.oco & 3) == 0 && (reinterpret_cast<uintptr_t>(p.y) & 15) == 0 &&
                                       (!p.bias || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0));
        const int total_mm = nunits * p.taps_per_seg;
        const int n_acc = total_mm < NMAIN ? total_mm : NMAIN;
#pragma unroll
        for (int cc = 0; cc < HALF; cc += 16) {
            float accv[16];
            const uint32_t taddr = tmem_acc + ((uint32_t)(quad * 32) << 16) + (uint32_t)(col0 + cc);
            {
                uint32_t r[16];
                G6D_TMEM_LD16(r, taddr + (uint32_t)(NMAIN * BN));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 16; ++j) accv[j] = __uint_as_float(r[j]) * KC::CROSS;
            }
#pragma unroll
            for (int a = 0; a < NMAIN; ++a) {
                if (a < n_acc) {
                    uint32_t r[16];
                    G6D_TMEM_LD16(r, taddr + (uint32_t)(a * BN));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) accv[j] += __uint_as_float(r[j]);
                }
            }
            const int n0 = n_base + col0 + cc;
            if (!partial) {
                if (p.bias) {
                    if (vec_ok && n0 + 16 <= p.Cout) {
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0) + j4);
                            accv[j4 * 4] += bb.x; accv[j4 * 4 + 1] += bb.y; accv[j4 * 4 + 2] += bb.z; accv[j4 * 4 + 3] += bb.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (n0 + j < p.Cout) accv[j] += __ldg(p.bias + n0 + j);
                    }
                }
                if (p.act != G6D_ACT_NONE) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) accv[j] = tc_act(accv[j], p.act);
                }
            }
            if (valid) {
                float* dst = partial ? p.ws + ((long long)split * p.M + m) * p.Cout + n0 : p.y + m * p.ocs + p.oco + n0;
                if (vec_ok && n0 + 16 <= p.Cout) {
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4)
                        reinterpret_cast<float4*>(dst)[j4] = make_float4(accv[j4 * 4], accv[j4 * 4 + 1], accv[j4 * 4 + 2], accv[j4 * 4 + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (n0 + j < p.Cout) dst[j] = accv[j];
                }
            }
            if (p.stats && !partial)      // tiles never span planes and a group is made of whole planes
                epilogue_stats(accv, valid, p.stats, (((long long)b * p.Do + zo) * p.Ho * p.Wo) / p.stats_rows, p.Cout, n0, lane);
        }
        tc_fence_before();
    } else if (warp == TC_PRODUCER_WARPS) {
        // =============================== B producer (TMA) ===============================
        if (lane == 0) {
            int bi = 0;
            for (int u = 0; u < nunits; ++u) {
                const int cb = cb_begin + u / p.nseg, seg = u % p.nseg;
                for (int t = 0; t < p.taps_per_seg; ++t, ++bi) {
                    const int s = bi % p.b_stages;
                    const uint32_t n_use = bi / p.b_stages;
                    mbar_wait(b_empty(s), (n_use & 1) ^ 1, 3, bi);
                    mbar_expect_tx(b_full(s), 2 * B_BYTES);
                    const int k = (seg * p.taps_per_seg + t) * p.Cin + cb * BK;
                    tma_load_2d(b_hi(s), &map_hi, b_full(s), k, n_base);
                    tma_load_2d(b_lo(s), &map_lo, b_full(s), k, n_base);
                }
            }
        }
    } else {
        // =============================== MMA issuer ===============================
        if (elect_one_sync()) {
            const uint32_t idesc = umma_idesc<KIND>(TC_BM, BN);
            int bi = 0;
            for (int u = 0; u < nunits; ++u) {
                const int sa = u % p.a_stages;
                mbar_wait(a_full(sa), (u / p.a_stages) & 1, 4, u);
                tc_fence_after();
                for (int t = 0; t < p.taps_per_seg; ++t, ++bi) {
                    const int sb = bi % p.b_stages;
                    mbar_wait(b_full(sb), (bi / p.b_stages) & 1, 5, bi);
                    tc_fence_after();
                    const int shift = p.mode == 1 ? t : (t / p.kw) * p.Wp + (t % p.kw);     // rows
                    const uint64_t dah = umma_desc_sw128(a_hi(sa) + shift * 128), dal = umma_desc_sw128(a_lo(sa) + shift * 128);
                    const uint64_t dbh = umma_desc_sw128(b_hi(sb)), dbl = umma_desc_sw128(b_lo(sb));
                    const uint32_t main_acc = tmem_acc + (uint32_t)((bi % NMAIN) * BN);
                    const uint32_t cross_acc = tmem_acc + (uint32_t)(NMAIN * BN);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t adv = (uint64_t)((ks * 32) >> 4);
                        umma<KIND>(cross_acc, dal + adv, dbh + adv, idesc, (bi > 0 || ks > 0) ? 1u : 0u);
                        umma<KIND>(cross_acc, dah + adv, dbl + adv, idesc, 1u);
                        umma<KIND>(main_acc, dah + adv, dbh + adv, idesc, (bi >= NMAIN || ks > 0) ? 1u : 0u);
                    }
                    umma_commit(b_empty(sb));
                }
                umma_commit(a_empty(sa));
            }
            umma_commit(tmem_full);
        }
    }
    __syncthreads();
    if (warp == TC_PRODUCER_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "n"(TMEM_COLS) : "memory");
    }
}

// G6D_CONV_FLAT: 0 = never use the A-reuse kernel, 1 = FLAT mode only (default), 2 = FLAT and ROW.
// Measured on B200 (tools/conv_breakdown.py): the MMAs are shared-memory-bandwidth bound
// (every MMA re-reads 4 KB of A and N*32 B of B; at N = 128 that alone is 128 B/clk/SM), so the
// 3x-reuse ROW mode does not pay for its junk columns, while FLAT (9x reuse, and the prologue
// applied once per element instead of once per tap) gains 26 % on the selector's first tower conv.
static int flat_level() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("G6D_CONV_FLAT"); v = (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1; }
    return v;
}
static bool flat_disabled() { return flat_level() == 0; }

static int fill_flat_params(const g6d_conv_desc* d, int kind, ConvFlatP& p, int* smem_bytes) {
    const int bk = kind_bk(kind);
    if (!d || !in_items_ok(d) || d->stride != 1 || (d->Cin % bk) != 0 || d->Cout < 16 || (d->in_cstride & 3) || (d->in_coff & 3)) return -1;
    const int Do = d->D + 2 * d->pd - d->kd + 1, Ho = d->H + 2 * d->ph - d->kh + 1, Wo = d->W + 2 * d->pw - d->kw + 1;
    if (Do != d->Do || Ho != d->Ho || Wo != d->Wo || Do < 1 || Ho < 1 || Wo < 1) return -1;
    if (d->kd * d->kh * d->kw == 1) return -1;                        // 1x1: nothing to reuse, persistent kernel
    const int bn = tc_block_n(d->Cout);
    const int Wp = d->W + 2 * d->pw;
    const int flat_rows = TC_BM + (d->kh - 1) * Wp + d->kw - 1;
    const int row_rows = TC_BM + d->kw - 1;
    const int budget = 220 * 1024;
    const int b_stage = 2 * bn * 128;
    // tiles never span image planes: small planes (selector 4x4 / 8x8 maps) would leave most of a
    // 128-row tile empty -> keep those on the batch-flattened kernel
    {
        const long long tiles = ((long long)Ho * Wp + TC_BM - 1) / TC_BM;
        if ((long long)Ho * Wo * 100 < tiles * TC_BM * 60) return -1;
    }
    auto a_stage = [](int rows) { return 2 * ((rows + 7) / 8 * 8) * 128; };
    int mode, rows, ntab;
    // FLAT when two A stages of the full halo + >= 3 B stages fit
    if (2 * a_stage(flat_rows) + 3 * b_stage + 4 * flat_rows + 2048 <= budget) { mode = 0; rows = flat_rows; ntab = 1; }
    else if (d->kw > 1 && flat_level() >= 2) { mode = 1; rows = row_rows; ntab = d->kh; }
    else return -1;
    p.B = d->B; p.D = d->D; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.ics = d->in_cstride; p.ico = d->in_coff;
    p.Cout = d->Cout; p.kd = d->kd; p.kh = d->kh; p.kw = d->kw; p.pd = d->pd; p.ph = d->ph; p.pw = d->pw;
    p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.ocs = d->out_cstride; p.oco = d->out_coff; p.pro = d->prologue; p.act = d->act;
    p.group_rows = d->group_rows > 0 ? d->group_rows : 1;
    p.in_items = d->in_items > 0 ? d->in_items : d->B;
    p.Wp = Wp; p.tiles_per_plane = (Ho * Wp + TC_BM - 1) / TC_BM; p.mode = mode;
    p.nseg = mode == 0 ? d->kd : d->kd * d->kh; p.taps_per_seg = mode == 0 ? d->kh * d->kw : d->kw;
    p.seg_rows = rows; p.rows_pad = (rows + 7) / 8 * 8; p.ntab = ntab; p.cblocks = d->Cin / bk;
    const long long M = (long long)d->B * Do * Ho * Wo;
    if (M >= (1ll << 31)) return -1;
    p.M = (int)M;
    const int tab_bytes = 4 * ntab * rows;
    int a_st = 2, b_st = 3;
    int used = a_st * a_stage(rows) + b_st * b_stage + tab_bytes + 2048;
    while (b_st < 4 && used + b_stage <= budget) { ++b_st; used += b_stage; }
    while (a_st < 4 && used + a_stage(rows) <= budget) { ++a_st; used += a_stage(rows); }
    if (used > budget) return -1;
    p.a_stages = a_st; p.b_stages = b_st;
    *smem_bytes = a_st * a_stage(rows) + b_st * b_stage + 256 + tab_bytes + 1024 + 64;
    // split over channel blocks when the tile grid cannot fill the machine, or to bound accumulate chains
    const long long ctas = (long long)d->B * Do * p.tiles_per_plane * ((d->Cout + bn - 1) / bn);
    const long long K = (long long)d->Cin * d->kd * d->kh * d->kw;
    int splits = 1;
    if (ctas < kNumSMs && p.cblocks >= 2) splits = (int)((kNumSMs + ctas - 1) / ctas);
    const int nmain = bn == 32 ? FlatCfg<32>::NMAIN : (bn == 64 ? FlatCfg<64>::NMAIN : FlatCfg<128>::NMAIN);
    const long long chain = d->max_chain_k > 0 ? (long long)d->max_chain_k * nmain : (K > 8192 ? TC_MAX_K_PER_CHAIN : 0);
    if (chain > 0) { const int ms = (int)((K + chain - 1) / chain); splits = splits < ms ? ms : splits; }
    splits = splits > p.cblocks ? p.cblocks : splits;
    splits = splits < 1 ? 1 : splits;
    p.cb_per_split = (p.cblocks + splits - 1) / splits;
    p.splits = (p.cblocks + p.cb_per_split - 1) / p.cb_per_split;
    return 0;
}

template <int BN, int KIND>
static int launch_flat(const ConvFlatP& p, int smem, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(conv_tcflat_kernel<BN, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("g6d_conv_tc(flat): cannot opt in to shared memory: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
        configured = true;
    }
    dim3 grid((unsigned)((long long)p.B * p.Do * p.tiles_per_plane), ceil_div(p.Cout, BN), p.splits);
    conv_tcflat_kernel<BN, KIND><<<grid, TC_THREADS, smem, st>>>(p, mh, ml);
    G6D_CHECK_LAUNCH("g6d_conv_tc(flat)");
    return G6D_OK;
}

template <int KIND>
static int dispatch_flat(int bn, const ConvFlatP& p, int smem, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
    if (bn == 128) return launch_flat<128, KIND>(p, smem, mh, ml, st);
    if (bn == 64) return launch_flat<64, KIND>(p, smem, mh, ml, st);
    return launch_flat<32, KIND>(p, smem, mh, ml, st);
}
template <int KIND>
static int dispatch_tc2(int bn, const ConvTcP& p, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
    if (bn == 128) return launch_tc2<128, KIND>(p, mh, ml, st);
    if (bn == 64) return launch_tc2<64, KIND>(p, mh, ml, st);
    return launch_tc2<32, KIND>(p, mh, ml, st);
}

}  // namespace g6d

using namespace g6d;

// Debug aid: copies the 8-int timeout record (0 = no timeout; else [1]=waiter role 1 A-producer/empty,
// 2 epilogue/tmem_full, 3 B-producer/empty, 4 MMA/full_a, 5 MMA/full_b, 6 MMA/tmem_empty; [2]=iteration;
// [3]=parity; [4..6]=block; [7]=thread) and clears it.  Synchronises the device.
extern "C" int g6d_conv_tc_debug(int* host_out8) {
    G6D_REQUIRE(host_out8 != nullptr, "g6d_conv_tc_debug: null");
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error("g6d_conv_tc_debug: sync: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
    e = cudaMemcpyFromSymbol(host_out8, g_tc_timeout, sizeof(int) * 8);
    if (e != cudaSuccess) { set_error("g6d_conv_tc_debug: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
    int zeros[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    cudaMemcpyToSymbol(g_tc_timeout, zeros, sizeof(zeros));
    return G6D_OK;
}

extern "C" int g6d_conv_tc_supported(const g6d_conv_desc* d, int kind) {
    if (!d || (kind != G6D_TC_TF32 && kind != G6D_TC_F16)) return 0;
    return in_items_ok(d) && pro_operands_fit(d) && (d->Cin % kind_bk(kind)) == 0 && d->Cout >= 16 && (d->in_cstride & 3) == 0 && (d->in_coff & 3) == 0 &&
           tc2_dims_ok(d) ? 1 : 0;
}

extern "C" long long g6d_conv_tc_workspace_bytes(const g6d_conv_desc* desc, int kind) {
    {
        ConvFlatP fp{}; int smem = 0;
        if (!flat_disabled() && (kind == G6D_TC_TF32 || kind == G6D_TC_F16) && fill_flat_params(desc, kind, fp, &smem) == 0)
            return fp.splits > 1 ? (long long)fp.splits * fp.M * fp.Cout * (long long)sizeof(float) : 0;
    }
    ConvTcP p{};
    if (fill_tc_params(desc, kind, p) != G6D_OK) return -1;
    return p.splits > 1 ? (long long)p.splits * p.M * p.Cout * (long long)sizeof(float) : 0;
}

// fused output statistics are possible when every 32-row epilogue slice lies in one group
static bool stats_ok_tc2(long long stats_rows, long long M) { return stats_rows > 0 && stats_rows % 32 == 0 && M % stats_rows == 0; }
static bool stats_ok_flat(const ConvFlatP& fp, long long stats_rows) {
    return stats_rows > 0 && stats_rows % 32 == 0 && stats_rows % ((long long)fp.Ho * fp.Wo) == 0 && (long long)fp.M % stats_rows == 0;
}

extern "C" int g6d_conv_tc_stats_supported(const g6d_conv_desc* desc, int kind, long long stats_rows) {
    if (!g6d_conv_tc_supported(desc, kind)) return 0;
    ConvFlatP fp{}; int smem = 0;
    if (!flat_disabled() && fill_flat_params(desc, kind, fp, &smem) == 0) return stats_ok_flat(fp, stats_rows) ? 1 : 0;
    const long long M = (long long)desc->B * desc->Do * desc->Ho * desc->Wo;
    return stats_ok_tc2(stats_rows, M) ? 1 : 0;
}

extern "C" int g6d_conv_tc(const g6d_conv_desc* desc, const float* x, const void* w_hi, const void* w_lo, int w_rows,
                           int kind, const float* bias, const float* pro_scale, const float* pro_shift, float* y,
                           void* ws, double* stats, long long stats_rows, g6d_stream_t stream) {
    G6D_REQUIRE(kind == G6D_TC_TF32 || kind == G6D_TC_F16, "g6d_conv_tc: bad operand kind %d", kind);
    if (stats) {
        G6D_REQUIRE(g6d_conv_tc_stats_supported(desc, kind, stats_rows), "g6d_conv_tc: fused statistics need groups of whole 32-row slices / planes (stats_rows %lld)", stats_rows);
        const long long M = (long long)desc->B * desc->Do * desc->Ho * desc->Wo;
        cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(double) * 2 * (M / stats_rows) * desc->Cout, as_stream(stream));
        if (e != cudaSuccess) { set_error("g6d_conv_tc: memset: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
    }
    {   // stride-1 multi-tap convolutions: A-reuse kernel
        ConvFlatP fp{}; int smem = 0;
        if (!flat_disabled() && fill_flat_params(desc, kind, fp, &smem) == 0) {
            G6D_REQUIRE(x && w_hi && w_lo && y, "g6d_conv_tc: null tensor pointer");
            G6D_REQUIRE(w_rows >= fp.Cout, "g6d_conv_tc: weight rows (%d) < Cout (%d)", w_rows, fp.Cout);
            if (fp.pro != G6D_PRO_NONE) G6D_REQUIRE(pro_scale && pro_shift, "g6d_conv_tc: prologue operands missing");
            if (fp.splits > 1) G6D_REQUIRE(ws != nullptr, "g6d_conv_tc: split workspace required (%d splits)", fp.splits);
            fp.x = x; fp.bias = bias; fp.ps = pro_scale; fp.pb = pro_shift; fp.y = y; fp.ws = (float*)ws;
            fp.stats = stats; fp.stats_rows = stats ? stats_rows : 1;
            const int bn = tc_block_n(fp.Cout);
            const int K = fp.kd * fp.kh * fp.kw * fp.Cin;
            CUtensorMap mh, ml;
            int rc2;
            if ((rc2 = make_weight_map(&mh, w_hi, w_rows, K, bn, kind)) != G6D_OK) return rc2;
            if ((rc2 = make_weight_map(&ml, w_lo, w_rows, K, bn, kind)) != G6D_OK) return rc2;
            cudaStream_t st = as_stream(stream);
            rc2 = kind == G6D_TC_F16 ? dispatch_flat<G6D_TC_F16>(bn, fp, smem, mh, ml, st)
                                     : dispatch_flat<G6D_TC_TF32>(bn, fp, smem, mh, ml, st);
            if (rc2 != G6D_OK) return rc2;
            if (fp.splits > 1) {
                const long long n = (long long)fp.M * fp.Cout;
                (void)n;
                launch_reduce(fp.ws, bias, y, fp.M, fp.Cout, fp.splits, fp.ocs, fp.oco, fp.act, fp.stats, fp.stats_rows, st);
                G6D_CHECK_LAUNCH("g6d_conv_tc(flat reduce)");
            }
            return G6D_OK;
        }
    }
    ConvTcP p{};
    int rc = fill_tc_params(desc, kind, p);
    if (rc != G6D_OK) return rc;
    G6D_REQUIRE(x && w_hi && w_lo && y, "g6d_conv_tc: null tensor pointer");
    G6D_REQUIRE(w_rows >= p.Cout, "g6d_conv_tc: weight rows (%d) < Cout (%d)", w_rows, p.Cout);
    if (p.pro != G6D_PRO_NONE) G6D_REQUIRE(pro_scale && pro_shift, "g6d_conv_tc: prologue operands missing");
    if (p.splits > 1) G6D_REQUIRE(ws != nullptr, "g6d_conv_tc: split-K workspace required (%d splits)", p.splits);
    p.x = x; p.bias = bias; p.ps = pro_scale; p.pb = pro_shift; p.y = y; p.ws = (float*)ws;
    p.stats = stats; p.stats_rows = stats ? stats_rows : 1;
    const int bn = tc_block_n(p.Cout);
    CUtensorMap mh, ml;
    if ((rc = make_weight_map(&mh, w_hi, w_rows, p.K, bn, kind)) != G6D_OK) return rc;
    if ((rc = make_weight_map(&ml, w_lo, w_rows, p.K, bn, kind)) != G6D_OK) return rc;
    cudaStream_t st = as_stream(stream);
    rc = kind == G6D_TC_F16 ? dispatch_tc2<G6D_TC_F16>(bn, p, mh, ml, st) : dispatch_tc2<G6D_TC_TF32>(bn, p, mh, ml, st);
    if (rc != G6D_OK) return rc;
    if (p.splits > 1) {
        const long long n = (long long)p.M * p.Cout;
        (void)n;
        launch_reduce(p.ws, bias, y, p.M, p.Cout, p.splits, p.ocs, p.oco, p.act, p.stats, p.stats_rows, st);
        G6D_CHECK_LAUNCH("g6d_conv_tc(splitk reduce)");
    }
    return G6D_OK;
}

extern "C" int g6d_split_operand(const float* in, void* hi, void* lo, long long n, int kind, g6d_stream_t stream) {
    G6D_REQUIRE(in && hi && lo && n > 0, "g6d_split_operand: bad args");
    G6D_REQUIRE(kind == G6D_TC_TF32 || kind == G6D_TC_F16, "g6d_split_operand: bad operand kind %d", kind);
    G6D_REQUIRE(kind != G6D_TC_F16 || (n & 63) == 0, "g6d_split_operand: fp16 operands are laid out in 64-element K-blocks (n = %lld)", n);
    if (kind == G6D_TC_F16)
        split_f16_kernel<<<ceil_div(n, 256), 256, 0, as_stream(stream)>>>(in, static_cast<__half*>(hi), static_cast<__half*>(lo), n);
    else
        split_tf32_kernel<<<ceil_div(n, 256), 256, 0, as_stream(stream)>>>(in, static_cast<float*>(hi), static_cast<float*>(lo), n);
    G6D_CHECK_LAUNCH("g6d_split_operand");
    return G6D_OK;
}

extern "C" int g6d_pack_conv_weight_tc(const float* w, void* out_hi, void* out_lo, int Cout, int Cin, int Cin_pad,
                                       int taps, int rows_pad, const float* cout_scale, int kind, g6d_stream_t stream) {
    G6D_REQUIRE(w && out_hi && out_lo && Cout > 0 && Cin > 0 && Cin_pad >= Cin && taps > 0 && rows_pad >= Cout,
                "g6d_pack_conv_weight_tc: bad args");
    G6D_REQUIRE(kind == G6D_TC_TF32 || kind == G6D_TC_F16, "g6d_pack_conv_weight_tc: bad operand kind %d", kind);
    const long long total = (long long)taps * Cin_pad * rows_pad;
    if (kind == G6D_TC_F16)
        pack_conv_weight_tc_kernel<G6D_TC_F16><<<ceil_div(total, 256), 256, 0, as_stream(stream)>>>(w, out_hi, out_lo, Cout, Cin,
                                                                                                    Cin_pad, taps, rows_pad, cout_scale);
    else
        pack_conv_weight_tc_kernel<G6D_TC_TF32><<<ceil_div(total, 256), 256, 0, as_stream(stream)>>>(w, out_hi, out_lo, Cout, Cin,
                                                                                                     Cin_pad, taps, rows_pad, cout_scale);
    G6D_CHECK_LAUNCH("g6d_pack_conv_weight_tc");
    return G6D_OK;
}

// ------------------------------------------------------------------------------------------
// Probe (debug/test only): does a K-major SWIZZLE_128B A operand tolerate a start address that is
// shifted by `shift` rows (shift*128 B, not 1024-aligned) when the data was written with the
// swizzle phase of its ABSOLUTE shared-memory row?  D[128 x 32] = A[shift .. shift+128) x B^T with
// K = 32, A[r][k] = r + k/64 (exactly representable), B = 32x32 identity.  `mode` selects how the
// descriptor's base_offset field is set: 0 -> 0, 1 -> (start_address >> 7) & 7.
namespace g6d {
__global__ void __launch_bounds__(128) umma_shift_probe_kernel(float* out, int shift, int mode) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* bp = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t a_base = base;                 // 160 rows x 128 B
    const uint32_t b_base = base + 160 * 128;     // 32 rows x 128 B (20480 is 1024-aligned)
    const uint32_t bar = b_base + 32 * 128;
    volatile uint32_t* slot = reinterpret_cast<volatile uint32_t*>(bp + 160 * 128 + 32 * 128 + 16);
    const int t = threadIdx.x;
    for (int r = t; r < 160; r += 128)
        for (int c = 0; c < 8; ++c) {
            float4 v = make_float4(r + (c * 4 + 0) / 64.f, r + (c * 4 + 1) / 64.f, r + (c * 4 + 2) / 64.f, r + (c * 4 + 3) / 64.f);
            *reinterpret_cast<float4*>(bp + r * 128 + ((c ^ (r & 7)) << 4)) = v;
        }
    for (int r = t; r < 32; r += 128)
        for (int c = 0; c < 8; ++c) {
            float4 v = make_float4(r == c * 4 ? 1.f : 0.f, r == c * 4 + 1 ? 1.f : 0.f, r == c * 4 + 2 ? 1.f : 0.f, r == c * 4 + 3 ? 1.f : 0.f);
            *reinterpret_cast<float4*>(bp + 160 * 128 + r * 128 + ((c ^ (r & 7)) << 4)) = v;
        }
    fence_proxy_async();
    if (t == 0) { mbar_init(bar, 1); fence_barrier_init(); }
    if (t < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 32;" ::"r"(smem_u32((const void*)slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot;
    if (t == 0) {
        const uint32_t start = a_base + shift * 128;
        uint64_t da = umma_desc_sw128(start);
        if (mode == 1) da |= (uint64_t)((start >> 7) & 7) << 49;
        const uint64_t db = umma_desc_sw128(b_base);
        const uint32_t idesc = umma_idesc<G6D_TC_TF32>(128, 32);
        for (int ks = 0; ks < 4; ++ks) umma<G6D_TC_TF32>(tmem, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc, ks > 0);
        umma_commit(bar);
    }
    mbar_wait(bar, 0, 9, 0);
    tc_fence_after();
    const int warp = t >> 5, lane = t & 31;
    for (int cc = 0; cc < 32; cc += 16) {
        uint32_t r[16];
        G6D_TMEM_LD16(r, tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)cc);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        for (int j = 0; j < 16; ++j) out[(warp * 32 + lane) * 32 + cc + j] = __uint_as_float(r[j]);
    }
    tc_fence_before();
    __syncthreads();
    if (t < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 32;" ::"r"(tmem) : "memory");
}
}  // namespace g6d

extern "C" int g6d_debug_umma_shift(float* out, int shift, int mode, g6d_stream_t stream) {
    G6D_REQUIRE(out && shift >= 0 && shift <= 31, "g6d_debug_umma_shift: bad args");
    g6d::umma_shift_probe_kernel<<<1, 128, 160 * 128 + 32 * 128 + 1024 + 64, g6d::as_stream(stream)>>>(out, shift, mode);
    G6D_CHECK_LAUNCH("g6d_debug_umma_shift");
    return G6D_OK;
}
