// Implicit-GEMM convolution, fp32 FFMA path (exact-fp32 parity mode).
//
// GEMM view: M = B*Do*Ho*Wo output positions, N = Cout, K = taps*Cin with channels-last
// activations, so every K-run of Cin elements is one contiguous channel vector of one input
// position.  CTA tile 128 x BN x 16, 256 threads, 8 x TN register tile, double-buffered shared
// memory with register prefetch.  The A-operand loader applies the folded InstanceNorm(+ReLU)
// or the selector's q (.) ref product to in-bounds elements only (zero padding stays zero, as in
// the reference where padding follows the norm: selector.py:27-69 / SURVEY.md A10).
//
// Small-M / huge-K layers (detector correlation with 15x15x512 kernels, refiner 4^3 layers)
// are split along K across blockIdx.z into a workspace and reduced deterministically.
#include "common.cuh"

namespace g6d {

struct ConvP {
    const float* x; const float* w; const float* bias; const float* ps; const float* pb;
    float* y; float* ws;
    int B, D, H, W, Cin, ics, ico, Cout, ldw, kd, kh, kw, stride, pd, ph, pw, Do, Ho, Wo, ocs, oco, pro, act;
    long long group_rows;
    int in_items;             // input items: output item b reads input item b % in_items
    int M, K, ktiles, splits, kt_per_split;
};

constexpr int BM = 128, BK = 16, NT = 256;

__device__ __forceinline__ float act_apply(float v, int act) {
    if (act == G6D_ACT_RELU) return fmaxf(v, 0.f);
    if (act == G6D_ACT_LEAKY01) return v > 0.f ? v : 0.1f * v;
    return v;
}

template <int TN>
__global__ void __launch_bounds__(NT, 2) conv_ffma_kernel(const ConvP p) {
    constexpr int BN = 16 * TN;
    constexpr int HN = BN / 2;                 // second column group offset (TN == 8 only)
    constexpr int B_F4 = (BK * BN / 4);        // float4 per B tile
    constexpr int B_PER_T = (B_F4 + NT - 1) / NT;
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Bs[2][BK][BN];

    const int t = threadIdx.x;
    const int tx = t & 15, ty = t >> 4;
    const int m_base = blockIdx.x * BM;
    const int n_base = blockIdx.y * BN;
    const int split = blockIdx.z;
    const int kt_begin = split * p.kt_per_split;
    const int kt_end = min(p.ktiles, kt_begin + p.kt_per_split);

    // ---- A loader state: 2 rows per thread, one float4 (4 consecutive k) each
    const int kq = t & 3;
    // rb: the input item a row reads; rg: the prologue group of its output item (once per tile, no divide in the K loop)
    int rb[2], rg[2], rz[2], ry[2], rx[2];
    bool rvalid[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        int m = m_base + (t >> 2) + 64 * i;
        rvalid[i] = m < p.M;
        int mm = rvalid[i] ? m : 0;
        int xo = mm % p.Wo; mm /= p.Wo;
        int yo = mm % p.Ho; mm /= p.Ho;
        int zo = mm % p.Do; mm /= p.Do;
        rb[i] = p.in_items == p.B ? mm : mm % p.in_items;
        rg[i] = p.pro == G6D_PRO_NONE ? 0 : (int)(mm / p.group_rows);
        rz[i] = zo * p.stride - p.pd;
        ry[i] = yo * p.stride - p.ph;
        rx[i] = xo * p.stride - p.pw;
    }

    float4 a_reg[2];
    float4 b_reg[B_PER_T];

    auto load_tile = [&](int kt) {
        const int k = kt * BK + kq * 4;
        const bool kvalid = k < p.K;
        int tap = 0, c = k;
        if (p.K != p.Cin) { tap = k / p.Cin; c = k - tap * p.Cin; }
        const int kx = tap % p.kw;
        const int tq = tap / p.kw;
        const int ky = tq % p.kh;
        const int kz = tq / p.kh;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int zi = rz[i] + kz, yi = ry[i] + ky, xi = rx[i] + kx;
            const bool inb = rvalid[i] && kvalid && (unsigned)zi < (unsigned)p.D && (unsigned)yi < (unsigned)p.H &&
                             (unsigned)xi < (unsigned)p.W;
            if (inb) {
                const long long pos = ((long long)(rb[i] * p.D + zi) * p.H + yi) * p.W + xi;
                v = __ldg(reinterpret_cast<const float4*>(p.x + pos * p.ics + p.ico + c));
                if (p.pro != G6D_PRO_NONE) {
                    float4 s, b;
                    const int gc = rg[i] * p.Cin + c;                   // 32-bit (host checks the range)
                    if (p.pro == G6D_PRO_CORR) {
                        s = __ldg(reinterpret_cast<const float4*>(p.ps + (((rg[i] * p.D + zi) * p.H + yi) * p.W + xi) * p.Cin + c));
                        b = __ldg(reinterpret_cast<const float4*>(p.pb + gc));
                    } else {
                        s = __ldg(reinterpret_cast<const float4*>(p.ps + gc));
                        b = __ldg(reinterpret_cast<const float4*>(p.pb + gc));
                    }
                    v.x = fmaf(v.x, s.x, b.x); v.y = fmaf(v.y, s.y, b.y);
                    v.z = fmaf(v.z, s.z, b.z); v.w = fmaf(v.w, s.w, b.w);
                    if (p.pro == G6D_PRO_AFFINE_RELU) {
                        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                    }
                }
            }
            a_reg[i] = v;
        }
#pragma unroll
        for (int j = 0; j < B_PER_T; ++j) {
            const int f = t + j * NT;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (f < B_F4) {
                const int kr = f / (BN / 4), nq = f % (BN / 4);
                const int kk = kt * BK + kr, n = n_base + nq * 4;
                if (kk < p.K && n < p.ldw) v = __ldg(reinterpret_cast<const float4*>(p.w + (long long)kk * p.ldw + n));
            }
            b_reg[j] = v;
        }
    };
    auto store_tile = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int r = (t >> 2) + 64 * i;
            As[buf][kq * 4 + 0][r] = a_reg[i].x;
            As[buf][kq * 4 + 1][r] = a_reg[i].y;
            As[buf][kq * 4 + 2][r] = a_reg[i].z;
            As[buf][kq * 4 + 3][r] = a_reg[i].w;
        }
#pragma unroll
        for (int j = 0; j < B_PER_T; ++j) {
            const int f = t + j * NT;
            if (f < B_F4) {
                const int kr = f / (BN / 4), nq = f % (BN / 4);
                *reinterpret_cast<float4*>(&Bs[buf][kr][nq * 4]) = b_reg[j];
            }
        }
    };

    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    if (kt_begin < kt_end) {
        load_tile(kt_begin);
        store_tile(0);
    }
    __syncthreads();
    int cur = 0;
    for (int kt = kt_begin; kt < kt_end; ++kt) {
        const bool more = kt + 1 < kt_end;
        if (more) load_tile(kt + 1);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[8], b[TN];
            *reinterpret_cast<float4*>(&a[0]) = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
            *reinterpret_cast<float4*>(&a[4]) = *reinterpret_cast<const float4*>(&As[cur][k][64 + ty * 4]);
            if constexpr (TN == 8) {
                *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
                *reinterpret_cast<float4*>(&b[TN - 4]) = *reinterpret_cast<const float4*>(&Bs[cur][k][HN + tx * 4]);
            } else if constexpr (TN == 4) {
                *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
            } else {
                *reinterpret_cast<float2*>(&b[0]) = *reinterpret_cast<const float2*>(&Bs[cur][k][tx * 2]);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (more) store_tile(cur ^ 1);
        __syncthreads();
        cur ^= 1;
    }

    // ---- epilogue
    const bool partial = p.splits > 1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m_base + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= p.M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int n;
            if constexpr (TN == 8) n = n_base + (j < 4 ? tx * 4 + j : HN + tx * 4 + (j - 4));
            else if constexpr (TN == 4) n = n_base + tx * 4 + j;
            else n = n_base + tx * 2 + j;
            if (n >= p.Cout) continue;
            float v = acc[i][j];
            if (partial) {
                p.ws[((long long)split * p.M + m) * p.Cout + n] = v;
            } else {
                if (p.bias) v += __ldg(p.bias + n);
                p.y[(long long)m * p.ocs + p.oco + n] = act_apply(v, p.act);
            }
        }
    }
}

__global__ void conv_splitk_reduce_kernel(const float* __restrict__ ws, const float* __restrict__ bias,
                                          float* __restrict__ y, int M, int Cout, int splits, int ocs, int oco,
                                          int act) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * Cout) return;
    const int n = (int)(i % Cout);
    const long long m = i / Cout;
    float v = 0.f;
    for (int s = 0; s < splits; ++s) v += ws[(long long)s * M * Cout + i];
    if (bias) v += bias[n];
    y[m * ocs + oco + n] = act_apply(v, act);
}

// ------------------------------------------------------------------------------------------
// First VGG layer: 3x3, Cin = 4 (RGB + a zero channel), Cout = 64, stride 1, pad 1.
// K = 36 is far too small for the GEMM tiling (the layer is bound by its 64-channel output
// write), so it gets a direct kernel: one thread per output pixel, 64 accumulators in registers,
// the 36 x 64 weights broadcast from shared memory, 128-bit input loads, 16 x 128-bit stores.
__global__ void __launch_bounds__(128) conv3x3_c4_o64_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                             const float* __restrict__ bias, float* __restrict__ y,
                                                             int B, int H, int W, int act) {
    __shared__ __align__(16) float ws[36 * 64];
    __shared__ float bs[64];
    for (int i = threadIdx.x; i < 36 * 64; i += blockDim.x) ws[i] = w[i];
    if (threadIdx.x < 64) bs[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
    __syncthreads();
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long M = (long long)B * H * W;
    if (m >= M) return;
    const int xo = (int)(m % W), yo = (int)((m / W) % H);
    const long long b = m / ((long long)W * H);
    float acc[64];
#pragma unroll
    for (int o = 0; o < 64; ++o) acc[o] = bs[o];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int yi = yo + ky - 1;
        if ((unsigned)yi >= (unsigned)H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int xi = xo + kx - 1;
            if ((unsigned)xi >= (unsigned)W) continue;
            const float4 v = __ldg(reinterpret_cast<const float4*>(x + ((b * H + yi) * W + xi) * 4));
            const float* wr = ws + (ky * 3 + kx) * 4 * 64;
#pragma unroll
            for (int o4 = 0; o4 < 16; ++o4) {
                const float4 w0 = *reinterpret_cast<const float4*>(wr + o4 * 4);
                const float4 w1 = *reinterpret_cast<const float4*>(wr + 64 + o4 * 4);
                const float4 w2 = *reinterpret_cast<const float4*>(wr + 128 + o4 * 4);
                const float4 w3 = *reinterpret_cast<const float4*>(wr + 192 + o4 * 4);   // 4th channel (zero for images)
                acc[o4 * 4 + 0] = fmaf(v.x, w0.x, fmaf(v.y, w1.x, fmaf(v.z, w2.x, fmaf(v.w, w3.x, acc[o4 * 4 + 0]))));
                acc[o4 * 4 + 1] = fmaf(v.x, w0.y, fmaf(v.y, w1.y, fmaf(v.z, w2.y, fmaf(v.w, w3.y, acc[o4 * 4 + 1]))));
                acc[o4 * 4 + 2] = fmaf(v.x, w0.z, fmaf(v.y, w1.z, fmaf(v.z, w2.z, fmaf(v.w, w3.z, acc[o4 * 4 + 2]))));
                acc[o4 * 4 + 3] = fmaf(v.x, w0.w, fmaf(v.y, w1.w, fmaf(v.z, w2.w, fmaf(v.w, w3.w, acc[o4 * 4 + 3]))));
            }
        }
    }
    float4* yr = reinterpret_cast<float4*>(y + m * 64);
#pragma unroll
    for (int o4 = 0; o4 < 16; ++o4) {
        float4 r = make_float4(act_apply(acc[o4 * 4], act), act_apply(acc[o4 * 4 + 1], act), act_apply(acc[o4 * 4 + 2], act),
                               act_apply(acc[o4 * 4 + 3], act));
        __stcs(yr + o4, r);
    }
}

// The same layer FUSED with the ReLU and the 2x2 max-pool that follow it in VGG (pretrain_models.py:
// features[0:4]; nothing on the path reads the full-resolution 64-channel map): a thread owns 16 output
// channels of one POOLED pixel (a quad of lanes = 64 channels = one 256-byte output row), keeps the
// 4x4 input window in registers and applies each tap's weights to the four conv outputs under the pool.
// Writes 1/4 of the bytes and saves the pool's read + write: the unfused pair moves 78.6 + 78.6 + 19.7 MB
// per 480x640 frame, this kernel 4.9 + 19.7 MB.  Accumulation order per output equals the unfused
// kernel's (taps ky-major, channels innermost-first; channel 3 is the zero padding), so the result is
// bit-identical to conv -> ReLU -> maxpool.
__global__ void __launch_bounds__(128) conv3x3_c4_o64_relu_pool_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                                       const float* __restrict__ bias, float* __restrict__ y,
                                                                       int B, int H, int W) {
    __shared__ __align__(16) float ws[36 * 64];
    __shared__ float bs[64];
    for (int i = threadIdx.x; i < 36 * 64; i += blockDim.x) ws[i] = w[i];
    if (threadIdx.x < 64) bs[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
    __syncthreads();
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int q = (int)(t & 3);                       // channels [16 q, 16 q + 16)
    const long long pp = t >> 2;                      // pooled pixel
    const int Hp = H >> 1, Wp = W >> 1;
    if (pp >= (long long)B * Hp * Wp) return;
    const int xp = (int)(pp % Wp), yp = (int)((pp / Wp) % Hp);
    const long long b = pp / ((long long)Wp * Hp);
    // 4x4 input window rows 2yp-1 .. 2yp+2, columns 2xp-1 .. 2xp+2 (zero outside the image)
    float3 win[4][4];
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
        const int yi = 2 * yp - 1 + dy;
#pragma unroll
        for (int dx = 0; dx < 4; ++dx) {
            const int xi = 2 * xp - 1 + dx;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if ((unsigned)yi < (unsigned)H && (unsigned)xi < (unsigned)W)
                v = __ldg(reinterpret_cast<const float4*>(x + ((b * H + yi) * W + xi) * 4));
            win[dy][dx] = make_float3(v.x, v.y, v.z);
        }
    }
    float acc[4][16];
#pragma unroll
    for (int o = 0; o < 16; ++o) { const float bv = bs[q * 16 + o]; acc[0][o] = bv; acc[1][o] = bv; acc[2][o] = bv; acc[3][o] = bv; }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const float* wr = ws + (ky * 3 + kx) * 4 * 64 + q * 16;
#pragma unroll
            for (int o4 = 0; o4 < 4; ++o4) {
                const float4 w0 = *reinterpret_cast<const float4*>(wr + o4 * 4);
                const float4 w1 = *reinterpret_cast<const float4*>(wr + 64 + o4 * 4);
                const float4 w2 = *reinterpret_cast<const float4*>(wr + 128 + o4 * 4);
#pragma unroll
                for (int px = 0; px < 4; ++px) {                       // the four conv outputs under the pool
                    const float3 v = win[(px >> 1) + ky][(px & 1) + kx];
                    float* a = acc[px] + o4 * 4;
                    a[0] = fmaf(v.x, w0.x, fmaf(v.y, w1.x, fmaf(v.z, w2.x, a[0])));
                    a[1] = fmaf(v.x, w0.y, fmaf(v.y, w1.y, fmaf(v.z, w2.y, a[1])));
                    a[2] = fmaf(v.x, w0.z, fmaf(v.y, w1.z, fmaf(v.z, w2.z, a[2])));
                    a[3] = fmaf(v.x, w0.w, fmaf(v.y, w1.w, fmaf(v.z, w2.w, a[3])));
                }
            }
        }
    }
    float4* yr = reinterpret_cast<float4*>(y + pp * 64 + q * 16);
#pragma unroll
    for (int o4 = 0; o4 < 4; ++o4) {
        float r[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int o = o4 * 4 + e;
            r[e] = fmaxf(fmaxf(fmaxf(acc[0][o], acc[1][o]), fmaxf(acc[2][o], acc[3][o])), 0.f);     // max-pool of the ReLUs
        }
        __stcs(yr + o4, make_float4(r[0], r[1], r[2], r[3]));
    }
}

static int fill_params(const g6d_conv_desc* d, ConvP& p) {
    G6D_REQUIRE(d != nullptr, "g6d_conv: null desc");
    G6D_REQUIRE(d->B > 0 && d->D > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0, "g6d_conv: bad dims");
    G6D_REQUIRE(d->kd > 0 && d->kh > 0 && d->kw > 0 && d->stride > 0, "g6d_conv: bad kernel/stride");
    G6D_REQUIRE((d->Cin & 3) == 0 && (d->in_cstride & 3) == 0 && (d->in_coff & 3) == 0,
                "g6d_conv: Cin (%d), in_cstride (%d), in_coff (%d) must be multiples of 4", d->Cin, d->in_cstride,
                d->in_coff);
    G6D_REQUIRE(d->in_coff + d->Cin <= d->in_cstride, "g6d_conv: input channel slice out of row");
    G6D_REQUIRE(in_items_ok(d), "g6d_conv: in_items (%d) must be 0 or divide B (%d)", d->in_items, d->B);
    G6D_REQUIRE(pro_operands_fit(d), "g6d_conv: prologue operands too large");
    G6D_REQUIRE(d->out_coff + d->Cout <= d->out_cstride, "g6d_conv: output channel slice out of row");
    const int Do = (d->D + 2 * d->pd - d->kd) / d->stride + 1;
    const int Ho = (d->H + 2 * d->ph - d->kh) / d->stride + 1;
    const int Wo = (d->W + 2 * d->pw - d->kw) / d->stride + 1;
    G6D_REQUIRE(Do == d->Do && Ho == d->Ho && Wo == d->Wo, "g6d_conv: output dims mismatch (%d,%d,%d) vs (%d,%d,%d)",
                d->Do, d->Ho, d->Wo, Do, Ho, Wo);
    G6D_REQUIRE(d->prologue >= 0 && d->prologue <= 3 && d->act >= 0 && d->act <= 2, "g6d_conv: bad prologue/act");
    if (d->prologue == G6D_PRO_AFFINE || d->prologue == G6D_PRO_AFFINE_RELU)
        G6D_REQUIRE(d->group_rows > 0, "g6d_conv: group_rows must be > 0 for affine prologue");
    const long long M = (long long)d->B * Do * Ho * Wo;
    const long long K = (long long)d->kd * d->kh * d->kw * d->Cin;
    G6D_REQUIRE(M < (1ll << 31) && K < (1ll << 31), "g6d_conv: problem too large");
    p.B = d->B; p.D = d->D; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.ics = d->in_cstride; p.ico = d->in_coff;
    p.Cout = d->Cout; p.ldw = (d->Cout + 3) & ~3; p.kd = d->kd; p.kh = d->kh; p.kw = d->kw; p.stride = d->stride;
    p.pd = d->pd; p.ph = d->ph; p.pw = d->pw; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.ocs = d->out_cstride;
    p.oco = d->out_coff; p.pro = d->prologue; p.act = d->act; p.group_rows = d->group_rows > 0 ? d->group_rows : 1;
    p.in_items = d->in_items > 0 ? d->in_items : d->B;
    p.M = (int)M; p.K = (int)K; p.ktiles = (int)((K + BK - 1) / BK);
    // split-K heuristic: fill ~2 CTAs per SM when the MN grid alone cannot
    const int bn = d->Cout > 64 ? 128 : (d->Cout > 32 ? 64 : 32);
    const long long ctas = (long long)ceil_div(M, BM) * ceil_div(d->Cout, bn);
    int splits = 1;
    if (ctas < kNumSMs && p.ktiles >= 16) {
        splits = (int)((2 * kNumSMs + ctas - 1) / ctas);
        splits = splits > p.ktiles / 8 ? p.ktiles / 8 : splits;
        splits = splits > 64 ? 64 : splits;
        splits = splits < 1 ? 1 : splits;
    }
    p.kt_per_split = (p.ktiles + splits - 1) / splits;
    p.splits = (p.ktiles + p.kt_per_split - 1) / p.kt_per_split;
    return G6D_OK;
}

}  // namespace g6d

using namespace g6d;

extern "C" long long g6d_conv_workspace_bytes(const g6d_conv_desc* desc) {
    ConvP p{};
    if (fill_params(desc, p) != G6D_OK) return -1;
    return p.splits > 1 ? (long long)p.splits * p.M * p.Cout * (long long)sizeof(float) : 0;
}

extern "C" int g6d_conv(const g6d_conv_desc* desc, const float* x, const float* w, const float* bias,
                        const float* pro_scale, const float* pro_shift, float* y, void* ws, g6d_stream_t stream) {
    ConvP p{};
    int rc = fill_params(desc, p);
    if (rc != G6D_OK) return rc;
    G6D_REQUIRE(x && w && y, "g6d_conv: null tensor pointer");
    if (p.pro != G6D_PRO_NONE) G6D_REQUIRE(pro_scale && pro_shift, "g6d_conv: prologue operands missing");
    if (p.splits > 1) G6D_REQUIRE(ws != nullptr, "g6d_conv: split-K workspace required (%d splits)", p.splits);
    p.x = x; p.w = w; p.bias = bias; p.ps = pro_scale; p.pb = pro_shift; p.y = y; p.ws = (float*)ws;
    cudaStream_t st = as_stream(stream);
    if (p.Cin == 4 && p.ics == 4 && p.ico == 0 && p.Cout == 64 && p.ocs == 64 && p.oco == 0 && p.kd == 1 && p.kh == 3 &&
        p.kw == 3 && p.stride == 1 && p.pd == 0 && p.ph == 1 && p.pw == 1 && p.D == 1 && p.pro == G6D_PRO_NONE &&
        p.in_items == p.B) {
        conv3x3_c4_o64_kernel<<<ceil_div(p.M, 128), 128, 0, st>>>(x, w, bias, y, p.B, p.H, p.W, p.act);
        G6D_CHECK_LAUNCH("g6d_conv(first layer)");
        return G6D_OK;
    }
    const int bn = p.Cout > 64 ? 128 : (p.Cout > 32 ? 64 : 32);
    dim3 grid(ceil_div(p.M, BM), ceil_div(p.Cout, bn), p.splits);
    if (bn == 128) conv_ffma_kernel<8><<<grid, NT, 0, st>>>(p);
    else if (bn == 64) conv_ffma_kernel<4><<<grid, NT, 0, st>>>(p);
    else conv_ffma_kernel<2><<<grid, NT, 0, st>>>(p);
    G6D_CHECK_LAUNCH("g6d_conv");
    if (p.splits > 1) {
        const long long n = (long long)p.M * p.Cout;
        conv_splitk_reduce_kernel<<<ceil_div(n, 256), 256, 0, st>>>(p.ws, bias, y, p.M, p.Cout, p.splits, p.ocs, p.oco,
                                                                     p.act);
        G6D_CHECK_LAUNCH("g6d_conv(splitk reduce)");
    }
    return G6D_OK;
}

extern "C" int g6d_vgg_first_block(const float* x, const float* w, const float* bias, float* y, int B, int H, int W,
                                   g6d_stream_t stream) {
    G6D_REQUIRE(x && w && y && B > 0 && H >= 2 && W >= 2 && (H & 1) == 0 && (W & 1) == 0, "g6d_vgg_first_block: bad args (H, W even)");
    const long long threads = (long long)B * (H / 2) * (W / 2) * 4;
    conv3x3_c4_o64_relu_pool_kernel<<<ceil_div(threads, 128), 128, 0, as_stream(stream)>>>(x, w, bias, y, B, H, W);
    G6D_CHECK_LAUNCH("g6d_vgg_first_block");
    return G6D_OK;
}

// ------------------------------------------------------------------------------------------
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin,
                                        int Cin_pad, int taps, int ldw, const float* __restrict__ scale) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)taps * Cin_pad * ldw;
    if (i >= total) return;
    const int o = (int)(i % ldw);
    const long long k = i / ldw;
    const int c = (int)(k % Cin_pad);
    const int tap = (int)(k / Cin_pad);
    float v = 0.f;
    if (o < Cout && c < Cin) {
        v = w[((long long)o * Cin + c) * taps + tap];
        if (scale) v *= scale[o];
    }
    out[i] = v;
}

extern "C" int g6d_pack_conv_weight(const float* w, float* out, int Cout, int Cin, int Cin_pad, int taps,
                                    const float* cout_scale, g6d_stream_t stream) {
    G6D_REQUIRE(w && out && Cout > 0 && Cin > 0 && Cin_pad >= Cin && taps > 0, "g6d_pack_conv_weight: bad args");
    const int ldw = (Cout + 3) & ~3;
    const long long total = (long long)taps * Cin_pad * ldw;
    pack_conv_weight_kernel<<<ceil_div(total, 256), 256, 0, as_stream(stream)>>>(w, out, Cout, Cin, Cin_pad, taps, ldw,
                                                                                 cout_scale);
    G6D_CHECK_LAUNCH("g6d_pack_conv_weight");
    return G6D_OK;
}

__global__ void transpose2d_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols, int ldo) {
    __shared__ float tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        tile[j][threadIdx.x] = (r < rows && c < cols) ? in[(long long)r * cols + c] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (c < cols && r < ldo) out[(long long)c * ldo + r] = (r < rows) ? tile[threadIdx.x][j] : 0.f;
    }
}

// in [rows, cols] -> out [cols, ldo] with ldo = rows rounded up to 4 (zero padded): the packed
// [K, Cout] layout g6d_conv expects, for weights that are produced on the device (detector
// reference features used as correlation kernels, detector.py:222-224).
extern "C" int g6d_transpose2d(const float* in, float* out, int rows, int cols, g6d_stream_t stream) {
    G6D_REQUIRE(in && out && rows > 0 && cols > 0, "g6d_transpose2d: bad args");
    const int ldo = (rows + 3) & ~3;
    dim3 grid(ceil_div(cols, 32), ceil_div(ldo, 32));
    transpose2d_kernel<<<grid, dim3(32, 8), 0, as_stream(stream)>>>(in, out, rows, cols, ldo);
    G6D_CHECK_LAUNCH("g6d_transpose2d");
    return G6D_OK;
}

// ------------------------------------------------------------------------------------------
// y[m,n] = act(x[m,:] . w[n,:] + b[n]); one CTA per output feature n streams its weight row once.
template <int MAXM>
__global__ void __launch_bounds__(256) linear_smallm_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ bias, float* __restrict__ y,
                                                            int M, int N, int K, int act) {
    const int n = blockIdx.x;
    const float4* wr = reinterpret_cast<const float4*>(w + (long long)n * K);
    float acc[MAXM];
#pragma unroll
    for (int m = 0; m < MAXM; ++m) acc[m] = 0.f;
    for (int k4 = threadIdx.x; k4 < K / 4; k4 += blockDim.x) {
        const float4 wv = ldg_stream(wr + k4);
#pragma unroll
        for (int m = 0; m < MAXM; ++m) {
            if (m < M) {
                const float4 xv = __ldg(reinterpret_cast<const float4*>(x + (long long)m * K) + k4);
                acc[m] = fmaf(wv.x, xv.x, fmaf(wv.y, xv.y, fmaf(wv.z, xv.z, fmaf(wv.w, xv.w, acc[m]))));
            }
        }
    }
    __shared__ float red[MAXM][8];
#pragma unroll
    for (int m = 0; m < MAXM; ++m) {
        const float v = warp_sum(acc[m]);
        if ((threadIdx.x & 31) == 0) red[m][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < MAXM && threadIdx.x < M) {
        float v = 0.f;
        for (int i = 0; i < 8; ++i) v += red[threadIdx.x][i];
        if (bias) v += bias[n];
        y[(long long)threadIdx.x * N + n] = act_apply(v, act);
    }
}

extern "C" int g6d_linear_smallm(const float* x, const float* w, const float* bias, float* y, int M, int N, int K,
                                 int act, g6d_stream_t stream) {
    G6D_REQUIRE(x && w && y && M > 0 && M <= 8 && N > 0 && K > 0 && (K & 3) == 0, "g6d_linear_smallm: bad args (M<=8, K%%4==0)");
    linear_smallm_kernel<8><<<N, 256, 0, as_stream(stream)>>>(x, w, bias, y, M, N, K, act);
    G6D_CHECK_LAUNCH("g6d_linear_smallm");
    return G6D_OK;
}
