// Selector-specific kernels: the HBM-bound correlation + rotated-similarity score (S2), the
// closed-form first-InstanceNorm statistics, and the small latency-bound tail ops (S4).
#include <stdlib.h>

#include "common.cuh"

namespace g6d {

// ------------------------------------------------------------------------------------------
// S2: score[s] = sum_p t_p^2 / max_p t_p with t_p = sum_c q[p,c] * ref[s,p,c]
// (selector.py:183-186,192-194).  ref [S,P,C] is read exactly once, as 128-bit streaming loads:
// one warp owns a position p of a slice (C = 512 -> 4 float4 per lane, 2 KB contiguous), the
// query row q[p,:] comes from L1/L2 (0.69 MB total, reused by every slice), the 512-term dot is
// finished with warp shuffles, and the per-slice sum/max with one shared-memory step.
// Grid: persistent-style, blockIdx.x strides over slices so the grid is a multiple of the SM
// count regardless of S.
template <int C>
__global__ void __launch_bounds__(256) sel_corr_score_kernel(const float* __restrict__ ref,
                                                             const float* __restrict__ q, int S, int P,
                                                             float* __restrict__ score) {
    constexpr int V = C / 128;  // float4 per lane
    extern __shared__ float t_sh[];  // [P] per-location inner products of the current slice
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarp = blockDim.x >> 5;
    __shared__ float s_red[8];
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        const float4* rs = reinterpret_cast<const float4*>(ref + (long long)s * P * C);
        float mx = -INFINITY;
        for (int p = warp; p < P; p += nwarp) {
            const float4* rp = rs + (long long)p * (C / 4);
            const float4* qp = reinterpret_cast<const float4*>(q + (long long)p * C);
            float4 rv[V];
#pragma unroll
            for (int i = 0; i < V; ++i) rv[i] = ldg_stream(rp + lane + 32 * i);
            float t = 0.f;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                const float4 qv = __ldg(qp + lane + 32 * i);
                t = fmaf(rv[i].x, qv.x, fmaf(rv[i].y, qv.y, fmaf(rv[i].z, qv.z, fmaf(rv[i].w, qv.w, t))));
            }
            t = warp_sum(t);
            if (lane == 0) t_sh[p] = t;
            mx = fmaxf(mx, t);
        }
        if (lane == 0) s_red[warp] = mx;
        __syncthreads();
        float m = s_red[0];
        for (int w = 1; w < nwarp; ++w) m = fmaxf(m, s_red[w]);
        __syncthreads();
        // score = sum_p t * (t / max), with the reference's operation order (selector.py:193-194)
        // and IEEE behaviour when max <= 0 (no epsilon in the reference).
        float acc = 0.f;
        for (int p = threadIdx.x; p < P; p += blockDim.x) { const float t = t_sh[p]; acc += t * (t / m); }
        acc = warp_sum(acc);
        if (lane == 0) s_red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            float a = 0.f;
            for (int w = 0; w < nwarp; ++w) a += s_red[w];
            score[s] = a;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// S2, all pyramid levels and all qn queries in ONE streaming pass (what select_que_imgs uses):
// phase 1 computes every per-location inner product t[g, row] for row = (level, slice, location)
// with a grid-stride loop over rows -- the grid is sized to fill every SM with 32 resident warps
// regardless of S (64 registers: the two rows stay in registers across the query loop), and each
// warp keeps two 2 KB reference rows (8 x 128-bit loads per lane, 128 KB per SM) in flight and
// dots them with the rows of all qn queries (small, L2-resident), so the reference
// stack is read from HBM once per batch, not once per query; phase 2 (tiny, L2-resident) reduces
// each (query, level, slice) to sum_p t*(t/max_p t).
struct ScoreLevels {
    const float* ref[3];   // [S, P_l, C]
    const float* q[3];     // [qn, P_l, C]
    int P[3];
    int S, qn;
    long long row_end[3];  // cumulative row counts: S*P_0, S*(P_0+P_1), S*(P_0+P_1+P_2)
};

template <int C>
__device__ __forceinline__ void row_load(const float4* __restrict__ rp, int lane, float4 (&rv)[C / 128]) {
#pragma unroll
    for (int i = 0; i < C / 128; ++i) rv[i] = ldg_stream(rp + lane + 32 * i);
}
template <int C>
__device__ __forceinline__ float row_dot(const float4 (&rv)[C / 128], const float4* __restrict__ qp, int lane) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < C / 128; ++i) {
        const float4 qv = __ldg(qp + lane + 32 * i);
        t = fmaf(rv[i].x, qv.x, fmaf(rv[i].y, qv.y, fmaf(rv[i].z, qv.z, fmaf(rv[i].w, qv.w, t))));
    }
    return t;
}

// FUSED: every CTA streams one CONTIGUOUS chunk of rows, then (one __threadfence per warp, one
// __syncthreads) adds the rows it contributed to each (query, level, slice) item it touched to that
// item's completion counter; the CTA that completes an item reduces its P inner products to the score
// with the reference's operation order (selector.py:192-194: s / max first, then sum of s * (s / max);
// IEEE behaviour for max <= 0, no epsilon).  ~6 qn atomics per CTA, no second launch.  t_out is
// [qn, rows], score [qn, 3, S], done [qn, 3, S].
template <int C, bool FUSED>
__global__ void __launch_bounds__(256, 4) sel_corr_dots_kernel(const ScoreLevels L, float* __restrict__ t_out,
                                                            int* __restrict__ done, float* __restrict__ score,
                                                            long long chunk) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long rows = L.row_end[2];
    auto locate = [&](long long row, const float4*& rp, const float4*& qp, int& item, int& P, long long& first) {
        // static selects (no dynamic indexing of the parameter struct -> no local-memory copy)
        const bool l0 = row < L.row_end[0], l1 = row < L.row_end[1];
        const long long lbase = l0 ? 0 : (l1 ? L.row_end[0] : L.row_end[1]);
        const long long local = row - lbase;                                                // = s*P_l + p
        P = l0 ? L.P[0] : (l1 ? L.P[1] : L.P[2]);
        const float* ref = l0 ? L.ref[0] : (l1 ? L.ref[1] : L.ref[2]);
        const float* q = l0 ? L.q[0] : (l1 ? L.q[1] : L.q[2]);
        const int sl = (int)(local / P);
        const int p = (int)(local - (long long)sl * P);
        item = (l0 ? 0 : (l1 ? 1 : 2)) * L.S + sl;
        first = lbase + (long long)sl * P;
        rp = reinterpret_cast<const float4*>(ref + local * C);
        qp = reinterpret_cast<const float4*>(q + (long long)p * C);              // query 0; query g at + g*P*C
    };
    long long begin, end, stride;
    if (FUSED) {        // contiguous chunk per CTA, row pairs dealt to its 8 warps
        begin = (long long)blockIdx.x * chunk;
        end = min(rows, begin + chunk);
        stride = 16;
    } else {            // grid-stride over all rows
        begin = 0; end = rows;
        stride = (((long long)gridDim.x * blockDim.x) >> 5) * 2;
    }
    const long long w0 = FUSED ? wib : (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    for (long long row = begin + w0 * 2; row < end; row += stride) {
        const float4 *r0, *q0, *r1, *q1;
        int item, P;
        long long first;
        locate(row, r0, q0, item, P, first);
        const bool two = row + 1 < end;
        const int P0 = P;
        locate(two ? row + 1 : row, r1, q1, item, P, first);
        float4 v0[C / 128], v1[C / 128];
        row_load<C>(r0, lane, v0);
        row_load<C>(r1, lane, v1);
        // same products and summation order for every query as a one-query call: bit-identical t
        for (int g = 0; g < L.qn; ++g) {
            float t0 = row_dot<C>(v0, q0 + (long long)g * P0 * (C / 4), lane);
            float t1 = row_dot<C>(v1, q1 + (long long)g * P * (C / 4), lane);
            t0 = warp_sum(t0);
            t1 = warp_sum(t1);
            if (lane == 0) {
                t_out[g * rows + row] = t0;
                if (two) t_out[g * rows + row + 1] = t1;
            }
        }
    }
    if (!FUSED) return;
    if (lane == 0) __threadfence();                // this warp's t values are visible device-wide ...
    __syncthreads();                               // ... before any thread of the CTA counts them in
    // the (item, query) pairs this chunk overlaps, dealt round-robin to the warps
    int n = 0;
    for (long long r = begin; r < end;) {
        const float4 *rp, *qp;
        int item, P;
        long long first;
        locate(r, rp, qp, item, P, first);
        const long long next = min(end, first + P);
        for (int g = 0; g < L.qn; ++g, ++n) {
            if ((n & 7) != wib) continue;
            const long long gi = (long long)g * 3 * L.S + item;
            int last = 0;
            if (lane == 0) last = atomicAdd(done + gi, (int)(next - r)) + (int)(next - r) == P;
            last = __shfl_sync(0xffffffffu, last, 0);
            if (last) {                                                   // warp-uniform
                if (lane == 0) done[gi] = 0;                              // leave the counters zero for the next call
                __threadfence();                                          // acquire: the other CTAs' t values
                const float* tp = t_out + g * rows + first;
                float m = -INFINITY;
                for (int p = lane; p < P; p += 32) m = fmaxf(m, __ldcg(tp + p));
                m = warp_max(m);
                float acc = 0.f;
                for (int p = lane; p < P; p += 32) { const float v = __ldcg(tp + p); acc += v * (v / m); }
                acc = warp_sum(acc);
                if (lane == 0) score[gi] = acc;         // [qn, 3, S]
            }
        }
        r = next;
    }
}

// one warp per (query, level, slice): score = sum_p t*(t/max_p t), reference operation order (unfused path)
__global__ void sel_corr_finish_kernel(const ScoreLevels L, const float* __restrict__ t, float* __restrict__ score) {
    const int lane = threadIdx.x & 31;
    const int item = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (item >= 3 * L.S * L.qn) return;
    const int g = item / (3 * L.S), li = item % (3 * L.S);
    const int l = li / L.S, s = li % L.S;
    const int P = l == 0 ? L.P[0] : (l == 1 ? L.P[1] : L.P[2]);
    const float* tp = t + g * L.row_end[2] + (l == 0 ? 0 : (l == 1 ? L.row_end[0] : L.row_end[1])) + (long long)s * P;
    float m = -INFINITY;
    for (int p = lane; p < P; p += 32) m = fmaxf(m, tp[p]);
    m = warp_max(m);
    float acc = 0.f;
    for (int p = lane; p < P; p += 32) { const float v = tp[p]; acc += v * (v / m); }
    acc = warp_sum(acc);
    if (lane == 0) score[item] = acc;       // [qn, 3, S]
}

// ------------------------------------------------------------------------------------------
// sum_s ref and sum_s ref^2 over the slice axis, doubles [P*C].  Load-time (once per object).
__global__ void sel_ref_sums_kernel(const float* __restrict__ ref, int S, long long PC, int s_chunk,
                                    double* __restrict__ sum1, double* __restrict__ sum2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= PC) return;
    const int s0 = blockIdx.y * s_chunk, s1 = min(S, s0 + s_chunk);
    double a = 0.0, b = 0.0;
    for (int s = s0; s < s1; ++s) {
        const double v = (double)ref[(long long)s * PC + i];
        a += v; b += v * v;
    }
    atomicAdd(sum1 + i, a);
    atomicAdd(sum2 + i, b);
}

// Per query g and channel c: mean_c = sum_p q[p,c]*A[p,c] / N, E2_c = sum_p q[p,c]^2*B[p,c] / N, N = S*P;
// then scale[p,c] = q[p,c]*rstd_c and shift[c] = -mean_c*rstd_c.  One block per (32 channels, query).
__global__ void sel_corr_prologue_kernel(const float* __restrict__ q, const double* __restrict__ sum1,
                                         const double* __restrict__ sum2, int S, int P, int C, float eps,
                                         float* __restrict__ scale, float* __restrict__ shift) {
    q += (long long)blockIdx.y * P * C;
    scale += (long long)blockIdx.y * P * C;
    shift += (long long)blockIdx.y * C;
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int row = threadIdx.x >> 5, nrow = blockDim.x >> 5;
    __shared__ double sm[8][32], sv[8][32];
    __shared__ float s_rstd[32];
    double m = 0.0, e2 = 0.0;
    if (c < C) {
        for (int p = row; p < P; p += nrow) {
            const double qv = (double)q[(long long)p * C + c];
            m += qv * sum1[(long long)p * C + c];
            e2 += qv * qv * sum2[(long long)p * C + c];
        }
    }
    sm[row][threadIdx.x & 31] = m; sv[row][threadIdx.x & 31] = e2;
    __syncthreads();
    if (row == 0 && c < C) {
        for (int r = 1; r < nrow; ++r) { m += sm[r][threadIdx.x]; e2 += sv[r][threadIdx.x]; }
        const double n = (double)S * (double)P;
        const double mean = m / n;
        double var = e2 / n - mean * mean;
        var = var < 0.0 ? 0.0 : var;
        const double rstd = 1.0 / sqrt(var + (double)eps);
        s_rstd[threadIdx.x] = (float)rstd;
        shift[c] = (float)(-mean * rstd);
    }
    __syncthreads();
    if (c < C) {
        const float r = s_rstd[threadIdx.x & 31];
        for (int p = row; p < P; p += nrow) scale[(long long)p * C + c] = q[(long long)p * C + c] * r;
    }
}

// vp_norm: InstanceNorm2d over n values per (group, level); scatter to feats[g*n + i, coff + l].  Block (l, g).
__global__ void sel_vp_norm_kernel(const float* __restrict__ score, int n, float eps, float* __restrict__ feats,
                                   int cstride, int coff) {
    const int l = blockIdx.x;
    const float* s = score + ((long long)blockIdx.y * gridDim.x + l) * n;
    feats += (long long)blockIdx.y * n * cstride;
    __shared__ double r1[32], r2[32];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { const double v = s[i]; a += v; b += v * v; }
    a = warp_sum(a); b = warp_sum(b);
    if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = a; r2[threadIdx.x >> 5] = b; }
    __syncthreads();
    a = 0.0; b = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += r1[w]; b += r2[w]; }
    const double mean = a / n;
    double var = b / n - mean * mean;
    var = var < 0.0 ? 0.0 : var;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float fm = (float)mean;
    for (int i = threadIdx.x; i < n; i += blockDim.x) feats[(long long)i * cstride + coff + l] = (s[i] - fm) * rstd;
    // the channels between the last score and the row end are padding the consumer multiplies by zero
    // weights: they must be finite, so the first block of each group clears them (no separate fill pass over feats)
    if (l == 0)
        for (int c = coff + (int)gridDim.x; c < cstride; ++c)
            for (int i = threadIdx.x; i < n; i += blockDim.x) feats[(long long)i * cstride + c] = 0.f;
}

// rows = groups * rfn; the embedding [rfn, C] is shared by every group
__global__ void sel_max_angle_add_kernel(const float* __restrict__ x, const float* __restrict__ embed,
                                         float* __restrict__ out, int rows, int rfn, int an, int C) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * C) return;
    const int c = (int)(i % C);
    const int r = (int)(i / C);
    float m = -INFINITY;
    for (int a = 0; a < an; ++a) m = fmaxf(m, x[((long long)r * an + a) * C + c]);
    out[i] = m + embed[(long long)(r % rfn) * C + c];
}

// attention: one block per (query token i, head h); channel c = d*heads + h.
// scores over keys in shared memory, softmax, then the weighted value sum.
__global__ void attention_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                                 float* __restrict__ out, int n, int C, int heads) {
    extern __shared__ float sh[];  // [n] probabilities + [D] query
    const int i = blockIdx.x, h = blockIdx.y;
    const long long go = (long long)blockIdx.z * n * C;      // group: n tokens of its own
    q += go; k += go; v += go; out += go;
    const int D = C / heads;
    float* prob = sh;
    float* qv = sh + n;
    for (int d = threadIdx.x; d < D; d += blockDim.x) qv[d] = q[(long long)i * C + d * heads + h];
    __syncthreads();
    const float inv = rsqrtf((float)D);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        float s = 0.f;
        for (int d = 0; d < D; ++d) s = fmaf(qv[d], k[(long long)j * C + d * heads + h], s);
        prob[j] = s * inv;
    }
    __syncthreads();
    __shared__ float red[32];
    float m = -INFINITY;
    for (int j = threadIdx.x; j < n; j += blockDim.x) m = fmaxf(m, prob[j]);
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float sum = 0.f;
    for (int j = threadIdx.x; j < n; j += blockDim.x) { const float e = expf(prob[j] - m); prob[j] = e; sum += e; }
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    sum = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += red[w];
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float acc = 0.f;
        for (int j = 0; j < n; ++j) acc = fmaf(prob[j], v[(long long)j * C + d * heads + h], acc);
        out[(long long)i * C + d * heads + h] = acc / sum;
    }
}

// Tiled attention over HEAD-MAJOR channels (c = head*D + d, D = 64): the layout the selector's packed
// conv_query / conv_key / conv_feats emit (their output rows are permuted at pack time, conv_merge's input
// columns likewise, so nothing is transposed at run time).  A block owns (8 query tokens, one head): the
// K and V tiles of 32 keys x 64 dims are staged in shared memory by coalesced 128-bit loads ONCE per
// block, scores for all n keys live in shared memory (n <= 2048), softmax(q.k / sqrt(D)) over keys as in
// attention.py:4-17.  The per-(token, head) kernel above re-reads every key row with a 32-byte stride:
// 4.3 GB of L2 traffic at n = 512 (a reference-sharded selector over 8 GPUs); this one reads 67 MB.
constexpr int ATT_TQ = 8, ATT_TK = 32, ATT_D = 64;
__global__ void __launch_bounds__(128) attention_hm_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                           const float* __restrict__ v, float* __restrict__ out, int n, int C) {
    extern __shared__ float sh[];
    const int npad = (n + 31) & ~31;
    float* qs = sh;                                  // [TQ][D]
    float* kt = qs + ATT_TQ * ATT_D;                 // [TK][D+1]
    float* sc = kt + ATT_TK * (ATT_D + 1);           // [TQ][npad]
    __shared__ float s_sum[ATT_TQ];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int i0 = blockIdx.x * ATT_TQ, h = blockIdx.y;
    const long long go = (long long)blockIdx.z * n * C;      // group: n tokens of its own
    q += go; k += go; v += go; out += go;
    const float inv = rsqrtf((float)ATT_D);
    for (int e = t; e < ATT_TQ * ATT_D; e += 128) {
        const int qi = e / ATT_D, d = e % ATT_D;
        qs[e] = i0 + qi < n ? q[(long long)(i0 + qi) * C + h * ATT_D + d] : 0.f;
    }
    // ---- scores
    for (int j0 = 0; j0 < n; j0 += ATT_TK) {
        __syncthreads();
        for (int e = t; e < ATT_TK * ATT_D / 4; e += 128) {             // 16 float4 per key row
            const int jj = e >> 4, d4 = e & 15;
            float4 kv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j0 + jj < n) kv = __ldg(reinterpret_cast<const float4*>(k + (long long)(j0 + jj) * C + h * ATT_D) + d4);
            float* dst = kt + jj * (ATT_D + 1) + d4 * 4;
            dst[0] = kv.x; dst[1] = kv.y; dst[2] = kv.z; dst[3] = kv.w;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int qi = warp + 4 * r;                                  // warp-uniform: the q row broadcasts
            const float* qr = qs + qi * ATT_D;
            const float* kr = kt + lane * (ATT_D + 1);
            float a = 0.f;
#pragma unroll 16
            for (int d = 0; d < ATT_D; ++d) a = fmaf(qr[d], kr[d], a);
            sc[qi * npad + j0 + lane] = a * inv;
        }
    }
    __syncthreads();
    // ---- softmax over the n keys, two query rows per warp
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int qi = warp + 4 * r;
        float* row = sc + qi * npad;
        float m = -INFINITY;
        for (int j = lane; j < n; j += 32) m = fmaxf(m, row[j]);
        m = warp_max(m);
        float sum = 0.f;
        for (int j = lane; j < n; j += 32) { const float e = expf(row[j] - m); row[j] = e; sum += e; }
        sum = warp_sum(sum);
        if (lane == 0) s_sum[qi] = sum;
    }
    // ---- weighted value sum: thread = (d, 4 query rows)
    const int d = t & 63, qh = t >> 6;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j0 = 0; j0 < n; j0 += ATT_TK) {
        __syncthreads();
        for (int e = t; e < ATT_TK * ATT_D / 4; e += 128) {
            const int jj = e >> 4, d4 = e & 15;
            float4 vv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j0 + jj < n) vv = __ldg(reinterpret_cast<const float4*>(v + (long long)(j0 + jj) * C + h * ATT_D) + d4);
            float* dst = kt + jj * (ATT_D + 1) + d4 * 4;
            dst[0] = vv.x; dst[1] = vv.y; dst[2] = vv.z; dst[3] = vv.w;
        }
        __syncthreads();
        const int jn = min(ATT_TK, n - j0);
        for (int jj = 0; jj < jn; ++jj) {
            const float vv = kt[jj * (ATT_D + 1) + d];
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[r] = fmaf(sc[(qh + 2 * r) * npad + j0 + jj], vv, acc[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int qi = qh + 2 * r;
        if (i0 + qi < n) out[(long long)(i0 + qi) * C + h * ATT_D + d] = acc[r] / s_sum[qi];
    }
}

__global__ void layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, float* __restrict__ out, int rows, int C, float eps) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* xr = x + (long long)row * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += xr[c];
    const float mean = warp_sum(s) / (float)C;
    float v = 0.f;
    for (int c = lane; c < C; c += 32) { const float d = xr[c] - mean; v = fmaf(d, d, v); }
    const float rstd = rsqrtf(warp_sum(v) / (float)C + eps);
    for (int c = lane; c < C; c += 32) out[(long long)row * C + c] = (xr[c] - mean) * rstd * gamma[c] + beta[c];
}

__global__ void sel_parse_kernel(const float* __restrict__ logits, const float* __restrict__ angles, int rfn,
                                 long long* __restrict__ out_idx, float* __restrict__ out) {
    const int qi = blockIdx.x;
    if (threadIdx.x != 0) return;
    const float* l = logits + (long long)qi * rfn;
    int best = 0;
    float bv = l[0];
    for (int r = 1; r < rfn; ++r)      // first maximum; NaN counts as the maximum (torch.argmax, selector.py:172)
        if (l[r] > bv || (l[r] != l[r] && bv == bv)) { bv = l[r]; best = r; }
    out_idx[qi] = best;
    out[qi * 2 + 0] = angles[(long long)qi * rfn + best];
    out[qi * 2 + 1] = bv;
}

}  // namespace g6d

using namespace g6d;

extern "C" int g6d_sel_corr_score(const float* ref, const float* q, int S, int P, int C, float* score,
                                  g6d_stream_t stream) {
    G6D_REQUIRE(ref && q && score && S > 0 && P > 0, "g6d_sel_corr_score: bad args");
    G6D_REQUIRE(C == 512 || C == 256 || C == 128, "g6d_sel_corr_score: C must be 128, 256 or 512 (got %d)", C);
    G6D_REQUIRE(P <= 8192, "g6d_sel_corr_score: P too large");
    const int grid = S < 8 * kNumSMs ? S : 8 * kNumSMs;
    const size_t smem = sizeof(float) * P;
    cudaStream_t st = as_stream(stream);
    if (C == 512) sel_corr_score_kernel<512><<<grid, 256, smem, st>>>(ref, q, S, P, score);
    else if (C == 256) sel_corr_score_kernel<256><<<grid, 256, smem, st>>>(ref, q, S, P, score);
    else sel_corr_score_kernel<128><<<grid, 256, smem, st>>>(ref, q, S, P, score);
    G6D_CHECK_LAUNCH("g6d_sel_corr_score");
    return G6D_OK;
}

extern "C" long long g6d_sel_corr_score3_workspace_bytes(int S, int P0, int P1, int P2, int qn) {
    if (S <= 0 || P0 <= 0 || P1 <= 0 || P2 <= 0 || qn <= 0) { set_error("g6d_sel_corr_score3_workspace_bytes: bad args"); return -1; }
    const long long rows = (long long)qn * S * ((long long)P0 + P1 + P2);
    return ((rows + 3) / 4) * 4 * (long long)sizeof(float);
}

extern "C" int g6d_sel_corr_score3(const float* ref0, const float* ref1, const float* ref2, const float* q0,
                                   const float* q1, const float* q2, int S, int P0, int P1, int P2, int C, int qn,
                                   float* score, float* ws, int* counters, g6d_stream_t stream) {
    G6D_REQUIRE(ref0 && ref1 && ref2 && q0 && q1 && q2 && score && ws && S > 0 && P0 > 0 && P1 > 0 && P2 > 0 && qn > 0,
                "g6d_sel_corr_score3: bad args");
    G6D_REQUIRE(C == 512, "g6d_sel_corr_score3: C must be 512 (got %d)", C);
    G6D_REQUIRE(3ll * S * qn < (1ll << 31), "g6d_sel_corr_score3: too many (query, level, slice) items");
    ScoreLevels L;
    L.ref[0] = ref0; L.ref[1] = ref1; L.ref[2] = ref2; L.q[0] = q0; L.q[1] = q1; L.q[2] = q2;
    L.P[0] = P0; L.P[1] = P1; L.P[2] = P2; L.S = S; L.qn = qn;
    L.row_end[0] = (long long)S * P0; L.row_end[1] = L.row_end[0] + (long long)S * P1;
    L.row_end[2] = L.row_end[1] + (long long)S * P2;
    cudaStream_t st = as_stream(stream);
    static int fused = -1;
    if (fused < 0) { const char* e = getenv("G6D_S2_FUSED"); fused = (e && e[0] == '0') ? 0 : 1; }
    // one wave: as many CTAs per SM as are actually resident (the chunked kernel must not need a second wave)
    static int occ[2] = {0, 0};
    if (occ[fused] == 0) {
        int n = 0;
        cudaError_t e = fused ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, sel_corr_dots_kernel<512, true>, 256, 0)
                              : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, sel_corr_dots_kernel<512, false>, 256, 0);
        occ[fused] = (e == cudaSuccess && n > 0) ? n : 4;
    }
    const long long pairs = (L.row_end[2] + 1) / 2;
    long long grid = (pairs + 7) / 8;                    // 8 warps per CTA, one row pair per warp per trip
    const long long full = (long long)occ[fused] * kNumSMs;
    if (grid > full) grid = full;
    if (fused && counters) {
        int* done = counters;
        long long chunk = (L.row_end[2] + grid - 1) / grid;
        chunk += chunk & 1;                                  // even: row pairs never straddle two CTAs
        grid = (L.row_end[2] + chunk - 1) / chunk;
        sel_corr_dots_kernel<512, true><<<(unsigned)grid, 256, 0, st>>>(L, ws, done, score, chunk);
        G6D_CHECK_LAUNCH("g6d_sel_corr_score3");
        return G6D_OK;
    }
    sel_corr_dots_kernel<512, false><<<(unsigned)grid, 256, 0, st>>>(L, ws, nullptr, nullptr, 0);
    G6D_CHECK_LAUNCH("g6d_sel_corr_score3(dots)");
    sel_corr_finish_kernel<<<ceil_div(3ll * S * qn * 32, 256), 256, 0, st>>>(L, ws, score);
    G6D_CHECK_LAUNCH("g6d_sel_corr_score3(finish)");
    return G6D_OK;
}

extern "C" int g6d_sel_ref_sums(const float* ref, int S, int P, int C, double* sum1, double* sum2,
                                g6d_stream_t stream) {
    G6D_REQUIRE(ref && sum1 && sum2 && S > 0 && P > 0 && C > 0, "g6d_sel_ref_sums: bad args");
    const long long PC = (long long)P * C;
    cudaStream_t st = as_stream(stream);
    cudaError_t e = cudaMemsetAsync(sum1, 0, sizeof(double) * PC, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(sum2, 0, sizeof(double) * PC, st);
    if (e != cudaSuccess) { set_error("g6d_sel_ref_sums: memset failed: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
    const int s_chunk = 16;
    dim3 grid(ceil_div(PC, 256), ceil_div(S, s_chunk));
    sel_ref_sums_kernel<<<grid, 256, 0, st>>>(ref, S, PC, s_chunk, sum1, sum2);
    G6D_CHECK_LAUNCH("g6d_sel_ref_sums");
    return G6D_OK;
}

extern "C" int g6d_sel_corr_prologue(const float* q, const double* sum1, const double* sum2, int S, int P, int C, int qn,
                                     float eps, float* scale, float* shift, g6d_stream_t stream) {
    G6D_REQUIRE(q && sum1 && sum2 && scale && shift && S > 0 && P > 0 && C > 0 && qn > 0 && qn <= 65535,
                "g6d_sel_corr_prologue: bad args");
    sel_corr_prologue_kernel<<<dim3(ceil_div(C, 32), qn), 256, 0, as_stream(stream)>>>(q, sum1, sum2, S, P, C, eps, scale, shift);
    G6D_CHECK_LAUNCH("g6d_sel_corr_prologue");
    return G6D_OK;
}

extern "C" int g6d_sel_vp_norm(const float* score, int groups, int L, int n, float eps, float* feats, int cstride, int coff,
                               g6d_stream_t stream) {
    G6D_REQUIRE(score && feats && groups > 0 && groups <= 65535 && L > 0 && n > 0 && coff + L <= cstride,
                "g6d_sel_vp_norm: bad args");
    sel_vp_norm_kernel<<<dim3(L, groups), 256, 0, as_stream(stream)>>>(score, n, eps, feats, cstride, coff);
    G6D_CHECK_LAUNCH("g6d_sel_vp_norm");
    return G6D_OK;
}

extern "C" int g6d_sel_max_angle_add(const float* x, const float* embed, float* out, int groups, int rfn, int an, int C,
                                     g6d_stream_t stream) {
    G6D_REQUIRE(x && embed && out && groups > 0 && rfn > 0 && an > 0 && C > 0 && (long long)groups * rfn < (1ll << 31),
                "g6d_sel_max_angle_add: bad args");
    const int rows = groups * rfn;
    sel_max_angle_add_kernel<<<ceil_div((long long)rows * C, 256), 256, 0, as_stream(stream)>>>(x, embed, out, rows, rfn, an, C);
    G6D_CHECK_LAUNCH("g6d_sel_max_angle_add");
    return G6D_OK;
}

extern "C" int g6d_attention(const float* q, const float* k, const float* v, float* out, int groups, int n, int C, int heads,
                             g6d_stream_t stream) {
    G6D_REQUIRE(q && k && v && out && groups > 0 && groups <= 65535 && n > 0 && n <= 8192 && heads > 0 && C % heads == 0,
                "g6d_attention: bad args");
    const size_t smem = sizeof(float) * (n + C / heads);
    attention_kernel<<<dim3(n, heads, groups), 64, smem, as_stream(stream)>>>(q, k, v, out, n, C, heads);
    G6D_CHECK_LAUNCH("g6d_attention");
    return G6D_OK;
}

extern "C" int g6d_attention_headmajor(const float* q, const float* k, const float* v, float* out, int groups, int n, int C,
                                       int heads, g6d_stream_t stream) {
    G6D_REQUIRE(q && k && v && out && groups > 0 && groups <= 65535 && n > 0 && n <= 2048 && heads > 0 &&
                C == heads * ATT_D && (C & 3) == 0, "g6d_attention_headmajor: bad args (n <= 2048, C = heads * 64)");
    const int npad = (n + 31) & ~31;
    const size_t smem = sizeof(float) * (ATT_TQ * ATT_D + ATT_TK * (ATT_D + 1) + (size_t)ATT_TQ * npad);
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(attention_hm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
        if (e != cudaSuccess) { set_error("g6d_attention_headmajor: %s", cudaGetErrorString(e)); return G6D_ECUDA; }
        configured = true;
    }
    attention_hm_kernel<<<dim3(ceil_div(n, ATT_TQ), heads, groups), 128, smem, as_stream(stream)>>>(q, k, v, out, n, C);
    G6D_CHECK_LAUNCH("g6d_attention_headmajor");
    return G6D_OK;
}

extern "C" int g6d_layernorm(const float* x, const float* gamma, const float* beta, float* out, int rows, int C,
                             float eps, g6d_stream_t stream) {
    G6D_REQUIRE(x && gamma && beta && out && rows > 0 && C > 0, "g6d_layernorm: bad args");
    layernorm_kernel<<<ceil_div(rows, 4), 128, 0, as_stream(stream)>>>(x, gamma, beta, out, rows, C, eps);
    G6D_CHECK_LAUNCH("g6d_layernorm");
    return G6D_OK;
}

extern "C" int g6d_sel_parse(const float* logits, const float* angles, int qn, int rfn, long long* out_idx, float* out,
                             g6d_stream_t stream) {
    G6D_REQUIRE(logits && angles && out_idx && out && qn > 0 && rfn > 0, "g6d_sel_parse: bad args");
    sel_parse_kernel<<<qn, 32, 0, as_stream(stream)>>>(logits, angles, rfn, out_idx, out);
    G6D_CHECK_LAUNCH("g6d_sel_parse");
    return G6D_OK;
}
