/*
 * gen6d_b200.h -- C ABI of libgen6d_b200.so: the sm_100a kernels behind the Gen6D inference
 * hot path (detector correlation head, selector similarity scoring, refiner feature volume +
 * conv stacks).
 *
 * The reference (liuyuan-pal/Gen6D) is pure PyTorch and has no FFI of its own (SURVEY.md 8b);
 * this header is the "lower face" of the drop-in boundary: the entry points that the Python
 * classes mirroring network/{detector,selector,refiner}.py bind with ctypes.  Each entry cites
 * the reference call site whose arithmetic it replaces.
 *
 * Conventions
 *  - every function returns 0 on success, a negative G6D_E* code otherwise;
 *    g6d_last_error() gives a thread-local message for the last failure on this thread;
 *  - all pointers are DEVICE pointers unless the parameter is named host_*; the caller owns
 *    every buffer (inputs, outputs, workspaces); the library never allocates device memory,
 *    never synchronises, and only enqueues work on the `stream` it is given (so calls can be
 *    captured into CUDA graphs);
 *  - activations are fp32, channels-last: [B, (D,) H, W, C] with C contiguous.  The NCHW
 *    tensors of the reference API are converted at the Python boundary with
 *    g6d_nchw_to_nhwc / g6d_nhwc_to_nchw;
 *  - convolution weights are packed [K, ldw] (ldw = Cout rounded up to 4) with
 *    K = ((kz*kh + ky)*kw + kx)*Cin + c
 *    (g6d_pack_conv_weight does this from the reference's [Cout, Cin, kd, kh, kw]).
 */
#ifndef GEN6D_B200_H
#define GEN6D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G6D_OK 0
#define G6D_EINVAL (-1)   /* bad argument / unsupported shape */
#define G6D_ECUDA (-2)    /* CUDA runtime error at launch */

typedef void* g6d_stream_t; /* cudaStream_t */

const char* g6d_last_error(void);
int g6d_version(void);
/* number of kernel launches issued through this library since load (all threads) */
long long g6d_launch_count(void);

/* ------------------------------------------------------------------ layout / image ops ---- */
/* utils/base_utils.py:117-118 color_map_forward (+ torchvision Normalize of
 * network/detector.py:156,189 when imagenet_norm != 0).  u8 [n_pixels,3] -> f32 [n_pixels,out_c],
 * out_c = 3 or 4 (channel 3 = 0: padding so the first VGG conv can use 128-bit loads). */
int g6d_preprocess_u8(const uint8_t* img, float* out, long long n_pixels, int out_c, int imagenet_norm,
                      g6d_stream_t stream);
/* One image warp: `src` is a device uint8 [rows, cols, 3] image; M is the row-major DST -> SRC map
 * (what OpenCV holds after its internal inversion: cv::invert of the 3x3 for warpPerspective; the
 * closed-form 2x3 inverse, rows M[0..2] and M[3..5], for warpAffine - M[6..8] unused there). */
typedef struct g6d_warp_job {
    const uint8_t* src;
    int rows, cols;
    double M[9];
} g6d_warp_job;
/* cv2.warpPerspective(src, H, (w, h), flags=INTER_LINEAR) with a zero constant border, bit-exact with
 * OpenCV's 8-bit fixed-point path, for n_jobs (image, matrix) pairs at once: the look-at crops of
 * network/refiner.py:285-325 (utils/database_utils.py:8-25 look_at_crop, :54-110
 * normalize_reference_views).  jobs: DEVICE array [n_jobs]; out u8 [n_jobs, h, w, 3]. */
int g6d_warp_perspective_u8(const g6d_warp_job* jobs, int n_jobs, uint8_t* out, int h, int w, g6d_stream_t stream);
/* cv2.warpAffine(src, M, (w, h), flags=INTER_LINEAR), same conventions: the detection crop of
 * estimator.py:184 (utils/base_utils.py:646-655 transformation_crop). */
int g6d_warp_affine_u8(const g6d_warp_job* jobs, int n_jobs, uint8_t* out, int h, int w, g6d_stream_t stream);

/* ---- camera algebra between the stages, on the device (estimator.py:176-214; utils/pose_utils.py:12-58,104-111,
 * 217-244; utils/database_utils.py:8-25,54-139; dataset/database.py:400-404,667-694).  With these four launches a
 * batched prediction detect -> select -> refine x N is one stream-ordered sequence with no host round trip.  The
 * *_host variants run the identical code on host memory (unit tests against the numpy restatement). */
typedef struct g6d_glue_camera {   /* one query frame; filled by the caller (numpy), float64 VALUES of:           */
    double K[9];                   /*   the intrinsics,                                                           */
    double Kinv[9];                /*   np.linalg.inv(K) evaluated in K's own dtype,                              */
    double f;                      /*   (K[0,0] + K[1,1]) / 2 evaluated in K's own dtype,                         */
    double f_sq;                   /*   f ** 2 evaluated in K's own dtype (a float32 K squares in float32)        */
} g6d_glue_camera;
typedef struct g6d_glue_refs {     /* the selector's reference views (device arrays, built once per object)       */
    const double* poses;           /* [rfn,12] normalised reference poses (estimator.py:167 ref_info['poses'])    */
    const double* cen;             /* [rfn,2]  projected object centre                                            */
    const double* f;               /* [rfn]    (K00 + K11) / 2                                                    */
    const double* dist;            /* [rfn]    |camera centre - object centre|                                    */
    double center[3];
} g6d_glue_refs;
typedef struct g6d_glue_views {    /* the refiner's database views in unit-sphere coordinates (device arrays)     */
    const double* poses;           /* [n,12] */
    const double* R_look;          /* [n,9]  look-at rotation of every view                                        */
    const double* RlookR;          /* [n,9]  R_look @ R                                                            */
    const double* f;               /* [n]    focal length of the normalised crop                                   */
    const double* Kinv;            /* [n,9]  */
    const unsigned long long* src; /* [n]    device address of the view's uint8 [rows, cols, 3] image              */
    const int* rows; const int* cols;
    const int* even_idx;           /* [n_even] table rows of the FPS re-spread subset (database_utils.py:129-134)  */
    const float* even_dirs;        /* [n_even,3] their unit viewing directions                                     */
    int n_views, n_even, ref_num, size;
    double norm_scale;             /* 2 / object diameter                                                          */
    float norm_offset[3];          /* -norm_scale * object centre (float32, as numpy holds it)                     */
    float size_scale;              /* float32(size * (1 - margin) / 2)                                             */
} g6d_glue_views;
/* det_out [qn,4] (x, y, scale, score; g6d_det_parse) -> the selector's crop jobs [qn] (g6d_warp_affine_u8), frame i at
 * frames + i*rows*cols*3 */
int g6d_glue_detection_jobs(const float* det_out, const uint8_t* frames, int rows, int cols, int qn, int size,
                            g6d_warp_job* jobs, g6d_stream_t stream);
int g6d_glue_detection_jobs_host(const float* det_out, const uint8_t* frames, int rows, int cols, int qn, int size,
                                 g6d_warp_job* jobs);
/* detection + selection (sel_idx [qn] int64, sel_out [qn,2] = angle, logit; g6d_sel_parse) -> poses float64 [qn,12] */
int g6d_glue_initial_poses(const float* det_out, const long long* sel_idx, const float* sel_out, const g6d_glue_refs* refs,
                           const g6d_glue_camera* cams, int qn, double* poses, g6d_stream_t stream);
int g6d_glue_initial_poses_host(const float* det_out, const long long* sel_idx, const float* sel_out, const g6d_glue_refs* refs,
                                const g6d_glue_camera* cams, int qn, double* poses);
/* poses [qn,12] (float64 storage; poses_are_f32: the values are float32 poses, as after a refinement) -> everything one
 * refinement stage reads: jobs [qn*(ref_num+1)] (query crop, then its views; g6d_warp_perspective_u8), que_K [qn,9],
 * que_pose [qn,12], rect [qn,12], ref_Ks [qn,ref_num,9], ref_poses [qn,ref_num,12] (float32), ref_rows [qn,ref_num] */
int g6d_glue_refine_problems(const g6d_glue_views* views, const g6d_glue_camera* cams, const uint8_t* frames, int rows, int cols,
                             const double* poses, int poses_are_f32, int qn, g6d_warp_job* jobs, float* que_K, float* que_pose,
                             float* rect, float* ref_Ks, float* ref_poses, int* ref_rows, g6d_stream_t stream);
int g6d_glue_refine_problems_host(const g6d_glue_views* views, const g6d_glue_camera* cams, const uint8_t* frames, int rows,
                                  int cols, const double* poses, int poses_are_f32, int qn, g6d_warp_job* jobs, float* que_K,
                                  float* que_pose, float* rect, float* ref_Ks, float* ref_poses, int* ref_rows);
/* network output [qn,7] (quaternion, offset, log2 scale) -> refined poses (float32 values in float64 storage) */
int g6d_glue_apply_refinements(const g6d_glue_views* views, const float* que_pose, const float* que_K, const float* rect,
                               const float* net_out, int qn, double* poses, g6d_stream_t stream);
int g6d_glue_apply_refinements_host(const g6d_glue_views* views, const float* que_pose, const float* que_K, const float* rect,
                                    const float* net_out, int qn, double* poses);

/* ---- pose smoothing of a tracked video (predict.py:18-26, 63-71; utils/base_utils.py:256-265 project_points;
 * utils/pose_utils.py:246-279 pnp).  One thread per lane (lanes <= 64): project the 8 box corners bbox [8,3] with the
 * lane's pose (float64 storage of float32 values) and cams[lane].K in float32, push them into the lane's history ring
 * hist [lanes,num,8,2] (float32) at slot count[lane] % num and increment count[lane], average the last min(count, num)
 * entries with weights[num - n .. num) / wsum[n - 1] in float64, and solve SOLVEPNP_ITERATIVE (non-coplanar DLT + LM,
 * float64) for the averaged points.  weights [num] = exp(-(arange(num) / std) ** 2)[::-1] and wsum[n - 1] = the numpy
 * sum of its last n entries, both from the caller.  Outputs: corners [lanes,8,2] float32, wpts [lanes,8,2] float64,
 * smoothed [lanes,12] float64 [R | t]. */
int g6d_track_smooth(const float* bbox, const double* poses, const g6d_glue_camera* cams, const double* weights, const double* wsum,
                     int lanes, int num, float* hist, int* count, float* corners, double* wpts, double* smoothed, g6d_stream_t stream);
int g6d_track_smooth_host(const float* bbox, const double* poses, const g6d_glue_camera* cams, const double* weights, const double* wsum,
                          int lanes, int num, float* hist, int* count, float* corners, double* wpts, double* smoothed);
/* (x - mean) / std on f32 [n_pixels, in_c] -> [n_pixels, out_c] (in_c, out_c in {3,4})
 * (network/detector.py:189, selector.py:115, refiner.py:65) */
int g6d_imagenet_norm(const float* in, float* out, long long n_pixels, int in_c, int out_c, g6d_stream_t stream);
/* NCHW [N,C,H,W] -> channels-last [N,H,W,out_c] (channels >= C zero) and back */
int g6d_nchw_to_nhwc(const float* in, float* out, int N, int C, int H, int W, int out_c, g6d_stream_t stream);
int g6d_nhwc_to_nchw(const float* in, float* out, int N, int C, int H, int W, int in_c, g6d_stream_t stream);
/* F.interpolate(mode='bilinear', align_corners=False) on channels-last data
 * (network/detector.py:240,243; network/refiner.py:75-76).  Output rows have `out_cstride`
 * channels and the C results land at channel offset `out_coff` (writes into concat buffers). */
int g6d_resize_bilinear(const float* in, float* out, int N, int Hi, int Wi, int Ho, int Wo, int C,
                        int out_cstride, int out_coff, g6d_stream_t stream);
/* F.interpolate default (nearest): src = floor(dst * in / out) (network/detector.py:201) */
int g6d_resize_nearest(const float* in, float* out, int N, int Hi, int Wi, int Ho, int Wo, int C, g6d_stream_t stream);
/* MaxPool 2x2 stride 2 over (H, W), output floor(H/2) x floor(W/2) like torch (VGG M layers;
 * selector MaxPool3d((1,2,2))) */
int g6d_maxpool2x2(const float* in, float* out, int N, int H, int W, int C, g6d_stream_t stream);
/* F.normalize(dim=1) == x / max(||x||_2, eps) over the channel axis of each row
 * (network/selector.py:118, network/refiner.py:69-71) */
int g6d_l2norm_channels(const float* in, float* out, long long rows, int C, float eps, g6d_stream_t stream);
/* y = act(x * scale[g,c] + shift[g,c]); rows_per_group consecutive rows share a group.
 * act: 0 none, 1 ReLU.  Materialises an InstanceNorm (+ReLU) where a consumer needs it.
 * Input rows have `in_cstride` channels (C taken from offset in_coff); same for output. */
int g6d_affine_act(const float* in, float* out, long long rows, int C, long long rows_per_group,
                   const float* scale, const float* shift, int act,
                   int in_cstride, int in_coff, int out_cstride, int out_coff, g6d_stream_t stream);
/* mean over `spatial` consecutive rows of act(x*scale+shift) -> [groups_of_rows, C]
 * (AvgPool3d((1,4,4)) of network/selector.py:76 applied after the fused IN+ReLU). */
int g6d_avgpool_affine(const float* in, float* out, long long n_out, int spatial, int C, long long rows_per_group,
                       const float* scale, const float* shift, int act, g6d_stream_t stream);
int g6d_add(const float* a, const float* b, float* out, long long n, g6d_stream_t stream);

/* ------------------------------------------------------------------ instance-norm stats ---- */
/* InstanceNorm{1,2,3}d(affine=False, eps) statistics (biased variance) of a channels-last
 * tensor: `rows` rows of C channels (taken at channel offset `coff` of rows `cstride` wide),
 * `rows_per_group` consecutive rows form one (sample, *) group.  Writes scale = rstd and
 * shift = -mean*rstd, each [groups, C], for consumption by prologues / g6d_affine_act.
 * ws: 2*groups*C doubles of workspace.  (network/selector.py:27-87, refiner.py:18-22,82-86) */
int g6d_instnorm_stats(const float* x, long long rows, int C, int cstride, int coff, long long rows_per_group,
                       float eps, float* scale, float* shift, double* ws, g6d_stream_t stream);

/* The two halves of g6d_instnorm_stats, for statistics that span GPUs (reference-sharded selector):
 * partial writes ws[g,c] = (sum, sum of squares) as doubles; the caller all-reduces ws across ranks;
 * finalize turns it into scale/shift with `count` = total rows per group over all ranks. */
int g6d_instnorm_partial(const float* x, long long rows, int C, int cstride, int coff, long long rows_per_group,
                         double* ws, g6d_stream_t stream);
int g6d_instnorm_finalize(const double* ws, long long groups, int C, long long count, float eps, float* scale,
                          float* shift, g6d_stream_t stream);

/* ------------------------------------------------------------------ convolution ------------ */
typedef struct g6d_conv_desc {
    int B, D, H, W, Cin;      /* input [B,D,H,W,*]; channels [in_coff, in_coff+Cin) of rows in_cstride wide */
    int in_cstride, in_coff;
    int Cout, kd, kh, kw;
    int stride;               /* same in all spatial dims that have k>1 */
    int pd, ph, pw;           /* zero padding */
    int Do, Ho, Wo;           /* output dims (validated) */
    int out_cstride, out_coff;
    int prologue;             /* G6D_PRO_* applied to in-bounds input elements before the MAC */
    long long group_rows;     /* prologue group of output item b: g = b / group_rows */
    int act;                  /* G6D_ACT_* epilogue after bias */
    int max_chain_k;          /* tensor-core path: 0 = default; > 0 bounds the K-elements accumulated into one TMEM
                                 accumulator (longer problems are split and summed in fp32 round-to-nearest).  The tensor
                                 core truncates on every accumulate, which biases long chains of SAME-SIGN products
                                 (detector correlation: post-ReLU features x post-ReLU features) by ~5e-8 per step. */
    int in_items;             /* input items: 0 = B (item b reads input item b); else a divisor of B and output item b
                                 reads input item b % in_items (one stack broadcast to B / in_items groups: the batched
                                 selector's first tower convolution, qn queries against one reference stack) */
} g6d_conv_desc;

#define G6D_PRO_NONE 0
#define G6D_PRO_AFFINE 1        /* x*scale[g,c] + shift[g,c]          (folded InstanceNorm)        */
#define G6D_PRO_AFFINE_RELU 2   /* relu(x*scale[g,c] + shift[g,c])    (folded InstanceNorm + ReLU) */
#define G6D_PRO_CORR 3          /* x*scale[g,pos,c] + shift[g,c] (scale [groups, D*H*W, Cin], shift [groups, Cin]):
                                   selector correlation volume q_g (.) ref with the first InstanceNorm3d folded in */
#define G6D_ACT_NONE 0
#define G6D_ACT_RELU 1
#define G6D_ACT_LEAKY01 2

/* Implicit-GEMM convolution (1x1 ... 3x3x3, stride 1/2) with fused prologue/bias/activation.
 * Replaces F.conv2d / Conv3d call sites: VGG (pretrain_models.py:17-31), detector correlation
 * (detector.py:222-224, reference features as kernels) and heads (:159-184), selector towers
 * (selector.py:27-77) and 1x1 convs (:79-111), refiner feature/volume nets (refiner.py:24-52,
 * 88-134).  w: packed [K, Cout]; bias may be NULL.  ws: split-K workspace of
 * g6d_conv_workspace_bytes(desc) bytes (may be NULL when that returns 0). */
int g6d_conv(const g6d_conv_desc* desc, const float* x, const float* w, const float* bias,
             const float* pro_scale, const float* pro_shift, float* y, void* ws, g6d_stream_t stream);
long long g6d_conv_workspace_bytes(const g6d_conv_desc* desc);
/* First VGG block in one kernel: 3x3 conv 4 -> 64 (RGB + zero channel, BN folded) + ReLU + 2x2 max-pool
 * (network/pretrain_models.py:17-31 features[0:4]); x [B,H,W,4], w packed [36,64] (g6d_pack_conv_weight),
 * y [B,H/2,W/2,64]; H, W even.  Bit-identical to g6d_conv -> ReLU -> g6d_maxpool2x2. */
int g6d_vgg_first_block(const float* x, const float* w, const float* bias, float* y, int B, int H, int W,
                        g6d_stream_t stream);
/* [Cout, Cin, kd, kh, kw] (reference layout) -> [taps*Cin_pad, ldw] with ldw = Cout rounded up
 * to 4; channels [Cin, Cin_pad) and columns [Cout, ldw) are zero; optional per-Cout scale
 * (eval-mode BatchNorm fold). */
int g6d_pack_conv_weight(const float* w, float* out, int Cout, int Cin, int Cin_pad, int taps,
                         const float* cout_scale, g6d_stream_t stream);
/* ---- tensor-core path (tcgen05, three-term operand split: fp32-faithful on the tensor pipe) ------
 * Same contract as g6d_conv, for problems g6d_conv_tc_supported accepts (Cin a multiple of the
 * kind's K-block, Cout >= 16).  A*B ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi with 11-bit-significand
 * halves; `kind` selects their container:
 *   G6D_TC_TF32: hi = tf32(x), lo = tf32(x - hi), fp32 arrays, K-block 32, tcgen05.mma kind::tf32;
 *   G6D_TC_F16 : hi = fp16(x), lo = fp16((x - hi) * 2^11), __half arrays, K-block 64, kind::f16 (twice
 *                the K per instruction and per operand byte; the kernels undo the 2^11 in the epilogue).
 *                Range contract: |x| <= 65504 (saturating), full accuracy for |x| >= 6.1e-5.
 * Weights are pre-split [w_rows >= Cout, K] K-major arrays (K = tap*Cin + c), see
 * g6d_pack_conv_weight_tc / g6d_split_operand.  A tiles are gathered + transformed + split by
 * producer warps, B tiles arrive by TMA, accumulators live in TMEM. */
#define G6D_TC_TF32 0
#define G6D_TC_F16 1
int g6d_conv_tc_supported(const g6d_conv_desc* desc, int kind);
/* debug probe: D[128x32] = A[shift..shift+128) x I for a row-shifted SWIZZLE_128B descriptor (mode: base_offset rule) */
int g6d_debug_umma_shift(float* out, int shift, int mode, g6d_stream_t stream);
/* debug: host_out8[0] != 0 if a pipeline wait inside g6d_conv_tc timed out (kernel bailed out); syncs */
int g6d_conv_tc_debug(int* host_out8);
long long g6d_conv_tc_workspace_bytes(const g6d_conv_desc* desc, int kind);
/* stats (optional, may be NULL): fused InstanceNorm statistics of the OUTPUT.  [M / stats_rows, Cout, 2] doubles
 * receive, per group of stats_rows consecutive output rows and channel, (sum y, sum y^2) -- what
 * g6d_instnorm_partial computes in a separate pass over y; feed them to g6d_instnorm_finalize.  Zeroed by
 * the call.  Allowed when g6d_conv_tc_stats_supported (groups made of whole 32-row slices / image planes). */
int g6d_conv_tc_stats_supported(const g6d_conv_desc* desc, int kind, long long stats_rows);
int g6d_conv_tc(const g6d_conv_desc* desc, const float* x, const void* w_hi, const void* w_lo, int w_rows, int kind,
                const float* bias, const float* pro_scale, const float* pro_shift, float* y, void* ws,
                double* stats, long long stats_rows, g6d_stream_t stream);
/* [Cout, Cin, taps] (reference layout) -> hi/lo [rows_pad, taps*Cin_pad] of the given kind; optional BN-fold scale */
int g6d_pack_conv_weight_tc(const float* w, void* out_hi, void* out_lo, int Cout, int Cin, int Cin_pad, int taps,
                            int rows_pad, const float* cout_scale, int kind, g6d_stream_t stream);
/* hi/lo split of a K-major fp32 operand [rows, K] into the given kind (detector reference features as
 * kernels).  G6D_TC_F16 operands use the kernels' K order inside every 64-element block (position p holds
 * source element 4*(p/8) + p%8 for p%8 < 4, else 32 + 4*(p/8) + p%8 - 4: it keeps the activation gathers
 * coalesced); K % 64 == 0.  g6d_pack_conv_weight_tc applies the same order. */
int g6d_split_operand(const float* in, void* hi, void* lo, long long n, int kind, g6d_stream_t stream);
/* [rows, K] row-major -> [K, rows] (detector reference features [rfn,k,k,512] -> correlation kernels) */
int g6d_transpose2d(const float* in, float* out, int rows, int cols, g6d_stream_t stream);
/* y[m, n] = act(sum_k x[m,k] w[n,k] + b[n]) for small m (<= 8): weight-bandwidth bound
 * (refiner regressor fc 32768->512, refiner.py:156-159).  w is [N, K] row-major. */
int g6d_linear_smallm(const float* x, const float* w, const float* bias, float* y, int M, int N, int K, int act,
                      g6d_stream_t stream);

/* ------------------------------------------------------------------ detector ---------------- */
#define G6D_DET_MAX_SCALES 8
typedef struct g6d_det_maps {
    int n_scales;
    int rfn, hs, ws;                 /* output resolution (h/8, w/8) */
    const float* map[G6D_DET_MAX_SCALES][3]; /* raw correlation [qn, Hl, Wl, rfn], level l = 0,1,2 */
    int H[G6D_DET_MAX_SCALES][3];
    int W[G6D_DET_MAX_SCALES][3];
    float mu[3], inv_sigma[3], clip; /* vgg_score_stats / vgg_score_max */
} g6d_det_maps;
/* Fuses detector.py:225-226 (nearest x2/x4), :207-216 (normalise + clip), :243 (bilinear resize
 * to (hs,ws)), :245 (stack), :246 score_conv (1x1x1 Conv3d 3S->64, ReLU, 64->64) and :247 (max
 * over references).  w1 [64, 3S] (channel = scale*3 + level), w2 [64, 64].  out [qn, hs, ws, 64]. */
int g6d_det_score_fuse(const g6d_det_maps* host_maps, int qn, const float* w1, const float* b1,
                       const float* w2, const float* b2, float* out, g6d_stream_t stream);
/* Row-decomposed form of the sliding inner product of detector.py:222-224: with the reference features
 * [rfn, k, k, C] packed as a 1 x k convolution of k*rfn output channels (channel = ky*rfn + r, zero
 * padding k/2 in both axes, so the result has H + k - 1 rows), partial [qn, H+k-1, W, k*rfn] holds the
 * contribution of kernel row ky to input row y'; out[q,y,x,r] = sum_ky partial[q, y+ky, x, ky*rfn + r]
 * is the k x k correlation map [qn, H, W, rfn].  rfn % 4 == 0. */
int g6d_det_corr_rowsum(const float* partial, float* out, int qn, int H, int W, int k, int rfn, g6d_stream_t stream);
/* detector.py:85-121: first-max flat argmax of scores [qn,hs,ws,1], then
 * position = ((x,y) + offset[y,x] + 0.5)*pool - 0.5, scale = 2**scale[y,x].
 * out [qn, 4] = (x, y, scale, score); out_idx [qn] (int64 flat index y*ws + x). */
int g6d_det_parse(const float* scores, const float* scales, const float* offsets, int qn, int hs, int ws,
                  int pool_ratio, float* out, long long* out_idx, g6d_stream_t stream);

/* ------------------------------------------------------------------ selector ---------------- */
/* Load-time sums over the reference stack ref [S, P, C]: sum_s ref and sum_s ref^2, as doubles
 * [P, C] each.  They give the first InstanceNorm3d's statistics of the correlation volume in
 * closed form at query time (SURVEY.md 8a S2 note). */
int g6d_sel_ref_sums(const float* ref, int S, int P, int C, double* sum1, double* sum2, g6d_stream_t stream);
/* From the qn queries q [qn, P, C] and the sums: scale[g,p,c] = q[g,p,c]*rstd_gc, shift[g,c] = -mean_gc*rstd_gc,
 * the G6D_PRO_CORR prologue operands of the first tower conv (selector.py:28,49,63 InstanceNorm3d over (S,h,w)
 * of que*ref), one launch for all queries. */
int g6d_sel_corr_prologue(const float* q, const double* sum1, const double* sum2, int S, int P, int C, int qn, float eps,
                          float* scale, float* shift, g6d_stream_t stream);
/* The rotated-similarity score, selector.py:183-186,192-194: s[p] = sum_c q[p,c]*ref[s,p,c];
 * score[s] = sum_p s[p]^2 / max_p s[p].  ref [S, P, C] is streamed once from HBM. */
int g6d_sel_corr_score(const float* ref, const float* q, int S, int P, int C, float* score, g6d_stream_t stream);
/* The same score for the three pyramid levels and qn queries in one streaming pass (what select_que_imgs
 * uses): q_l [qn, P_l, C], score [qn, 3, S]; every reference row is read once and dotted with all qn query
 * rows (each query's score is bit-identical to a one-query call).  ws: g6d_sel_corr_score3_workspace_bytes(S,
 * P0, P1, P2, qn) bytes (per-location inner products, L2-resident).  counters: 3*qn*S ints, one per (query,
 * level, slice), ZERO on entry and left zero on exit (allocate + clear once, reuse for every call on the same
 * stream): the CTA that completes the last location of a slice reduces it, so the whole op is one launch.
 * counters == NULL: two launches. */
long long g6d_sel_corr_score3_workspace_bytes(int S, int P0, int P1, int P2, int qn);
int g6d_sel_corr_score3(const float* ref0, const float* ref1, const float* ref2, const float* q0, const float* q1,
                        const float* q2, int S, int P0, int P1, int P2, int C, int qn, float* score, float* ws, int* counters,
                        g6d_stream_t stream);
/* vp_norm (InstanceNorm2d(3), selector.py:78,201) for `groups` queries: normalise each of the L score rows of
 * score [groups, L, n] (biased var, eps) and scatter into feats[groups * n, cstride] at row g*n + i, channel coff + l. */
/* (channels [coff + L, cstride) of every feats row -- padding that the consumer multiplies by zero weights -- are set to 0) */
int g6d_sel_vp_norm(const float* score, int groups, int L, int n, float eps, float* feats, int cstride, int coff,
                    g6d_stream_t stream);
/* selector.py:203-204 for `groups` queries: out[g*rfn + r, c] = max_a x[g*rfn + r, a, c] + embed[r, c] */
int g6d_sel_max_angle_add(const float* x, const float* embed, float* out, int groups, int rfn, int an, int C,
                          g6d_stream_t stream);
/* attention.py:4-17 with the reference's channel->(d, head) mapping c = d*heads + head, over `groups`
 * independent sets of n tokens: q,k,v [groups * n, C] -> out [groups * n, C]; softmax(q_h^T k_h / sqrt(C/heads))
 * over the keys of the token's own group. n <= 8192. */
int g6d_attention(const float* q, const float* k, const float* v, float* out, int groups, int n, int C, int heads,
                  g6d_stream_t stream);
/* The same attention over HEAD-MAJOR channels (c = head*64 + d): the layout a caller gets for free by
 * permuting the output rows of conv_query / conv_key / conv_feats (and the input columns of conv_merge)
 * once at pack time.  Tiled (8 queries x 1 head per block, K / V tiles staged in shared memory by coalesced
 * loads): what the selector uses, and what keeps the replicated tail of a reference-sharded selector
 * (n = all references over all GPUs) cheap.  n <= 2048, C = heads * 64. */
int g6d_attention_headmajor(const float* q, const float* k, const float* v, float* out, int groups, int n, int C,
                            int heads, g6d_stream_t stream);
/* nn.LayerNorm(C) over the channel axis of each row (attention.py:19-26) */
int g6d_layernorm(const float* x, const float* gamma, const float* beta, float* out, int rows, int C, float eps,
                  g6d_stream_t stream);
/* selector.py:172-175: idx = first argmax of logits [qn, rfn]; out [qn,2] = (angle[idx], logit[idx]) */
int g6d_sel_parse(const float* logits, const float* angles, int qn, int rfn, long long* out_idx, float* out,
                  g6d_stream_t stream);

/* ------------------------------------------------------------------ refiner ----------------- */
/* refiner.py:183-247 + operator.py:4-17: for every voxel of the sn^3 unit-cube grid rotated by
 * the input pose (row vector @ R_in, R_in = que_poses[:, :3, :3]), project into each of the R
 * reference views and the query view (P = K @ pose), bilinear-sample (zeros padding,
 * align_corners=False) the C-channel feature maps, and write mean / unbiased std over the
 * references and the query sample.
 *   ref_feats [Q, R, fh, fw, C], que_feats [Q, fh, fw, C]
 *   ref_Ks [Q, R, 3, 3], ref_poses [Q, R, 3, 4], que_Ks [Q, 3, 3], que_poses [Q, 3, 4]
 *   mean_in [Q, sn^3, 2C]: channels [0,C) mean, [C,2C) query sample;  stdv [Q, sn^3, C]
 * img_h/img_w: the image size the projections refer to (128), NOT the feature size. */
int g6d_ref_volume_fill(const float* ref_feats, const float* que_feats, const float* ref_Ks,
                        const float* ref_poses, const float* que_Ks, const float* que_poses, int Q, int R,
                        int fh, int fw, int C, int sn, int img_h, int img_w, float* mean_in, float* stdv,
                        g6d_stream_t stream);
/* refiner.py:161-166 tail: r = normalize(x Wr^T + br) (4), t (2), s (1) from x [M,512];
 * w [7, K] rows = fcr(4), fct(2), fcs(1).  out [M, 7] = (qw,qx,qy,qz, tx,ty, log2 scale). */
int g6d_ref_pose_heads(const float* x, const float* w, const float* b, float* out, int M, int K, g6d_stream_t stream);

/* ------------------------------------------------------------------ evaluation (row f4) ---- */
/* utils/pose_utils.py:149-158,192-196 (compute_pose_errors / the symmetric branch of
 * compute_metrics_impl) with utils/base_utils.py:256-265 project_points and :390-394: for each of
 * n_poses (predicted, ground-truth) pairs, out[p] = (mean reprojection error in pixels, mean 3-D
 * point error = ADD, mean closest-point error = ADD-S or NaN when symmetric == 0) over the n_pts
 * object points.  pts [n_pts,3], poses [n_poses,3,4], Ks [n_poses,3,3], out [n_poses,3], all f32 on
 * the device; ws: g6d_pose_errors_workspace_bytes(n_pts, n_poses) bytes. */
long long g6d_pose_errors_workspace_bytes(int n_pts, int n_poses);
int g6d_pose_errors(const float* pts, int n_pts, const float* poses_pr, const float* poses_gt, const float* Ks,
                    int n_poses, int symmetric, float* out, void* ws, g6d_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GEN6D_B200_H */
