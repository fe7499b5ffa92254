"""Torch-tensor front end of the C ABI.

PyTorch is used here only as the device-memory allocator and stream provider: every function
checks its tensors (CUDA, contiguous, dtype), takes raw pointers and calls into
libgen6d_b200.so on torch's current stream.  Activations are fp32 channels-last.
"""
import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import ACT_LEAKY01, ACT_NONE, ACT_RELU, PRO_AFFINE, PRO_AFFINE_RELU, PRO_CORR, PRO_NONE  # noqa: F401


WARP_JOB_BYTES = 88   # sizeof(g6d_warp_job)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t, dtype=torch.float32):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise ValueError(f'expected a contiguous CUDA {dtype} tensor, got {t.dtype} {t.device} '
                         f'contiguous={t.is_contiguous()} shape={tuple(t.shape)}')
    return C.c_void_p(t.data_ptr())


_PROFILE = None   # when enabled: {name: [(start_event, end_event, work), ...]}


def _call(name, *args, work=None, tag=None):
    if _PROFILE is not None and work is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(getattr(_lib.lib(), name)(*args), name)
        e1.record()
        _PROFILE.setdefault(name, []).append((e0, e1, work))
        if tag is not None:
            _PROFILE.setdefault('#calls', []).append((e0, e1, work, name, tag))
        return
    _lib.check(getattr(_lib.lib(), name)(*args), name)


def enable_profiling():
    """Time every launch of the roofline kernels with CUDA events on the launching stream
    (bench.py).  `work` is the algorithmic FLOPs (conv) or bytes (streaming kernels) of the call."""
    global _PROFILE
    _PROFILE = {}
    return _PROFILE


def collect_profile(prof):
    global _PROFILE
    torch.cuda.synchronize()
    _PROFILE = None
    out = {k: {'ms': sum(r[0].elapsed_time(r[1]) for r in v), 'work': float(sum(r[2] for r in v)), 'n': len(v)}
           for k, v in prof.items() if k != '#calls'}
    if '#calls' in prof:
        out['#calls'] = [(r[0].elapsed_time(r[1]), r[2], r[3], r[4]) for r in prof['#calls']]
    return out


def require_cuda():
    if not torch.cuda.is_available():
        raise _lib.Gen6DLibraryError('no CUDA device: the Gen6D hot path has no CPU fallback')
    _lib.lib()


# ------------------------------------------------------------------------------- layout / images
def preprocess_u8(img, out_c=4, imagenet_norm=True):
    """u8 [..., H, W, 3] -> f32 [..., H, W, out_c]: /255 (+ ImageNet normalisation)."""
    out = torch.empty(*img.shape[:-1], out_c, device=img.device, dtype=torch.float32)
    _call('g6d_preprocess_u8', _p(img, torch.uint8), _p(out), img.numel() // 3, out_c, int(imagenet_norm), _stream())
    return out


def _warp(name, jobs, n_jobs, h, w):
    if jobs.dtype != torch.uint8 or jobs.numel() != n_jobs * WARP_JOB_BYTES:
        raise ValueError(f'{name}: jobs must be the packed bytes of {n_jobs} g6d_warp_job records')
    out = torch.empty(n_jobs, h, w, 3, device=jobs.device, dtype=torch.uint8)
    _call(name, _p(jobs, torch.uint8), n_jobs, _p(out, torch.uint8), h, w, _stream())
    return out


def warp_perspective_u8(jobs, n_jobs, h, w):
    """cv2.warpPerspective (u8, INTER_LINEAR, zero border), bit-exact, for n_jobs (image, H) pairs.
    jobs: device uint8 tensor holding n_jobs packed g6d_warp_job records (geometry.pack_warp_jobs)."""
    return _warp('g6d_warp_perspective_u8', jobs, n_jobs, h, w)


def warp_affine_u8(jobs, n_jobs, h, w):
    """cv2.warpAffine counterpart of warp_perspective_u8."""
    return _warp('g6d_warp_affine_u8', jobs, n_jobs, h, w)


# ------------------------------------------------------------------------------- camera algebra between the stages
def glue_detection_jobs(det_out, frames, size):
    """det_out [qn,4] (g6d_det_parse) + frames u8 [qn,h,w,3] -> packed g6d_warp_job records [qn*88] of the selector crops."""
    qn, h, w, _ = frames.shape
    jobs = torch.empty(qn * WARP_JOB_BYTES, device=frames.device, dtype=torch.uint8)
    _call('g6d_glue_detection_jobs', _p(det_out), _p(frames, torch.uint8), h, w, qn, size, _p(jobs, torch.uint8), _stream())
    return jobs


def glue_initial_poses(det_out, sel_idx, sel_out, refs_struct, cams):
    """Detection + selection -> initial poses float64 [qn,12] (geometry.poses_from_similarity on the device)."""
    qn = det_out.shape[0]
    poses = torch.empty(qn, 12, device=det_out.device, dtype=torch.float64)
    _call('g6d_glue_initial_poses', _p(det_out), _p(sel_idx, torch.int64), _p(sel_out), C.byref(refs_struct), _p(cams, torch.float64),
          qn, _p(poses, torch.float64), _stream())
    return poses


def glue_refine_problems(views_struct, ref_num, cams, frames, poses, poses_are_f32):
    """poses float64 [qn,12] -> (jobs u8 [qn*(ref_num+1)*88], que_K [qn,3,3], que_pose [qn,3,4], rect [qn,3,4],
    ref_Ks [qn,R,3,3], ref_poses [qn,R,3,4], ref_rows i32 [qn,R]): geometry.refine_problems on the device."""
    qn, h, w, _ = frames.shape
    dev, f32 = frames.device, torch.float32
    jobs = torch.empty(qn * (ref_num + 1) * WARP_JOB_BYTES, device=dev, dtype=torch.uint8)
    que_K, que_pose, rect = torch.empty(qn, 3, 3, device=dev, dtype=f32), torch.empty(qn, 3, 4, device=dev, dtype=f32), \
        torch.empty(qn, 3, 4, device=dev, dtype=f32)
    ref_Ks, ref_poses = torch.empty(qn, ref_num, 3, 3, device=dev, dtype=f32), torch.empty(qn, ref_num, 3, 4, device=dev, dtype=f32)
    rows = torch.empty(qn, ref_num, device=dev, dtype=torch.int32)
    _call('g6d_glue_refine_problems', C.byref(views_struct), _p(cams, torch.float64), _p(frames, torch.uint8), h, w,
          _p(poses, torch.float64), int(poses_are_f32), qn, _p(jobs, torch.uint8), _p(que_K), _p(que_pose), _p(rect), _p(ref_Ks),
          _p(ref_poses), _p(rows, torch.int32), _stream())
    return jobs, que_K, que_pose, rect, ref_Ks, ref_poses, rows


def glue_apply_refinements(views_struct, que_pose, que_K, rect, net_out):
    """Network output [qn,7] -> refined poses (float32 values) float64 [qn,12]: geometry.apply_refinements on the device."""
    qn = net_out.shape[0]
    poses = torch.empty(qn, 12, device=net_out.device, dtype=torch.float64)
    _call('g6d_glue_apply_refinements', C.byref(views_struct), _p(que_pose), _p(que_K), _p(rect), _p(net_out), qn,
          _p(poses, torch.float64), _stream())
    return poses


def track_smooth(bbox, poses, cams, weights, wsum, hist, count):
    """One tracked frame of pose smoothing per lane (csrc/track.cu): bbox f32 [8,3], poses f64 [M,12], cams f64 [M,20],
    weights / wsum f64 [num] (glue.smoothing_weights), history ring hist f32 [M,num,8,2] and count i32 [M] (updated in
    place) -> (corners f32 [M,8,2], averaged corners f64 [M,8,2], smoothed poses f64 [M,12])."""
    M, num = poses.shape[0], weights.shape[0]
    corners = torch.empty(M, 8, 2, device=poses.device, dtype=torch.float32)
    wpts = torch.empty(M, 8, 2, device=poses.device, dtype=torch.float64)
    smoothed = torch.empty(M, 12, device=poses.device, dtype=torch.float64)
    _call('g6d_track_smooth', _p(bbox), _p(poses, torch.float64), _p(cams, torch.float64), _p(weights, torch.float64),
          _p(wsum, torch.float64), M, num, _p(hist), _p(count, torch.int32), _p(corners), _p(wpts, torch.float64),
          _p(smoothed, torch.float64), _stream())
    return corners, wpts, smoothed


def imagenet_norm(x, out_c=4):
    out = torch.empty(*x.shape[:-1], out_c, device=x.device, dtype=torch.float32)
    _call('g6d_imagenet_norm', _p(x), _p(out), x.numel() // x.shape[-1], x.shape[-1], out_c, _stream())
    return out


def nchw_to_nhwc(x, out_c=None):
    N, Cc, H, W = x.shape
    out_c = out_c or Cc
    out = torch.empty(N, H, W, out_c, device=x.device, dtype=torch.float32)
    _call('g6d_nchw_to_nhwc', _p(x), _p(out), N, Cc, H, W, out_c, _stream())
    return out


def nhwc_to_nchw(x, channels=None):
    N, H, W, cs = x.shape
    Cc = channels or cs
    out = torch.empty(N, Cc, H, W, device=x.device, dtype=torch.float32)
    _call('g6d_nhwc_to_nchw', _p(x), _p(out), N, Cc, H, W, cs, _stream())
    return out


def resize_bilinear(x, Ho, Wo, out=None, out_coff=0):
    N, Hi, Wi, Cc = x.shape
    if out is None:
        out = torch.empty(N, Ho, Wo, Cc, device=x.device, dtype=torch.float32)
    _call('g6d_resize_bilinear', _p(x), _p(out), N, Hi, Wi, Ho, Wo, Cc, out.shape[-1], out_coff, _stream())
    return out


def resize_nearest(x, Ho, Wo):
    N, Hi, Wi, Cc = x.shape
    out = torch.empty(N, Ho, Wo, Cc, device=x.device, dtype=torch.float32)
    _call('g6d_resize_nearest', _p(x), _p(out), N, Hi, Wi, Ho, Wo, Cc, _stream())
    return out


def maxpool2x2(x):
    N, H, W, Cc = x.shape
    out = torch.empty(N, H // 2, W // 2, Cc, device=x.device, dtype=torch.float32)
    _call('g6d_maxpool2x2', _p(x), _p(out), N, H, W, Cc, _stream())
    return out


def l2norm_channels(x, eps=1e-12):
    out = torch.empty_like(x)
    _call('g6d_l2norm_channels', _p(x), _p(out), x.numel() // x.shape[-1], x.shape[-1], eps, _stream())
    return out


def instnorm_stats(x, rows_per_group, channels=None, coff=0, eps=1e-5):
    """x [..., cstride]; statistics over groups of `rows_per_group` consecutive rows.
    Returns (scale, shift), each [groups, C]: InstanceNorm(x) == x*scale + shift."""
    cstride = x.shape[-1]
    Cc = channels or cstride
    rows = x.numel() // cstride
    groups = rows // rows_per_group
    scale = torch.empty(groups, Cc, device=x.device, dtype=torch.float32)
    shift = torch.empty_like(scale)
    ws = torch.empty(groups * Cc * 2, device=x.device, dtype=torch.float64)
    _call('g6d_instnorm_stats', _p(x), rows, Cc, cstride, coff, rows_per_group, eps, _p(scale), _p(shift),
          _p(ws, torch.float64), _stream())
    return scale, shift


def instnorm_partial(x, rows_per_group, channels=None, coff=0):
    """Per (group, channel) (sum, sum of squares) as float64 [groups, C, 2] -- all-reducible across GPUs."""
    cstride = x.shape[-1]
    Cc = channels or cstride
    rows = x.numel() // cstride
    groups = rows // rows_per_group
    ws = torch.empty(groups, Cc, 2, device=x.device, dtype=torch.float64)
    _call('g6d_instnorm_partial', _p(x), rows, Cc, cstride, coff, rows_per_group, _p(ws, torch.float64), _stream())
    return ws


def instnorm_finalize(ws, count, eps=1e-5):
    """ws [groups, C, 2] (after any cross-rank reduction), count = rows per group over all ranks."""
    groups, Cc, _ = ws.shape
    scale = torch.empty(groups, Cc, device=ws.device, dtype=torch.float32)
    shift = torch.empty_like(scale)
    _call('g6d_instnorm_finalize', _p(ws, torch.float64), groups, Cc, count, eps, _p(scale), _p(shift), _stream())
    return scale, shift


def affine_act(x, scale, shift, rows_per_group, act=ACT_NONE, channels=None, in_coff=0, out=None, out_coff=0):
    ics = x.shape[-1]
    Cc = channels or ics
    rows = x.numel() // ics
    if out is None:
        out = torch.empty(*x.shape[:-1], Cc, device=x.device, dtype=torch.float32)
    _call('g6d_affine_act', _p(x), _p(out), rows, Cc, rows_per_group, _p(scale), _p(shift), act, ics, in_coff,
          out.shape[-1], out_coff, _stream())
    return out


def avgpool_affine(x, spatial, scale=None, shift=None, rows_per_group=1, act=ACT_NONE):
    """x [n_out*spatial, C] -> [n_out, C]: mean over `spatial` rows of act(x*scale+shift)."""
    Cc = x.shape[-1]
    n_out = x.numel() // Cc // spatial
    out = torch.empty(n_out, Cc, device=x.device, dtype=torch.float32)
    _call('g6d_avgpool_affine', _p(x), _p(out), n_out, spatial, Cc, rows_per_group, _p(scale), _p(shift), act, _stream())
    return out


def add(a, b):
    out = torch.empty_like(a)
    _call('g6d_add', _p(a), _p(b), _p(out), a.numel(), _stream())
    return out


# ------------------------------------------------------------------------------- convolution
@dataclass
class PackedConv:
    """Convolution weights in the library's [K, ldw] layout (+ bias), see g6d_pack_conv_weight."""
    w: Optional[torch.Tensor]   # FFMA layout (None for tensor-core-only operands)
    bias: Optional[torch.Tensor]
    cin: int          # padded input channels the packed weight expects
    cout: int
    k: tuple          # (kd, kh, kw)
    stride: int = 1
    pad: tuple = (0, 0, 0)
    w_hi: Optional[torch.Tensor] = None   # tensor-core path: [rows, K] hi / lo operand split (K-major)
    w_lo: Optional[torch.Tensor] = None
    kind: int = _lib.TC_TF32              # container of w_hi / w_lo: TC_TF32 (fp32 arrays) or TC_F16 (half arrays)
    rows: Optional[tuple] = None          # (k, rfn) of a row-decomposed detector correlation (see g6d_det_corr_rowsum)
    max_chain_k: int = 0                  # > 0: bound on the K-elements per tensor-core accumulate chain (same-sign operands)


def conv_path():
    """'tc' (tcgen05 split-operand kernels, default) or 'ffma' (fp32 CUDA-core fallback for A/B checks): env G6D_CONV_PATH."""
    return os.environ.get('G6D_CONV_PATH', 'tc')


def conv_kind():
    """Operand kind of the tensor-core path, env G6D_CONV_KIND: 'f16' (default; fp16 hi + 2^11-scaled fp16
    lo halves, kind::f16 MMAs: twice the K per instruction and per byte) or 'tf32' (tf32 halves: any fp32 range)."""
    return _lib.TC_TF32 if os.environ.get('G6D_CONV_KIND', 'f16') == 'tf32' else _lib.TC_F16


def tc_kind_for(cin_pad):
    """The kind a layer with `cin_pad` input channels is packed for (None: not tensor-core eligible)."""
    if cin_pad % 64 == 0 and conv_kind() == _lib.TC_F16:
        return _lib.TC_F16
    return _lib.TC_TF32 if cin_pad % 32 == 0 else None


def _tc_dtype(kind):
    return torch.float16 if kind == _lib.TC_F16 else torch.float32


def pack_conv(weight, bias=None, stride=1, pad=None, cin_pad=None, cout_scale=None, bias_override=None):
    """weight: reference layout [Cout, Cin, *k] (1-3 spatial dims) on the GPU."""
    cout, cin = weight.shape[:2]
    ks = tuple(weight.shape[2:])
    k3 = (1,) * (3 - len(ks)) + ks
    if pad is None:
        pad = tuple(kk // 2 for kk in k3)
    elif isinstance(pad, int):
        pad = tuple(pad if kk > 1 else 0 for kk in k3)
    else:
        pad = (0,) * (3 - len(pad)) + tuple(pad)
    cin_pad = cin_pad or ((cin + 3) // 4 * 4)
    taps = k3[0] * k3[1] * k3[2]
    ldw = (cout + 3) // 4 * 4
    w = weight.detach().to(torch.float32).contiguous()
    out = torch.empty(taps * cin_pad, ldw, device=w.device, dtype=torch.float32)
    _call('g6d_pack_conv_weight', _p(w), _p(out), cout, cin, cin_pad, taps,
          _p(cout_scale.contiguous()) if cout_scale is not None else None, _stream())
    b = bias_override if bias_override is not None else bias
    b = b.detach().to(torch.float32).contiguous() if b is not None else None
    pc = PackedConv(out, b, cin_pad, cout, k3, stride, pad)
    kind = tc_kind_for(cin_pad)
    if kind is not None and cout >= 16:
        rows = (cout + 7) // 8 * 8
        pc.kind = kind
        pc.w_hi = torch.empty(rows, taps * cin_pad, device=w.device, dtype=_tc_dtype(kind))
        pc.w_lo = torch.empty_like(pc.w_hi)
        _call('g6d_pack_conv_weight_tc', _p(w), _p(pc.w_hi, pc.w_hi.dtype), _p(pc.w_lo, pc.w_lo.dtype), cout, cin, cin_pad,
              taps, rows, _p(cout_scale.contiguous()) if cout_scale is not None else None, kind, _stream())
    return pc


def split_operand(x, kind=None):
    """fp32 [rows, K] -> (hi, lo, kind): the K-major B operand of the tensor-core path (detector
    reference features used as correlation kernels)."""
    kind = tc_kind_for(x.shape[-1]) if kind is None else kind
    hi = torch.empty(x.shape, device=x.device, dtype=_tc_dtype(kind))
    lo = torch.empty_like(hi)
    _call('g6d_split_operand', _p(x), _p(hi, hi.dtype), _p(lo, lo.dtype), x.numel(), kind, _stream())
    return hi, lo, kind


def transpose_to_packed(x2d):
    """[rows, K] -> packed [K, ldw(rows)] weights (detector reference features as kernels)."""
    rows, cols = x2d.shape
    out = torch.empty(cols, (rows + 3) // 4 * 4, device=x2d.device, dtype=torch.float32)
    _call('g6d_transpose2d', _p(x2d), _p(out), rows, cols, _stream())
    return out


def conv(x, pc, prologue=PRO_NONE, pro_scale=None, pro_shift=None, group_rows=1, act=ACT_NONE,
         in_coff=0, out=None, out_coff=0, stats_rows=None, batch=None):
    """x [B_in, D, H, W, cs] or [B_in, H, W, cs]; returns [B, Do, Ho, Wo, Cout] (or 4-D for 4-D input).
    batch: output items B (default B_in), a multiple of B_in: output item b reads input item b % B_in (one input
    stack broadcast to B / B_in prologue groups, e.g. PRO_CORR with scale [B / group_rows, H*W, C]).
    The prologue group of output item b is b // group_rows.
    stats_rows: also return the InstanceNorm moments of the OUTPUT, (y, ws) with ws float64
    [groups, Cout, 2] = per group of `stats_rows` consecutive output rows (sum y, sum y^2) -- fused into the
    convolution's epilogue on the tensor-core path (no extra pass over y), else by g6d_instnorm_partial;
    pass ws to instnorm_finalize (after any cross-GPU all-reduce)."""
    four = x.dim() == 4
    if four:
        B_in, H, W, cs = x.shape
        D = 1
    else:
        B_in, D, H, W, cs = x.shape
    B = batch or B_in
    if B % B_in:
        raise ValueError(f'conv: batch {B} is not a multiple of the input items {B_in}')
    kd, kh, kw = pc.k
    pd, ph, pw = pc.pad
    s = pc.stride
    Do, Ho, Wo = (D + 2 * pd - kd) // s + 1, (H + 2 * ph - kh) // s + 1, (W + 2 * pw - kw) // s + 1
    if out is None:
        shape = (B, Ho, Wo, pc.cout) if four else (B, Do, Ho, Wo, pc.cout)
        out = torch.empty(shape, device=x.device, dtype=torch.float32)
    d = _lib.ConvDesc(B=B, D=D, H=H, W=W, Cin=pc.cin, in_cstride=cs, in_coff=in_coff, Cout=pc.cout, kd=kd, kh=kh,
                      kw=kw, stride=s, pd=pd, ph=ph, pw=pw, Do=Do, Ho=Ho, Wo=Wo, out_cstride=out.shape[-1],
                      out_coff=out_coff, prologue=prologue, group_rows=group_rows, act=act, max_chain_k=pc.max_chain_k,
                      in_items=B_in if B != B_in else 0)
    work = 2.0 * B * Do * Ho * Wo * pc.cout * kd * kh * kw * pc.cin
    M = B * Do * Ho * Wo
    stats = None
    if pc.w_hi is not None and conv_path() == 'tc' and _lib.lib().g6d_conv_tc_supported(C.byref(d), pc.kind):
        nbytes = _lib.lib().g6d_conv_tc_workspace_bytes(C.byref(d), pc.kind)
        if nbytes < 0:
            _lib.check(-1, 'g6d_conv_tc_workspace_bytes')
        ws = torch.empty(nbytes // 4, device=x.device, dtype=torch.float32) if nbytes > 0 else None
        fuse = (stats_rows is not None and fused_stats_enabled() and
                _lib.lib().g6d_conv_tc_stats_supported(C.byref(d), pc.kind, stats_rows))
        if fuse:
            stats = torch.empty(M // stats_rows, pc.cout, 2, device=x.device, dtype=torch.float64)
        _call('g6d_conv_tc', C.byref(d), _p(x), _p(pc.w_hi, pc.w_hi.dtype), _p(pc.w_lo, pc.w_lo.dtype), pc.w_hi.shape[0],
              pc.kind, _p(pc.bias), _p(pro_scale), _p(pro_shift), _p(out), _p(ws), _p(stats, torch.float64), stats_rows or 0,
              _stream(), work=work,
              tag=f'M={M} N={pc.cout} K={kd * kh * kw * pc.cin} k={kd}x{kh}x{kw} s={s} pro={prologue}')
    else:
        if pc.w is None:
            raise _lib.Gen6DLibraryError('this operand was packed for the tensor-core path only and the problem is not supported there')
        nbytes = _lib.lib().g6d_conv_workspace_bytes(C.byref(d))
        if nbytes < 0:
            _lib.check(-1, 'g6d_conv_workspace_bytes')
        ws = torch.empty(nbytes // 4, device=x.device, dtype=torch.float32) if nbytes > 0 else None
        _call('g6d_conv', C.byref(d), _p(x), _p(pc.w), _p(pc.bias), _p(pro_scale), _p(pro_shift), _p(out), _p(ws), _stream(),
              work=work)
    if stats_rows is None:
        return out
    if stats is None:       # not fusable here (FFMA path, groups smaller than an epilogue slice): separate pass over the output
        stats = instnorm_partial(out, rows_per_group=stats_rows, channels=pc.cout, coff=out_coff)
    return out, stats


def fused_stats_enabled():
    """G6D_FUSED_STATS=0 computes every InstanceNorm statistic with the separate g6d_instnorm_partial pass (A/B checks)."""
    return os.environ.get('G6D_FUSED_STATS', '1') != '0'


def vgg_first_block(x, pc):
    """x [B,H,W,4] -> [B,H/2,W/2,64]: first VGG conv (BN folded) + ReLU + 2x2 max-pool in one kernel."""
    B, H, W, _ = x.shape
    out = torch.empty(B, H // 2, W // 2, 64, device=x.device, dtype=torch.float32)
    _call('g6d_vgg_first_block', _p(x), _p(pc.w), _p(pc.bias), _p(out), B, H, W, _stream())
    return out


def linear_smallm(x, w, bias, act=ACT_NONE):
    """x [M<=8, K], w [N, K] (row-major) -> [M, N]."""
    M, K = x.shape
    N = w.shape[0]
    out = torch.empty(M, N, device=x.device, dtype=torch.float32)
    _call('g6d_linear_smallm', _p(x), _p(w), _p(bias), _p(out), M, N, K, act, _stream())
    return out


# ------------------------------------------------------------------------------- detector
def det_score_fuse(maps, sizes, rfn, hs, ws, stats, clip, w1, b1, w2, b2, qn):
    """maps[s][l]: raw correlation [qn, Hl, Wl, rfn]; sizes[s][l] = (Hl, Wl). -> [qn, hs, ws, 64]."""
    m = _lib.DetMaps()
    m.n_scales, m.rfn, m.hs, m.ws = len(maps), rfn, hs, ws
    for s, lv in enumerate(maps):
        for l, t in enumerate(lv):
            m.map[s][l] = _p(t).value
            m.H[s][l], m.W[s][l] = sizes[s][l]
    for l in range(3):
        m.mu[l] = float(stats[l][0])
        m.inv_sigma[l] = 1.0 / float(stats[l][1])
    m.clip = float(clip)
    out = torch.empty(qn, hs, ws, 64, device=w1.device, dtype=torch.float32)
    _call('g6d_det_score_fuse', C.byref(m), qn, _p(w1), _p(b1), _p(w2), _p(b2), _p(out), _stream())
    return out


def det_corr_rowsum(partial, k, rfn):
    """partial [qn, H+k-1, W, k*rfn] (1 x k convolution, channel = ky*rfn + r) -> k x k correlation [qn, H, W, rfn]."""
    qn, Hp, W, _ = partial.shape
    H = Hp - (k - 1)
    out = torch.empty(qn, H, W, rfn, device=partial.device, dtype=torch.float32)
    _call('g6d_det_corr_rowsum', _p(partial), _p(out), qn, H, W, k, rfn, _stream())
    return out


def det_parse(scores, scales, offsets, pool_ratio=8):
    """scores/scales [qn,hs,ws,1], offsets [qn,hs,ws,2] -> (out [qn,4] = x,y,scale,score; idx [qn] int64)."""
    qn, hs, ws, _ = scores.shape
    out = torch.empty(qn, 4, device=scores.device, dtype=torch.float32)
    idx = torch.empty(qn, device=scores.device, dtype=torch.int64)
    _call('g6d_det_parse', _p(scores), _p(scales), _p(offsets), qn, hs, ws, pool_ratio, _p(out),
          _p(idx, torch.int64), _stream())
    return out, idx


# ------------------------------------------------------------------------------- selector
def sel_ref_sums(ref):
    """ref [S, P, C] -> (sum, sum of squares) over S, float64 [P, C]."""
    S, Pn, Cc = ref.shape
    s1 = torch.empty(Pn, Cc, device=ref.device, dtype=torch.float64)
    s2 = torch.empty_like(s1)
    _call('g6d_sel_ref_sums', _p(ref), S, Pn, Cc, _p(s1, torch.float64), _p(s2, torch.float64), _stream())
    return s1, s2


def sel_corr_prologue(q, s1, s2, S, eps=1e-5):
    """q [P, C] -> (scale [P, C], shift [C]); or qn queries at once, q [qn, P, C] -> ([qn, P, C], [qn, C])."""
    qn, Pn, Cc = (1,) + tuple(q.shape) if q.dim() == 2 else q.shape
    scale = torch.empty(q.shape, device=q.device, dtype=torch.float32)
    shift = torch.empty(q.shape[:-2] + (Cc,), device=q.device, dtype=torch.float32)
    _call('g6d_sel_corr_prologue', _p(q), _p(s1, torch.float64), _p(s2, torch.float64), S, Pn, Cc, qn, eps, _p(scale),
          _p(shift), _stream())
    return scale, shift


def sel_corr_score(ref, q, out=None):
    S, Pn, Cc = ref.shape
    if out is None:
        out = torch.empty(S, device=ref.device, dtype=torch.float32)
    _call('g6d_sel_corr_score', _p(ref), _p(q), S, Pn, Cc, _p(out), _stream(),
          work=4.0 * (S * Pn * Cc + Pn * Cc + S))
    return out


def sel_corr_score3(refs, qs, counters=None):
    """refs: 3 x [S, P_l, C]; qs: 3 x [P_l, C] -> score [3, S], or qn queries at once, qs: 3 x [qn, P_l, C] ->
    score [qn, 3, S], in one streaming pass over refs.
    counters: int32 [3*qn*S], zero (the kernel leaves it zero): one launch; None: dots + finish kernels."""
    S, Cc = refs[0].shape[0], refs[0].shape[2]
    Ps = [r.shape[1] for r in refs]
    qn = 1 if qs[0].dim() == 2 else qs[0].shape[0]
    out = torch.empty(qs[0].shape[:-2] + (3, S), device=refs[0].device, dtype=torch.float32)
    ws = torch.empty(_lib.lib().g6d_sel_corr_score3_workspace_bytes(S, *Ps, qn) // 4, device=refs[0].device, dtype=torch.float32)
    _call('g6d_sel_corr_score3', _p(refs[0]), _p(refs[1]), _p(refs[2]), _p(qs[0]), _p(qs[1]), _p(qs[2]), S, Ps[0], Ps[1],
          Ps[2], Cc, qn, _p(out), _p(ws), _p(counters, torch.int32), _stream(),
          work=4.0 * (S * sum(Ps) * Cc + qn * (sum(Ps) * Cc + 3 * S)))
    return out


def sel_vp_norm(score, feats, coff, eps=1e-5):
    """score [L, n] -> feats rows i; or [groups, L, n] -> feats rows g*n + i (channel coff + l)."""
    groups, Ln, n = (1,) + tuple(score.shape) if score.dim() == 2 else score.shape
    _call('g6d_sel_vp_norm', _p(score), groups, Ln, n, eps, _p(feats), feats.shape[-1], coff, _stream())


def sel_max_angle_add(x, embed):
    """x [groups*rfn, an, C], embed [rfn, C] (shared by the groups) -> [groups*rfn, C]."""
    rows, an, Cc = x.shape
    rfn = embed.shape[0]
    if rows % rfn:
        raise ValueError(f'sel_max_angle_add: {rows} rows are not a whole number of {rfn}-reference groups')
    out = torch.empty(rows, Cc, device=x.device, dtype=torch.float32)
    _call('g6d_sel_max_angle_add', _p(x), _p(embed), _p(out), rows // rfn, rfn, an, Cc, _stream())
    return out


def attention(q, k, v, heads, head_major=False, groups=1):
    """q, k, v [groups*n, C] -> [groups*n, C]: each group of n consecutive tokens attends within itself.
    head_major=False: the reference's channel order c = d*heads + head;
    True: c = head*D + d (the tiled kernel; producers / consumer permuted at pack time)."""
    rows, Cc = q.shape
    if rows % groups:
        raise ValueError(f'attention: {rows} tokens are not {groups} equal groups')
    out = torch.empty_like(q)
    _call('g6d_attention_headmajor' if head_major else 'g6d_attention', _p(q), _p(k), _p(v), _p(out), groups, rows // groups,
          Cc, heads, _stream())
    return out


def layernorm(x, gamma, beta, eps=1e-5):
    rows, Cc = x.shape
    out = torch.empty_like(x)
    _call('g6d_layernorm', _p(x), _p(gamma), _p(beta), _p(out), rows, Cc, eps, _stream())
    return out


def sel_parse(logits, angles):
    qn, rfn = logits.shape
    idx = torch.empty(qn, device=logits.device, dtype=torch.int64)
    out = torch.empty(qn, 2, device=logits.device, dtype=torch.float32)
    _call('g6d_sel_parse', _p(logits), _p(angles), qn, rfn, _p(idx, torch.int64), _p(out), _stream())
    return idx, out


# ------------------------------------------------------------------------------- refiner
def ref_volume_fill(ref_feats, que_feats, ref_Ks, ref_poses, que_Ks, que_poses, sn, img_h, img_w):
    Q, R, fh, fw, Cc = ref_feats.shape
    mean_in = torch.empty(Q, sn, sn, sn, 2 * Cc, device=ref_feats.device, dtype=torch.float32)
    stdv = torch.empty(Q, sn, sn, sn, Cc, device=ref_feats.device, dtype=torch.float32)
    _call('g6d_ref_volume_fill', _p(ref_feats), _p(que_feats), _p(ref_Ks), _p(ref_poses), _p(que_Ks), _p(que_poses),
          Q, R, fh, fw, Cc, sn, img_h, img_w, _p(mean_in), _p(stdv), _stream(),
          work=4.0 * Q * ((R + 1) * fh * fw * Cc + 3 * Cc * sn ** 3))
    return mean_in, stdv


def ref_pose_heads(x, w, b):
    M, K = x.shape
    out = torch.empty(M, 7, device=x.device, dtype=torch.float32)
    _call('g6d_ref_pose_heads', _p(x), _p(w), _p(b), _p(out), M, K, _stream())
    return out
