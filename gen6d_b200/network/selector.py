"""Viewpoint selector on the sm_100a kernels.  Mirrors network/selector.py (+ attention.py) of the
reference: class name, cfg keys, checkpoint keys, load_ref_imgs / select_que_imgs numpy API and
extract_ref_feats / compute_view_point_feats / forward tensor API.

Device-side data layout (see DESIGN.md): the cached reference stack is channels-last and
slice-major, ref[l] = [S = rfn*an (r-major, a-minor), h_l, w_l, 512], which is simultaneously
 * the streaming operand of the correlation-score kernel (one 2 KB row per (slice, location)),
 * the input tensor of the first tower convolution, whose loader forms the (never
   materialised) correlation volume q (.) ref with the first InstanceNorm3d folded in.
"""
import numpy as np
import torch

from .. import ops
from .backbone import pack_vgg, vgg_v1
from .base import Branches, PackedModule, linear_as_conv
from .params import SEL_TOWER_POST, SEL_TOWERS, VGG11BNParams, selector_modules

IN_EPS = 1e-5


class LocalComm:
    """Single-process stand-in for gen6d_b200.dist.Comm (no sharding)."""
    rank, world, capturable = 0, 1, True

    def all_reduce_sum(self, t):
        return t

    def all_gather_cat(self, t, dim=0):
        return t

    def shard_range(self, n):
        return 0, n


FEAT_PAD = 516  # 512 correlation features + 3 similarity scores, padded to a multiple of 4


class ViewpointSelector(PackedModule):
    default_cfg = {'selector_angle_num': 5}

    def __init__(self, cfg):
        self.cfg = {**self.default_cfg, **cfg}
        super().__init__()
        self.backbone = VGG11BNParams()
        for name, mod in selector_modules(self.cfg['selector_angle_num']).items():
            setattr(self, name, mod)
        self.ref_feats_cache = None   # 3 x [S_local, h, w, 512]
        self.ref_sums = None          # per level (sum, sum of squares) over ALL S, float64 [h*w, 512]
        self.ref_pose_embed = None    # [rfn_local, 512]
        self.ref_shape = None         # (rfn_local, an)
        self.rfn_total = None         # references over all shards
        self.comm = LocalComm()       # gen6d_b200.dist.Comm when the reference axis is sharded over GPUs

    # ------------------------------------------------------------------ weights
    def _pack(self):
        an = self.cfg['selector_angle_num']
        p = {'vgg': pack_vgg(self.backbone)}
        p['towers'] = []
        for lvl in range(3):
            tower = self.corr_conv_list[lvl]
            p['towers'].append([(ops.pack_conv(tower[s].weight, tower[s].bias, pad=(0, 1, 1)), SEL_TOWER_POST[lvl][s])
                                for s in sorted(SEL_TOWERS[lvl])])
        cf = self.corr_feats_conv
        p['cf0'] = ops.pack_conv(cf[0].weight, cf[0].bias, pad=0)
        p['cf3'] = ops.pack_conv(cf[3].weight, cf[3].bias, pad=0)
        sp = self.score_process
        p['sp0'] = ops.pack_conv(sp[0].weight, sp[0].bias, pad=0, cin_pad=FEAT_PAD)
        p['sp2'] = ops.pack_conv(sp[2].weight, sp[2].bias, pad=0)
        # attention.py:50-68 splits channels as c = d*8 + head; the tiled attention kernel wants each head's 64
        # dims contiguous (c' = head*64 + d).  Permuting the OUTPUT rows of conv_query / conv_key / conv_feats
        # and the INPUT columns of conv_merge once here makes the projections emit / consume that order.
        heads, dh = 8, 64
        hm = torch.arange(512, device=self.device)
        hm = (hm % dh) * heads + hm // dh                     # position c' = h*64 + d  <-  reference channel d*8 + h
        p['atts'] = []
        for att in self.atts:
            pk = {k: linear_as_conv(getattr(att, k).weight[hm], getattr(att, k).bias[hm]) for k in ('conv_query', 'conv_key', 'conv_feats')}
            pk['conv_merge'] = linear_as_conv(att.conv_merge.weight[:, hm], att.conv_merge.bias)
            p['atts'].append(pk | {'ln_w': att.norm.norm.weight.float().contiguous(),
                                   'ln_b': att.norm.norm.bias.float().contiguous()})
        p['mlps'] = [(linear_as_conv(m[0].weight, m[0].bias), linear_as_conv(m[3].weight, m[3].bias)) for m in self.mlps]
        p['score_predict'] = [linear_as_conv(self.score_predict[i].weight, self.score_predict[i].bias) for i in (0, 2)]
        # angle_predict consumes feats.permute(0,1,3,2).reshape(qn, f*an, rfn): channel = f*an + a
        # (selector.py:212-214).  Our per-reference row is [an, FEAT_PAD] flattened (a*FEAT_PAD + f),
        # so permute (and zero-pad) the first layer's input columns once here.
        w0 = self.angle_predict[0].weight.reshape(512, 515, an)            # [o, f, a]
        w0p = torch.zeros(512, an, FEAT_PAD, device=w0.device, dtype=torch.float32)
        w0p[:, :, :515] = w0.permute(0, 2, 1)
        p['angle_predict'] = [linear_as_conv(w0p.reshape(512, an * FEAT_PAD, 1), self.angle_predict[0].bias)] + \
                             [linear_as_conv(self.angle_predict[i].weight, self.angle_predict[i].bias) for i in (2, 4)]
        p['vpe'] = [linear_as_conv(self.view_point_encoder[i].weight, self.view_point_encoder[i].bias) for i in (0, 2, 4)]
        return p

    # ------------------------------------------------------------------ features
    def _feats(self, imgs_norm4):
        """selector.py:113-119: VGG + per-pixel L2 normalisation; input already ImageNet-normalised."""
        return [ops.l2norm_channels(f) for f in vgg_v1(self.packed()['vgg'], imgs_norm4)]

    @staticmethod
    def viewpoints(ref_poses, object_center, object_vert):
        """Normalised viewpoint directions (selector.py:131-147), fp32 on the host: camera centres
        relative to the object in the (x, y, vert) frame anchored on the FIRST reference."""
        ref_poses = torch.as_tensor(ref_poses, dtype=torch.float32).cpu()
        center = torch.as_tensor(object_center, dtype=torch.float32).cpu()
        vert = torch.as_tensor(object_vert, dtype=torch.float32).cpu()
        cam = (-ref_poses[:, :3, :3].permute(0, 2, 1) @ ref_poses[:, :3, 3:])[..., 0] - center[None]
        fwd = cam[0]
        y = torch.linalg.cross(vert, fwd)
        x = torch.linalg.cross(y, vert)
        nrm = lambda v: v / torch.clamp(torch.linalg.norm(v), min=1e-12)
        R = torch.stack([nrm(x), nrm(y), nrm(vert)], 0)
        cam = cam @ R.T
        return cam / torch.clamp(torch.linalg.norm(cam, dim=1, keepdim=True), min=1e-12)

    def _load_nhwc(self, ref_norm4, rfn, an, ref_poses, object_center, object_vert, chunk=64):
        """ref_norm4: this rank's references [r0, r1) of the rfn in total, [S_local = (r1-r0)*an (r-major), h, w, 4]
        ImageNet-normalised (selector.py:121-148); ref_poses are those of ALL rfn references.  The callers
        slice the image set BEFORE it is uploaded / converted, so a rank never holds more than its shard."""
        p = self.packed()
        self.rfn_total = rfn
        r0, r1 = self.comm.shard_range(rfn)
        assert ref_norm4.shape[0] == (r1 - r0) * an
        vp_all = self.viewpoints(ref_poses, object_center, object_vert)   # frame anchored on GLOBAL ref 0
        rfn = r1 - r0
        S = rfn * an
        levels = [[], [], []]
        for s0 in range(0, S, chunk):
            for l, f in enumerate(self._feats(ref_norm4[s0:s0 + chunk])):
                levels[l].append(f)
        self.ref_feats_cache = [torch.cat(lv, 0) if len(lv) > 1 else lv[0] for lv in levels]
        sums = [ops.sel_ref_sums(f.reshape(S, -1, f.shape[-1])) for f in self.ref_feats_cache]
        # closed-form first-InstanceNorm statistics need the sums over ALL references: one all-reduce at load
        self.ref_sums = [(self.comm.all_reduce_sum(a), self.comm.all_reduce_sum(b)) for a, b in sums]
        self.ref_shape = (rfn, an)
        vp = torch.zeros(rfn, 4, dtype=torch.float32)
        vp[:, :3] = vp_all[r0:r1]
        x = vp.to(self.device).reshape(rfn, 1, 1, 4)
        for i, pc in enumerate(p['vpe']):
            x = ops.conv(x, pc, act=ops.ACT_RELU if i < 2 else ops.ACT_NONE)
        self.ref_pose_embed = x.reshape(rfn, 512)
        self.bump_generation()          # captured graphs / worker clones hold pointers to the previous reference set

    def comm_stats(self):
        """Collectives issued per select pass (one batch of queries) by the sharded path (counted on the last eager /
        capture pass)."""
        return dict(getattr(self.comm, 'calls', {}))

    def _s2_counters(self, qn):
        """Completion counters of the fused S2 kernel for qn queries: zero between calls (the kernel restores
        that), one buffer per batch size (captured graphs of several sizes keep theirs), private to this handle
        (worker clones run concurrently on other streams and get their own)."""
        n = 3 * qn * self.ref_shape[0] * self.ref_shape[1]
        bufs = self.__dict__.setdefault('_s2_done', {})
        c = bufs.get(n)
        if c is None or c.device != self.device:
            c = bufs[n] = torch.zeros(n, device=self.device, dtype=torch.int32)
        return c

    def _finalize(self, ws, rows_total):
        """InstanceNorm scale / shift from the (sum, sum-of-squares) moments a convolution's epilogue
        produced (fp64).  The group may span GPUs: the moments are all-reduced first, so the statistics are
        exact, not per-shard."""
        return ops.instnorm_finalize(self.comm.all_reduce_sum(ws), rows_total, IN_EPS)

    # Batched layout: every tensor after the first tower convolution holds qn*S items, query-major (item
    # g*S + s for query g and reference slice s), so each per-query InstanceNorm group is a run of consecutive
    # rows and every kernel runs once per batch at M scaled by qn.

    def _tower_step(self, st, pc, last, cat_buf, level, S, qn):
        """One convolution of corr_conv_list[level] (selector.py:27-69).  The first reads the shared reference
        stack (S items) with query g's correlation prologue for output items g*S .. g*S+S-1."""
        x = st['x']
        h, w = x.shape[1], x.shape[2]
        if last:
            ops.conv(x, pc, prologue=st['pro'], pro_scale=st['ps'], pro_shift=st['pb'], group_rows=S, out=cat_buf,
                     out_coff=256 * level, batch=qn * S)
            return None
        rows = S * h * w                                              # stride-1 same-size convolution: rows per query
        y, ws = ops.conv(x, pc, prologue=st['pro'], pro_scale=st['ps'], pro_shift=st['pb'], group_rows=S, stats_rows=rows,
                         batch=qn * S)
        return y, ws, rows

    def _advance(self, st, post, y, ps, pb):
        # InstanceNorm3d statistics over (S, h, w) of the raw conv output; the normalisation itself (and the
        # ReLU) is applied by the next conv's loader.  MaxPool commutes with the positive-slope affine, so
        # pooling the raw tensor first is exact.
        st['ps'], st['pb'] = ps, pb
        st['pro'] = ops.PRO_AFFINE_RELU if 'r' in post else ops.PRO_AFFINE
        st['x'] = ops.maxpool2x2(y) if 'p' in post else y

    def _tower_states(self, q_feats, S_total):
        state = []
        for q, ref, (s1, s2) in zip(q_feats, self.ref_feats_cache, self.ref_sums):
            qn, h, w, c = q.shape
            scale, shift = ops.sel_corr_prologue(q.reshape(qn, h * w, c), s1, s2, S_total, IN_EPS)     # one launch per level
            state.append({'x': ref, 'pro': ops.PRO_CORR, 'ps': scale, 'pb': shift})
        return state

    def _towers(self, q_feats, cat_buf, S, S_total, qn):
        """The three towers, each on its own branch stream (they only meet in cat_buf)."""
        towers = self.packed()['towers']
        state = self._tower_states(q_feats, S_total)     # prologue launches on the main stream, before the fork
        br = Branches(3)
        keep = []

        def run(l, st):
            convs = towers[l]
            for i, (pc, post) in enumerate(convs):
                res = self._tower_step(st, pc, i + 1 == len(convs), cat_buf, l, S, qn)
                if res is None:
                    break
                y, ws, rows = res
                ps, pb = self._finalize(ws, rows // self.ref_shape[0] * self.rfn_total)
                self._advance(st, post, y, ps, pb)
                keep.append(st['x'])

        for l, st in enumerate(state):
            br.run(l, lambda l=l, st=st: run(l, st))
        br.join()

    def _towers_sharded(self, q_feats, cat_buf, S, S_total, qn):
        """The three towers with the reference axis sharded over GPUs, ROUND-synchronous: round r runs the
        r-th convolution of every tower that still has one (concurrently, on branch streams), then ONE
        all-reduce carries the InstanceNorm moments [qn, C, 2] of all of them (5 rounds for the 6 + 4 + 2
        convolutions instead of 9 per-layer all-reduces; SURVEY 8e).  Same arithmetic as _towers."""
        towers = self.packed()['towers']
        nbr = 3 if self.comm.capturable else 1
        state, keep = self._tower_states(q_feats, S_total), []
        for st in state:
            st['i'] = 0
        for _ in range(max(len(t) for t in towers)):
            br = Branches(nbr)          # forks from the main stream: after the previous round's finalize / pool kernels
            pend = []
            for l, st in enumerate(state):
                convs = towers[l]
                if st['i'] >= len(convs):
                    continue
                pc, post = convs[st['i']]
                last = st['i'] + 1 == len(convs)
                res = br.run(l, lambda l=l, st=st, pc=pc, last=last: self._tower_step(st, pc, last, cat_buf, l, S, qn))
                st['i'] += 1
                if res is not None:
                    pend.append((st, post, res))
            br.join()
            if not pend:
                continue
            flat = torch.cat([ws.reshape(-1) for _, _, (_, ws, _) in pend]) if len(pend) > 1 else pend[0][2][1].reshape(-1)
            flat = self.comm.all_reduce_sum(flat)                 # one collective for every tower's moments of this round
            o = 0
            for st, post, (y, ws, rows) in pend:
                n = ws.numel()
                ps, pb = ops.instnorm_finalize(flat[o:o + n].reshape(ws.shape), rows // self.ref_shape[0] * self.rfn_total, IN_EPS)
                o += n
                keep.append((y, ws))
                self._advance(st, post, y, ps, pb)

    def _select_batch(self, q_feats):
        """selector.py:177-215 for qn queries in one pass.  q_feats: 3 x [qn, h, w, 512].
        -> logits [qn, rfn], angles [qn, rfn], scores [qn, 3, S]"""
        p = self.packed()
        rfn, an = self.ref_shape
        S = rfn * an
        S_total = self.rfn_total * an
        qn = q_feats[0].shape[0]
        dev = self.device
        cat_buf = torch.empty(qn * S, 4, 4, 768, device=dev, dtype=torch.float32)
        feats = torch.empty(qn * S, FEAT_PAD, device=dev, dtype=torch.float32)   # cols 0-511: cf3, 512-514 + pad: vp_norm
        scores = ops.sel_corr_score3([r.reshape(S, -1, r.shape[-1]) for r in self.ref_feats_cache],
                                     [q.reshape(qn, -1, q.shape[-1]) for q in q_feats], counters=self._s2_counters(qn))
        if self.comm.world == 1:
            self._towers(q_feats, cat_buf, S, S_total, qn)
        else:
            self._towers_sharded(q_feats, cat_buf, S, S_total, qn)
        # corr_feats_conv (selector.py:71-77): 1x1 768->512, IN, ReLU, 1x1 512->512, AvgPool(4,4).
        # The second 1x1 conv is linear, so the 4x4 average is taken first (16x less work).
        y, ws = ops.conv(cat_buf, p['cf0'], stats_rows=S * 16)
        ps, pb = self._finalize(ws, S_total * 16)
        y = ops.avgpool_affine(y.reshape(qn * S * 16, 512), 16, ps, pb, rows_per_group=S * 16, act=ops.ACT_RELU)
        ops.conv(y.reshape(qn * S, 1, 1, 512), p['cf3'], out=feats.reshape(qn * S, 1, 1, FEAT_PAD), out_coff=0)
        if self.comm.world == 1:
            ops.sel_vp_norm(scores, feats, 512, IN_EPS)                 # vp_norm, selector.py:201
        else:   # InstanceNorm2d over ALL (rfn, an): gather the scores along the slice axis, normalise, keep our rows
            all_scores = self.comm.all_gather_cat(scores, dim=2).contiguous()
            tmp = torch.empty(qn * S_total, 4, device=dev, dtype=torch.float32)
            ops.sel_vp_norm(all_scores, tmp, 0, IN_EPS)
            r0, _ = self.comm.shard_range(self.rfn_total)
            feats.reshape(qn, S, FEAT_PAD)[:, :, 512:516] = tmp.reshape(qn, S_total, 4)[:, r0 * an:r0 * an + S]
        x = ops.conv(feats.reshape(qn * S, 1, 1, FEAT_PAD), p['sp0'], act=ops.ACT_RELU)
        x = ops.conv(x, p['sp2']).reshape(qn * rfn, an, 512)
        sf = ops.sel_max_angle_add(x, self.ref_pose_embed)              # selector.py:203-204
        # everything below couples all references (attention, InstanceNorm1d over rfn): gather the
        # per-reference score features once ([qn, rfn, 512] = 128 KB per query at 64 refs) and run the tail replicated
        rfn_local, rfn = rfn, self.rfn_total
        if self.comm.world > 1:
            sf = self.comm.all_gather_cat(sf.reshape(qn, rfn_local, 512), dim=1).reshape(qn * rfn, 512).contiguous()
        for att, (m0, m3) in zip(p['atts'], p['mlps']):
            x4 = sf.reshape(qn * rfn, 1, 1, 512)
            qv = ops.conv(x4, att['conv_query']).reshape(qn * rfn, 512)
            kv = ops.conv(x4, att['conv_key']).reshape(qn * rfn, 512)
            vv = ops.conv(x4, att['conv_feats']).reshape(qn * rfn, 512)
            msg = ops.attention(qv, kv, vv, heads=8, head_major=True, groups=qn)
            msg = ops.conv(msg.reshape(qn * rfn, 1, 1, 512), att['conv_merge']).reshape(qn * rfn, 512)
            msg = ops.layernorm(msg, att['ln_w'], att['ln_b'], 1e-5)
            y = ops.conv(torch.cat([sf, msg], 1).reshape(qn * rfn, 1, 1, 1024), m0)
            ps, pb = ops.instnorm_stats(y, rows_per_group=rfn, eps=IN_EPS)      # InstanceNorm1d over rfn, per query
            y = ops.conv(y, m3, prologue=ops.PRO_AFFINE_RELU, pro_scale=ps, pro_shift=pb, group_rows=rfn)
            ps, pb = ops.instnorm_stats(y, rows_per_group=rfn, eps=IN_EPS)
            y = ops.affine_act(y.reshape(qn * rfn, 512), ps, pb, rows_per_group=rfn, act=ops.ACT_RELU)
            sf = ops.add(y, sf)
        x = ops.conv(sf.reshape(qn * rfn, 1, 1, 512), p['score_predict'][0], act=ops.ACT_RELU)
        logits = ops.conv(x, p['score_predict'][1]).reshape(qn, rfn)
        x = feats.reshape(qn * rfn_local, 1, 1, an * FEAT_PAD)          # angles are per-reference: local
        for i, pc in enumerate(p['angle_predict']):
            x = ops.conv(x, pc, act=ops.ACT_RELU if i < 2 else ops.ACT_NONE)
        angles = self.comm.all_gather_cat(x.reshape(qn, rfn_local), dim=1)
        return logits, angles, scores

    def _select_nhwc(self, que_norm4):
        if self.ref_feats_cache is None:
            raise RuntimeError('ViewpointSelector: load_ref_imgs / extract_ref_feats must be called first')
        return self._select_batch(self._feats(que_norm4))

    def _select_u8(self, u8):
        """uint8 crop(s) on the device -> (ref_idx [qn], (angle, logit) [qn,2], logits [qn,rfn])."""
        logits, angles, _ = self._select_nhwc(ops.preprocess_u8(u8, out_c=4, imagenet_norm=True))
        idx, out = ops.sel_parse(logits, angles)
        return idx, out, logits

    # ------------------------------------------------------------------ reference tensor API
    def extract_ref_feats(self, ref_imgs, ref_poses, object_center, object_vert, is_train=False):
        """ref_imgs [an,rfn,3,h,w] in [0,1] (selector.py:121-148; is_train=False path only)."""
        if is_train:
            raise NotImplementedError('inference-only build: random forward-view selection is a training feature')
        with torch.no_grad():
            an, rfn, _, h, w = ref_imgs.shape
            r0, r1 = self.comm.shard_range(rfn)
            x = ref_imgs[:, r0:r1].permute(1, 0, 2, 3, 4).reshape((r1 - r0) * an, 3, h, w).float().contiguous()
            x = ops.imagenet_norm(ops.nchw_to_nhwc(x), out_c=4)
            self._load_nhwc(x, rfn, an, ref_poses, object_center, object_vert)

    def compute_view_point_feats(self, que_imgs):
        """que_imgs [qn,3,h,w] in [0,1] -> logits [qn,rfn], angles [qn,rfn] (selector.py:177-215)."""
        with torch.no_grad():
            x = ops.imagenet_norm(ops.nchw_to_nhwc(que_imgs.float().contiguous()), out_c=4)
            logits, angles, _ = self._select_nhwc(x)
        return logits, angles

    def forward(self, data):
        self.extract_ref_feats(data['ref_imgs'], data['ref_imgs_info']['poses'], data['object_center'],
                               data['object_vert'], 'eval' not in data)
        logits, angles = self.compute_view_point_feats(data['que_imgs_info']['imgs'])
        return {'ref_vp_logits': logits, 'angles_pr': angles}

    # ------------------------------------------------------------------ reference numpy API
    def load_ref_imgs(self, ref_imgs, ref_poses, object_center, object_vert):
        """@param ref_imgs: uint8 [an,rfn,h,w,3]; ref_poses [rfn,3,4]; object_center [3]; object_vert [3]
        (selector.py:150-163)"""
        with torch.no_grad():
            an, rfn, h, w, _ = ref_imgs.shape
            r0, r1 = self.comm.shard_range(rfn)
            u8 = torch.from_numpy(np.ascontiguousarray(ref_imgs[:, r0:r1].transpose(1, 0, 2, 3, 4))).to(self.device)
            u8 = u8.reshape((r1 - r0) * an, h, w, 3)            # one-off load: no pinned staging ring for ~100s of MB
            x = ops.preprocess_u8(u8, out_c=4, imagenet_norm=True)
            self._load_nhwc(x, rfn, an, ref_poses.astype(np.float32), object_center.astype(np.float32),
                            object_vert.astype(np.float32))

    def _select_warped(self, size):
        def fn(jobs):
            crop = ops.warp_affine_u8(jobs, jobs.numel() // ops.WARP_JOB_BYTES, size, size)
            return (crop,) + tuple(self._select_u8(crop))
        return fn

    def select_from_frame(self, frame_dev, M, size):
        """estimator.py:184-186 in one device stage: cut the detection crop out of the frame with the
        2x3 similarity M (g6d_warp_affine_u8, bit-exact with the reference's cv2.warpAffine), then
        select_que_imgs on it.  frame_dev: uint8 [h,w,3] on the device.  Returns the select_que_imgs
        dict plus 'que_imgs' (the crop, uint8 [1,size,size,3], as the reference hands it on)."""
        from .. import geometry as G
        fn = self._select_warped(size)
        with torch.no_grad():
            jobs = self._to_dev(G.pack_warp_jobs([frame_dev], [G.affine_dst_to_src(M)]))
            if self.comm.capturable:
                crop, idx, out, logits = self.stages.run(f'select_warp{size}', fn, [jobs])
            else:
                crop, idx, out, logits = fn(jobs)           # host-staged collectives inside: run eagerly
            crop, idx, out, logits = [self._to_host(t) for t in (crop, idx, out, logits)]
        return {'ref_idx': idx, 'angles': out[:, 0].copy(), 'scores': logits, 'que_imgs': crop}

    def select_from_frames(self, frames_dev, Ms, size):
        """Batched select_from_frame: crop i is cut out of frames_dev[i] (uint8 [qn,h,w,3] on the device)
        with the 2x3 similarity Ms[i]; one stage (one graph launch, one D2H) for the whole batch."""
        from .. import geometry as G
        fn = self._select_warped(size)
        with torch.no_grad():
            jobs = self._to_dev(G.pack_warp_jobs([frames_dev[i] for i in range(len(Ms))], [G.affine_dst_to_src(M) for M in Ms]))
            if self.comm.capturable:
                crop, idx, out, logits = self.stages.run(f'select_warp{size}', fn, [jobs])
            else:
                crop, idx, out, logits = fn(jobs)
            crop, idx, out, logits = [self._to_host(t) for t in (crop, idx, out, logits)]
        return {'ref_idx': idx, 'angles': out[:, 0].copy(), 'scores': logits, 'que_imgs': crop}

    def select_que_imgs(self, que_imgs):
        """@param que_imgs: uint8 [qn,h,w,3] -> {'ref_idx': i64 [qn], 'angles': f32 [qn], 'scores': f32 [qn,rfn]}
        (selector.py:165-175; the angle is returned un-rescaled, as the reference does)"""
        with torch.no_grad():
            u8 = self._to_dev(que_imgs)
            if self.comm.capturable:    # NCCL collectives are captured with the kernels; gloo (host-staged) runs eagerly
                idx, out, logits = self.stages.run('select', self._select_u8, [u8])
            else:
                idx, out, logits = self._select_u8(u8)
            idx, out, logits = self._to_host(idx), self._to_host(out), self._to_host(logits)
        return {'ref_idx': idx, 'angles': out[:, 0].copy(), 'scores': logits}
