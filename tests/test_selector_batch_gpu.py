"""The viewpoint selector batched over the queries of a batch: every kernel the batched pass uses against the same
kernel called once per query (bit for bit where the per-row arithmetic is the same), and select_que_imgs on a
batch of crops against one crop at a time."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def g(seed):
    gen = torch.Generator(device='cpu')
    gen.manual_seed(seed)
    return gen


@pytest.fixture(scope='module')
def ops():
    from gen6d_b200 import ops
    ops.require_cuda()
    return ops


def corr_problem(S, h, w, qn, cout=128, seed=0):
    """One reference stack [S,h,w,512], qn queries' correlation prologues, a 3x3 tower convolution."""
    from gen6d_b200 import ops
    x = F.normalize(torch.rand(S, h, w, 512, generator=g(seed)), dim=3).cuda()
    scale = (torch.rand(qn, h * w, 512, generator=g(seed + 1)) + 0.5).cuda()
    shift = (torch.randn(qn, 512, generator=g(seed + 2)) * 0.1).cuda()
    wt = (torch.randn(cout, 512, 1, 3, 3, generator=g(seed + 3)) * 0.02).cuda()
    pc = ops.pack_conv(wt, torch.randn(cout, generator=g(seed + 4)).cuda(), pad=(0, 1, 1))
    return x, scale, shift, pc


def corr_batched_vs_loop(ops, S, h, w, qn):
    x, scale, shift, pc = corr_problem(S, h, w, qn)
    rows = S * h * w
    y, ws = ops.conv(x, pc, prologue=ops.PRO_CORR, pro_scale=scale, pro_shift=shift, group_rows=S, stats_rows=rows,
                     batch=qn * S)
    assert y.shape == (qn * S, h, w, pc.cout) and ws.shape == (qn, pc.cout, 2)
    for q in range(qn):
        yq, wq = ops.conv(x, pc, prologue=ops.PRO_CORR, pro_scale=scale[q].contiguous(), pro_shift=shift[q].contiguous(),
                          group_rows=S, stats_rows=rows)
        assert torch.equal(y[q * S:(q + 1) * S], yq), q
        torch.testing.assert_close(ws[q], wq[0], rtol=1e-6, atol=1e-6)        # moments: atomics, order-dependent last bits


# 8x8 planes run on the batch-flattened persistent kernel, 16x16 on the A-reuse (flat) kernel; both sizes keep every
# problem split-free (>= 148 tiles per query), so the batched call and the per-query calls do the same arithmetic per row
CORR_SHAPES = [(320, 8, 8), (160, 16, 16)]


@pytest.mark.parametrize('S,h,w', CORR_SHAPES)
def test_conv_corr_broadcast_equals_per_query(ops, S, h, w):
    corr_batched_vs_loop(ops, S, h, w, qn=3)


def test_conv_corr_broadcast_ffma_path():
    """The same on the fp32 CUDA-core path (G6D_CONV_PATH is read per call, so it runs in a process of its own)."""
    code = ('import sys; sys.path[:0] = [%r, %r]\n'
            'from test_selector_batch_gpu import corr_batched_vs_loop, CORR_SHAPES\n'
            'from gen6d_b200 import ops\n'
            'assert ops.conv_path() == "ffma"\n'
            'for S, h, w in CORR_SHAPES: corr_batched_vs_loop(ops, S, h, w, qn=2)\n'
            'print("ffma ok")\n') % (ROOT, os.path.join(ROOT, 'tests'))
    env = dict(os.environ, G6D_CONV_PATH='ffma')
    r = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and 'ffma ok' in r.stdout, r.stdout + r.stderr


def test_conv_broadcast_rejects_non_divisor(ops):
    x, scale, shift, pc = corr_problem(6, 8, 8, 2)
    with pytest.raises(ValueError):
        ops.conv(x, pc, prologue=ops.PRO_CORR, pro_scale=scale, pro_shift=shift, group_rows=6, batch=9)


@pytest.mark.parametrize('S', [7, 320])
@pytest.mark.parametrize('fused', [True, False])
def test_corr_score3_batched_equals_per_query(ops, S, fused):
    qn, Ps = 4, (256, 64, 16)
    refs = [F.normalize(torch.rand(S, P, 512, generator=g(10 + i)), dim=2).cuda() for i, P in enumerate(Ps)]
    qs = [F.normalize(torch.rand(qn, P, 512, generator=g(20 + i)), dim=2).cuda() for i, P in enumerate(Ps)]
    cb = torch.zeros(3 * qn * S, dtype=torch.int32, device='cuda') if fused else None
    c1 = torch.zeros(3 * S, dtype=torch.int32, device='cuda') if fused else None
    for _ in range(2):                               # the counters come back zero, call after call
        got = ops.sel_corr_score3(refs, qs, counters=cb)
        assert got.shape == (qn, 3, S)
        for q in range(qn):
            want = ops.sel_corr_score3(refs, [t[q].contiguous() for t in qs], counters=c1)
            assert torch.equal(got[q], want), q
        if fused:
            assert int(cb.abs().sum()) == 0 and int(c1.abs().sum()) == 0


def test_corr_prologue_batched_equals_per_query(ops):
    S, P, qn = 40, 64, 3
    ref = F.normalize(torch.rand(S, P, 512, generator=g(30)), dim=2).cuda()
    q = F.normalize(torch.rand(qn, P, 512, generator=g(31)), dim=2).cuda()
    s1, s2 = ops.sel_ref_sums(ref)
    scale, shift = ops.sel_corr_prologue(q, s1, s2, S)
    assert scale.shape == (qn, P, 512) and shift.shape == (qn, 512)
    for i in range(qn):
        a, b = ops.sel_corr_prologue(q[i].contiguous(), s1, s2, S)
        assert torch.equal(scale[i], a) and torch.equal(shift[i], b)


@pytest.mark.parametrize('head_major', [True, False])
def test_grouped_attention_equals_per_group(ops, head_major):
    qn, n, Cc = 5, 64, 512
    q, k, v = [torch.randn(qn * n, Cc, generator=g(40 + i)).cuda() for i in range(3)]
    got = ops.attention(q, k, v, heads=8, head_major=head_major, groups=qn)
    for i in range(qn):
        sl = slice(i * n, (i + 1) * n)
        want = ops.attention(q[sl].contiguous(), k[sl].contiguous(), v[sl].contiguous(), heads=8, head_major=head_major)
        assert torch.equal(got[sl], want), i


def test_vp_norm_and_max_angle_add_per_group(ops):
    qn, rfn, an = 4, 16, 5
    S = rfn * an
    scores = torch.randn(qn, 3, S, generator=g(50)).cuda()
    feats = torch.full((qn * S, 516), float('nan'), device='cuda')
    ops.sel_vp_norm(scores, feats, 512)
    for i in range(qn):
        one = torch.full((S, 516), float('nan'), device='cuda')
        ops.sel_vp_norm(scores[i].contiguous(), one, 512)
        assert torch.equal(feats[i * S:(i + 1) * S, 512:], one[:, 512:]), i
    assert not torch.isnan(feats[:, 512:]).any()          # each group's padding channel is cleared
    x = torch.randn(qn * rfn, an, 512, generator=g(51)).cuda()
    embed = torch.randn(rfn, 512, generator=g(52)).cuda()
    got = ops.sel_max_angle_add(x, embed)
    for i in range(qn):
        assert torch.equal(got[i * rfn:(i + 1) * rfn], ops.sel_max_angle_add(x[i * rfn:(i + 1) * rfn].contiguous(), embed))


@pytest.fixture(scope='module')
def selector():
    from golden import cases
    from gen6d_b200.network import name2network
    from gen6d_b200.weights import seeded_state_dict
    c = cases.selector_case(rfn=16, an=5, qn=10)
    net = name2network['selector'](c['cfg'])
    net.load_state_dict(seeded_state_dict(net, cases.WEIGHT_SEED))
    net.cuda().eval()
    net.load_ref_imgs(c['ref_imgs'], c['ref_poses'], c['object_center'], c['object_vert'])
    singles = [net.select_que_imgs(c['que_imgs'][i:i + 1]) for i in range(len(c['que_imgs']))]
    return net, c['que_imgs'], singles


@pytest.mark.parametrize('qn', [1, 3, 10])
def test_select_que_imgs_batch_equals_one_at_a_time(selector, qn):
    net, imgs, singles = selector
    got = net.select_que_imgs(imgs[:qn])
    assert got['ref_idx'].tolist() == [int(s['ref_idx'][0]) for s in singles[:qn]]
    dl = float(np.abs(got['scores'] - np.concatenate([s['scores'] for s in singles[:qn]])).max())
    da = float(np.abs(got['angles'] - np.concatenate([s['angles'] for s in singles[:qn]])).max())
    print(f'qn={qn}: max |dlogit| {dl:.3g}, max |dangle| {da:.3g}')
    assert dl <= 3e-4 and da <= 3e-4


def test_batched_select_graph_replay_is_deterministic(selector):
    net, imgs, _ = selector
    a = net.select_que_imgs(imgs)
    for _ in range(3):
        b = net.select_que_imgs(imgs)
        assert np.array_equal(a['ref_idx'], b['ref_idx'])
        assert np.array_equal(a['scores'], b['scores']) and np.array_equal(a['angles'], b['angles'])
