"""GPU: training of the LSTM baseline -- the backward kernels against float64 autograd, ``ViT_LSTM.train_engine``'s
backward through time against the CPU reference (tests/lstm_rollout_reference.py), and the agent's
``train_rollout_step`` / ``student_batch`` / ``train_iteration`` (renderer, trunk, policy, optimisers)."""
import os
import tempfile
import types

import numpy as np
import pytest
import torch

import lstm_rollout_reference as ref
from oracle import model_oracle as mo
from oracle import teacher_oracle as to
from oracle import warp_oracle as wo

pytestmark = pytest.mark.gpu


def _rel(a, b):
    """max |a - b| / max |b|"""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


# ------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("has_prev,has_next", [(False, False), (True, False), (False, True), (True, True)])
def test_lstm_cell_bwd_vs_fp64(built_lib, has_prev, has_next):
    from avdn_b200 import _lib
    B, H, pitch = 5, 37, 50
    g = torch.Generator().manual_seed(1)
    gates = torch.randn(B, 4 * H, generator=g) * 2
    cp = torch.randn(B, H, generator=g) if has_prev else None
    dh_buf = torch.randn(B, pitch, generator=g)
    dc_next = torch.randn(B, H, generator=g) if has_next else None
    gd = gates.double().requires_grad_(True)
    cpd = cp.double().requires_grad_(True) if has_prev else None
    i, f, gg, o = torch.sigmoid(gd[:, :H]), torch.sigmoid(gd[:, H:2 * H]), torch.tanh(gd[:, 2 * H:3 * H]), torch.sigmoid(gd[:, 3 * H:])
    c = f * (cpd if has_prev else 0) + i * gg
    h = o * torch.tanh(c)
    loss = (h * dh_buf[:, 3:3 + H].double()).sum() + ((c * dc_next.double()).sum() if has_next else 0)
    loss.backward()
    d = "cuda"
    c32 = c.detach().float().to(d)
    dgates = torch.full((B, 4 * H), 7.0, device=d)
    dc_prev = torch.full((B, H), 7.0, device=d)
    gates_d, cp_d, dh_d = gates.to(d), None if cp is None else cp.to(d), dh_buf.to(d)
    dcn_d = None if dc_next is None else dc_next.to(d)
    dh_view = dh_d[:, 3:]
    p = _lib.ptr
    _lib.call("avdn_lstm_cell_bwd", p(gates_d), p(cp_d), p(c32), p(dh_view), dh_d.stride(0), p(dcn_d), p(dgates),
              p(dc_prev), B, H)
    assert _rel(dgates, gd.grad) < 1e-5, _rel(dgates, gd.grad)
    if has_prev:
        assert _rel(dc_prev, cpd.grad) < 1e-5
    else:
        assert torch.all(dc_prev == 7.0)                       # not written for the zero state


@pytest.mark.parametrize("B,L,D", [(64, 250, 768), (3, 7, 768), (4, 1, 768)])
@pytest.mark.parametrize("with_ctx", [False, True])
def test_lang_attn_bwd_vs_fp64(built_lib, B, L, D, with_ctx):
    from avdn_b200 import _lib
    d = "cuda"
    g = torch.Generator(device=d).manual_seed(B * L)
    ctx = torch.randn(B, L, D, device=d, generator=g)
    tgt = torch.randn(B, D, device=d, generator=g) / D ** 0.5
    dw_buf = torch.randn(B, D + 16, device=d, generator=g)
    dw = dw_buf[:, 16:]
    attn = torch.empty(B, L, device=d)
    wbuf = torch.empty(B, D, device=d)
    p = _lib.ptr
    _lib.call("avdn_lang_attn_fwd", p(ctx), p(tgt), B, L, D, p(attn), p(wbuf), D)
    d_target = torch.full((B, D), 3.0, device=d)
    base = torch.randn(B, L, D, device=d, generator=g)
    d_ctx = base.clone() if with_ctx else None
    _lib.call("avdn_lang_attn_bwd", p(ctx), p(tgt), p(attn), p(dw), dw_buf.stride(0), B, L, D, p(d_target), p(d_ctx))
    cd, td = ctx.double().requires_grad_(True), tgt.double().requires_grad_(True)
    a = torch.softmax(torch.einsum("bld,bd->bl", cd, td), dim=1)
    (torch.einsum("bl,bld->bd", a, cd) * dw.double()).sum().backward()
    assert _rel(d_target, td.grad) < 1e-4, _rel(d_target, td.grad)
    if with_ctx:
        assert _rel(d_ctx - base, cd.grad) < 1e-4, _rel(d_ctx - base, cd.grad)


def test_frame_attn_bwd_without_fc2_vs_fp64(built_lib):
    from avdn_b200 import _lib
    d = "cuda"
    B, T = 3, 4
    g = torch.Generator(device=d).manual_seed(5)
    frames = torch.randn(B * T, 512, 49, device=d, generator=g)
    cls = torch.relu(torch.randn(B, 49, device=d, generator=g))
    w_in = torch.randn(49, 49, device=d, generator=g) / 7
    w_out = torch.randn(49, 98, device=d, generator=g) / 10
    attn, wc, e49 = torch.empty(B * T, 512, device=d), torch.empty(B * T, 49, device=d), torch.empty(B * T, 49, device=d)
    p = _lib.ptr
    _lib.call("avdn_frame_attn_fwd", p(frames), p(cls), p(w_in), p(w_out), None, None, B, T, p(attn), p(wc), p(e49), None)
    d_e = torch.randn(B * T, 49, device=d, generator=g)
    d_frames = torch.full_like(frames, 9.0)
    dwi, dwo = torch.ones(49, 49, device=d), torch.ones(49, 98, device=d)
    d_cls = torch.ones(B, 49, device=d)
    _lib.call("avdn_frame_attn_bwd_cls", p(frames), p(cls), p(w_in), p(w_out), None, B, T, p(attn), p(wc), p(e49), p(d_e),
              p(d_frames), p(dwi), p(dwo), None, None, p(d_cls))
    fd = frames.double().view(B, T, 512, 49).requires_grad_(True)
    cd, wid, wod = (x.double().requires_grad_(True) for x in (cls, w_in, w_out))
    tot = 0
    for t in range(T):
        e, _ = mo.soft_dot_attention(cd, fd[:, t], wid, wod)
        tot = tot + (e * d_e.view(B, T, 49)[:, t].double()).sum()
    tot.backward()
    assert _rel(d_frames, fd.grad.reshape(B * T, 512, 49)) < 1e-4
    assert _rel(dwi - 1, wid.grad) < 1e-4 and _rel(dwo - 1, wod.grad) < 1e-4
    assert _rel(d_cls - 1, cd.grad) < 1e-4


def test_direction_embed_bwd_vs_fp64(built_lib):
    from avdn_b200 import _lib
    d = "cuda"
    B, N = 640, 32
    g = torch.Generator(device=d).manual_seed(2)
    deg = torch.randint(0, 360, (B,), device=d, generator=g).float() + torch.rand(B, device=d, generator=g)
    d_out = torch.randn(B, N, device=d, generator=g)
    dw, db = torch.ones(N, 2, device=d), torch.ones(N, device=d)
    _lib.call("avdn_direction_embed_bwd", _lib.ptr(deg), _lib.ptr(d_out), B, N, _lib.ptr(dw), _lib.ptr(db))
    a = (deg.cpu() / 180 * 3.14159)                              # float32, as the forward evaluates it
    x = torch.stack([torch.sin(a), torch.cos(a)], 1).double()
    assert _rel(dw - 1, d_out.cpu().double().T @ x) < 1e-5
    assert _rel(db - 1, d_out.cpu().double().sum(0)) < 1e-5


# ------------------------------------------------------------------------------ backward through time vs the reference
def _policy(seed=3, train=False):
    from avdn_b200.models.vln_model import ViT_LSTM
    torch.manual_seed(seed)
    m = ViT_LSTM(types.SimpleNamespace(), torch.nn.Identity()).cuda()
    return m.train(train)


def _drop_masks(m, p, seed, B, T):
    from avdn_b200 import _lib
    from avdn_b200.models.vln_model import SITE_INPUT, SITE_FC, SITE_DEC

    def keep(n, site):
        out = torch.empty(n, device="cuda")
        _lib.call("avdn_dropout_keep_scale", _lib.ptr(out), n, p, seed, site)
        return out.cpu()

    inp, fc = keep(T * B * 49, SITE_INPUT).view(T, B, 49), keep(T * B * 128, SITE_FC).view(T, B, 128)
    return [dict(input=inp[t], fc=fc[t], h0=keep(B * 256, SITE_DEC + 2 * t).view(B, 256),
                 h1=keep(B * 32, SITE_DEC + 2 * t + 1).view(B, 32)) for t in range(T)]


@pytest.mark.parametrize("B", [4, 64])
@pytest.mark.parametrize("T", [1, 3, 10])
@pytest.mark.parametrize("dropout", [False, True])
def test_backward_through_time_vs_reference(built_lib, B, T, dropout):
    L = 250
    m = _policy(train=dropout)
    g = torch.Generator().manual_seed(B + T)
    frames = torch.randn(B, T, 512, 49, generator=g)
    deg = torch.randint(0, 360, (B, T), generator=g).float()
    cls = torch.relu(torch.randn(B, 49, generator=g))
    lang = torch.randn(B, L, 768, generator=g)
    gt_xy, gt_alt, gt_prog = torch.rand(B, T, 2, generator=g) * 2 - 1, torch.rand(B, T, generator=g), torch.rand(B, T, generator=g)
    att = torch.zeros(B, T, 224, 224, dtype=torch.uint8)          # fixation maps for half the samples: the NSS term
    att[::2, :, 40:100, 60:140] = 255
    eng = m.train_engine(B, L, T, "cuda")
    p, seed = m.dropout_config()
    assert (p > 0) == dropout
    c = lambda x: x.cuda()
    eng.forward(c(frames).view(B * T, 512, 49), c(deg), c(cls), c(lang), p, seed)
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    tr = lambda x: c(x).transpose(0, 1).contiguous()
    eng.loss(tr(gt_xy), tr(gt_alt), tr(gt_prog), tr(att), 0.1, 0, 0.2 / B, loss)
    d_lang, d_cls = torch.zeros(B, L, 768, device="cuda"), torch.zeros(B, 49, device="cuda")
    d_frames = eng.backward(d_lang, d_cls)
    drop = _drop_masks(m, p, seed, B, T) if dropout else None
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.used_parameters().items()}
    fr, cl, la = (x.clone().requires_grad_(True) for x in (frames, cls, lang))
    total = ref.rollout_loss(sd, fr, deg, cl, la, gt_xy, gt_alt, gt_prog, gt_saliency=att.double() / 255, nss_w=0.1,
                             train_ml=0.2, drop=drop)
    total.backward()
    total = float(total.detach())
    assert abs(float(loss) - total) <= 1e-5 * abs(total), (float(loss), total)
    for n in [n for n in sd if sd[n].grad is None]:       # W_hh at T = 1: the zero state never reaches it
        assert n.endswith("weight_hh") and T == 1 and not eng.G[n].any(), n
        del sd[n]
    report = {n: _rel(eng.G[n], sd[n].grad) for n in sd}
    report.update(frames=_rel(d_frames.view(B, T, 512, 49), fr.grad), lang=_rel(d_lang, la.grad), cls=_rel(d_cls, cl.grad))
    assert max(report.values()) < 1e-3, report


# --------------------------------------------------------------------------------------------------------- agent
SIZE = 1024


def _agent(lr=0.0, **kw):
    from avdn_b200.xview_lstm.agent import NavCMTAgent
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(mo.yolov3_trunk_cfg())
    args = types.SimpleNamespace(darknet_model_file=f.name, darknet_weight_file=None, max_action_len=4, lr=lr, nss_w=0.1,
                                 nss_r=0, ml_weight=0.2, no_dropout=True, **kw)
    torch.manual_seed(0)
    a = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    if lr == 0.0:
        for opt in a.optimizers:
            opt.wd = 0.0
    a.renderer.add_map("m", wo.synthetic_tile(seed=2, size=SIZE), wo.synthetic_attention_tile(seed=2, size=SIZE))
    return a


def _greedy_batch(B, L, seed):
    from bench_rollout import synthetic_rollout_batch
    b = synthetic_rollout_batch(B, L, seed, size=SIZE)
    out = {k: v.cuda() for k, v in b.items()}
    out["tile_idx"] = None
    return out


def _gps_to_px(corners, geo):
    """env.py:189-196: corners [...,4,2] (lat, lng), geo [...,5] broadcast over the four corners."""
    x = np.rint((corners[..., 1] - geo[..., 1, None]) / geo[..., 4, None])
    y = np.rint((geo[..., 2, None] - corners[..., 0]) / geo[..., 4, None])
    return np.stack([x, y], -1).astype(np.int32)


def _teacher_batch(B, T, L, seed):
    """Poses along a straight ground-truth path from the greedy batch's start, random targets."""
    gb = _greedy_batch(B, L, seed)
    c0 = gb["corners_gps"].cpu().numpy()
    geo = gb["geo"].cpu().numpy()
    step = np.array([0.0004, -0.0003])
    gt_paths = [np.stack([c0[i] + k * step for k in range(T + 2)]) for i in range(B)]
    poses = np.stack([gt_paths[i][:T] for i in range(B)])                              # [B,T,4,2]
    px = np.stack([_gps_to_px(poses[i], geo[i]) for i in range(B)])
    g = torch.Generator().manual_seed(seed)
    tb = dict(corners_px=torch.from_numpy(px).cuda(), tile_idx=None, lang_feature=gb["lang_feature"],
              cls_hidden=gb["cls_hidden"], directions=torch.randint(0, 360, (B, T), generator=g).float().cuda(),
              gt_xy=(torch.rand(B, T, 2, generator=g) * 2 - 1).cuda(), gt_alt=torch.rand(B, T, generator=g).cuda(),
              gt_prog=torch.rand(B, T, generator=g).cuda())
    return tb, gb, gt_paths


@pytest.mark.parametrize("bn_per_step", [False, True])
def test_train_rollout_step_vs_reference(built_lib, bn_per_step):
    from avdn_b200 import agent_common
    from avdn_b200.models import dark_net as DN
    B, T, L = 4, 4, 12
    a = _agent()
    tb, _, _ = _teacher_batch(B, T, L, 1)
    ours = a.train_rollout_step(tb, sync_loss=True, step=False, bn_per_step=bn_per_step)
    teng, tengs, eng, bufs = a._ctx
    frames = bufs["frames"].detach().cpu().view(B, T, 512, 49)
    att = bufs["att"].cpu().view(B, T, 224, 224).double() / 255
    sd = {k: v.detach().cpu() for k, v in a.vln_model.used_parameters().items()}
    total = ref.rollout_loss(sd, frames, tb["directions"].cpu(), tb["cls_hidden"].cpu(), tb["lang_feature"].cpu(),
                             tb["gt_xy"].cpu(), tb["gt_alt"].cpu(), tb["gt_prog"].cpu(), gt_saliency=att, nss_w=0.1,
                             train_ml=0.2)
    assert abs(ours - float(total)) <= 1e-4 * abs(float(total)), (ours, float(total))
    # the trunk's gradient arena is what a separate trunk backward of the step's d_frames produces (up to the order of
    # the trunk backward's atomic reductions, which differs from run to run)
    g_step = a.vision_model_optimizer.g.clone()
    a.vision_model_optimizer.zero_grad()
    l0 = sum(e.launches for e in tengs) if tengs else teng.launches
    agent_common.rollout_trunk_backward(a, teng, tengs, l0, eng.d_frames, B, T)
    assert _rel(a.vision_model_optimizer.g, g_step) < 1e-5, _rel(a.vision_model_optimizer.g, g_step)
    if bn_per_step:                # features of step t = a lone train-mode trunk pass over that step's views
        vm = a.vision_model
        x5 = bufs["x"].view(B, T, 224, 224, 4)
        for t in range(T):
            e = vm.engine(B, 224, 224, "cuda", slot=100 + t)
            f = DN._trunk_forward(vm, e, x5[:, t].contiguous(), True)
            assert torch.equal(frames[:, t], f.view(B, 512, 49).cpu()), t


def test_train_iteration_student_feedback(built_lib):
    B, T, L = 4, 4, 12
    a = _agent()
    tb, gb, gt_paths = _teacher_batch(B, T, L, 2)
    sb = a.student_batch(gb, gt_paths, max_action_len=T)
    res = a._bufs[(B, T)]                     # the buffers of student_batch's greedy rollout (its return values)
    corners = res["corners_hist"][:T].cpu().numpy()                                  # [T,B,4,2]
    geo = gb["geo"].cpu().numpy()
    for t in range(T):
        assert np.array_equal(sb["corners_px"][:, t].cpu().numpy(), _gps_to_px(corners[t], geo))
    assert torch.equal(sb["directions"], res["dir_hist"][:T].float().t())
    ended = res["ended_hist"].cpu().numpy()
    for t in range(T):
        for i in range(B):
            r, alt, prog = to.teacher_action(corners[t, i], gt_paths[i], bool(t > 0 and ended[t - 1, i]), "student")
            np.testing.assert_allclose(sb["gt_xy"][i, t].cpu().numpy(), r, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(float(sb["gt_alt"][i, t]), alt, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(float(sb["gt_prog"][i, t]), prog, rtol=1e-5, atol=1e-6)
    # one iteration = the teacher rollout (nss_w 0) + the student rollout, gradients added (lr 0: weights stay)
    total = a.train_iteration(tb, sb, sync_loss=True)
    g_it = [o.g.clone() for o in a.optimizers]
    l1 = a.train_rollout_step(tb, sync_loss=True, step=False, nss_w=0.0)
    g1 = [o.g.clone() for o in a.optimizers]
    l2 = a.train_rollout_step(sb, sync_loss=True, step=False, nss_w=0.1)
    g2 = [o.g.clone() for o in a.optimizers]
    assert abs(total - (l1 + l2)) <= 1e-6 * abs(total), (total, l1, l2)
    for gi, x, y in zip(g_it, g1, g2):
        assert _rel(gi, x + y) < 1e-4, _rel(gi, x + y)


def test_greedy_rollout_after_training_uses_the_trained_state(built_lib):
    """After three training iterations the greedy rollout gives the same bits as a fresh agent loaded from the trained
    agent's state_dict: no stale packed weights, CUDA graphs of the trunk or BatchNorm coefficients.  Each rollout
    starts from the zero recurrent state (src/xview_lstm/agent.py:546-550), so two rollouts of one agent agree too."""
    B, T, L = 4, 4, 12
    a = _agent(lr=1e-4)
    tb, gb, gt_paths = _teacher_batch(B, T, L, 3)
    before = a.rollout_greedy(gb, max_action_len=T)["output"].clone()      # packs the weights, captures the graph
    assert torch.equal(a.rollout_greedy(gb, max_action_len=T)["output"], before)
    for _ in range(3):
        sb = a.student_batch(gb, gt_paths, max_action_len=T)
        a.train_iteration(tb, sb)
    res = {k: v.clone() for k, v in a.rollout_greedy(gb, max_action_len=T).items()}
    fresh = _agent(lr=1e-4)
    fresh.vln_model.load_state_dict(a.vln_model.state_dict())
    res2 = fresh.rollout_greedy(gb, max_action_len=T)
    assert not torch.equal(before, res["output"])
    for k in ("output", "corners", "directions", "ended"):
        assert torch.equal(res[k], res2[k]), k


def test_training_lowers_the_loss(built_lib):
    B, T, L = 4, 4, 12
    a = _agent(lr=1e-4)
    tb, _, _ = _teacher_batch(B, T, L, 4)
    losses = [a.train_rollout_step(tb, sync_loss=True) for _ in range(30)]
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses
