"""GPU: the LSTM agent's drop-in loop -- ``attach_lang_model``, ``rollout(train_ml, not_in_train, nss_w)``,
``train(loader, n_epochs, feedback, nss_w_weighting)``, ``test(loader, ...)``, ``save`` / ``load`` over ``agent.env``
(src/xview_lstm/agent.py) -- and ``avdn_saliency_metrics``, the one-launch human-attention scoring of its
teacher-feedback validation, against a float64 torch restatement of the ET agent's per-sample loop."""
import os
import tempfile
import types

import numpy as np
import pytest
import torch

import lstm_rollout_reference as ref
from oracle import bert_oracle as bo
from oracle import model_oracle as mo
from oracle import teacher_oracle as to
from oracle import warp_oracle as wo
from test_agent_dropin_gpu import BL, SIZE, TR, _Tok, _items

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _host_scores(sal, gt, nss_r):
    """xview_et/agent.py ``_eval_rollout`` scoring of one sample in float64 torch: NSS (agent.py:256-270), the
    clipped map's precision and recall.  ``sal`` [224,224] f32 (the upsampled map), ``gt`` [224,224] f64 in [0,1]."""
    s = sal.double().view(1, -1)
    n = (s - s.mean(1, keepdim=True)) / s.std(1, keepdim=True)
    if nss_r == 1:
        n = n / 2 + 1
    elif nss_r == -1:
        n = n / 2 - 1
    f = gt.view(1, -1)
    nss = float(-((n * f).sum(1) / (f.sum(1) + 0.001)).mean())
    p = sal.clip(0, 1).double()
    tp, sp = float((p * gt).sum()), float(p.sum())
    return tp / sp if sp != 0 else 0.0, tp / float(gt.sum()), nss


def _metrics(h, att, nss_r):
    from avdn_b200 import _lib
    out = torch.full((h.shape[0], 4), float("nan"), dtype=torch.float64, device="cuda")
    _lib.call("avdn_saliency_metrics", _lib.ptr(h), _lib.ptr(att), h.shape[0], nss_r, _lib.ptr(out))
    return out


def _upsample(h):
    from avdn_b200 import _lib
    sal = torch.empty((h.shape[0], 224, 224), dtype=torch.float32, device="cuda")
    _lib.call("avdn_upsample_saliency", _lib.ptr(h), h.shape[0], _lib.ptr(sal))
    return sal


# ------------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("nss_r", [-1, 0, 1])
def test_saliency_metrics_vs_fp64(built_lib, nss_r):
    N = 640
    g = torch.Generator().manual_seed(11 + nss_r)
    h = torch.randn(N, 64, generator=g) * 0.6 + 0.3
    h[1::5] = -h[1::5].abs() - 0.01                       # negative maps: the clip is all zero, precision 0
    h[2::7] *= 40                                        # large values: the clip saturates
    att = torch.zeros(N, 224, 224, dtype=torch.uint8)
    yy, xx = torch.meshgrid(torch.arange(224), torch.arange(224), indexing="ij")
    for i in range(N):
        if i % 4 == 3:
            continue                                     # all-zero fixation map: reported with a fixation sum of 0
        cy, cx, r = torch.randint(0, 224, (3,), generator=g).tolist()
        disc = (yy - cy) ** 2 + (xx - cx) ** 2 <= (r % 80 + 5) ** 2
        att[i][disc] = 255 if i % 2 else torch.randint(1, 256, (1,), generator=g).item()
    h, att = h.cuda(), att.cuda()
    out = _metrics(h, att, nss_r)
    assert torch.equal(out, _metrics(h, att, nss_r))     # a fixed reduction order: two launches agree bit for bit
    sal = _upsample(h)
    gt = att.double() / 255
    fs = gt.view(N, -1).sum(1).cpu()
    o = out.cpu()
    assert torch.equal(o[:, 3] == 0, fs == 0)
    assert (o[:, 3] - fs).abs().max() <= 1e-9 * fs.max()
    n_zero_prec = 0
    for i in range(N):
        if fs[i] == 0:
            continue
        prec, rec, nss = _host_scores(sal[i], gt[i], nss_r)
        for k, v in enumerate((prec, rec, nss)):
            assert abs(float(o[i, k]) - v) <= 1e-9 * max(abs(v), 1e-12), (i, k, float(o[i, k]), v)
        n_zero_prec += prec == 0.0
    assert n_zero_prec > 0


def test_saliency_metrics_rejects_bad_arguments(built_lib):
    from avdn_b200 import _lib
    h = _lib.lib()
    assert h.avdn_saliency_metrics(None, None, 4, 0, None, None) == -1
    assert "null" in _lib.last_error()
    x = torch.zeros(64, device="cuda")
    assert h.avdn_saliency_metrics(_lib.ptr(x), _lib.ptr(x), 1, 2, _lib.ptr(x), None) == -1
    assert h.avdn_saliency_metrics(_lib.ptr(x), _lib.ptr(x), -1, 0, _lib.ptr(x), None) == -1


# ------------------------------------------------------------------------------------------------------- agent
def _make_agent(seed=0, **kw):
    from transformers import BertConfig
    from avdn_b200.models.bert import CustomBERTModel
    from avdn_b200.xview_lstm.agent import NavCMTAgent
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(mo.yolov3_trunk_cfg())
    args = types.SimpleNamespace(darknet_model_file=f.name, darknet_weight_file=None, lr=1e-5, nss_w=0.1, nss_r=0,
                                 ml_weight=0.2, teacher_weight=1.0, max_action_len=4, no_dropout=True,
                                 train_val_on_full=False, vision_only=False, optim="adamW", **kw)
    torch.manual_seed(seed)
    agent = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    agent.tokenizer = _Tok(400)
    agent.attach_lang_model(CustomBERTModel(BertConfig(num_hidden_layers=1, vocab_size=400, max_position_embeddings=64)))
    return agent


def _env(B=4):
    from avdn_b200.env import ANDHNavBatch
    env = ANDHNavBatch(batch_size=B, device="cuda")
    tile, att = wo.synthetic_tile(seed=4, size=SIZE), wo.synthetic_attention_tile(seed=4, size=SIZE)
    env.map_batch["m0"], env.attention_map_batch["m0"] = tile, att
    env.batch = _items(B, 7)
    return env, tile, att


@pytest.fixture(scope="module")
def setup(built_lib):
    agent = _make_agent()
    env, tile, att = _env()
    agent.env = env
    return agent, env, tile, att


def _zero_lr(agent, lr=0.0):
    for opt in agent.optimizers:
        opt.lr, opt.wd = lr, 0.0
        opt.zero_grad()


def test_teacher_training_rollout_vs_reference(setup):
    agent, env, tile, att = setup
    B = env.batch_size
    _zero_lr(agent)
    agent.loss, agent.feedback, agent.env_name = 0, "teacher", "train"
    n_log = len(agent.logs["IL_loss"])
    traj = agent.rollout(train_ml=0.2, nss_w=0.1)
    ours = float(agent.loss)
    lr = agent._last_rollout
    steps = lr["steps"]
    # ---- the pose sequence is the oracle simulator driven by the oracle teacher ----
    corners = lr["corners"].cpu().numpy()
    ended = lr["ended"].cpu().numpy().astype(bool)
    items = env.batch
    c = np.stack([np.asarray(it["gt_path_corners"][0]) for it in items])
    d = np.array([it["angle"] for it in items], dtype=np.float64)
    e = np.zeros(B, dtype=bool)
    bounds = np.tile(np.concatenate([BL, TR]), (B, 1))
    tx, ta, tp = lr["tgt_xy"].cpu().numpy(), lr["tgt_alt"].cpu().numpy(), lr["tgt_prog"].cpu().numpy()
    for t in range(steps):
        assert np.allclose(corners[t], c, rtol=0, atol=1e-9), t
        out = np.zeros((B, 4), dtype=np.float32)
        for i in range(B):
            xy, alt, prog = to.teacher_action(c[i], items[i]["gt_path_corners"], e[i], feedback="teacher")
            assert np.allclose(tx[t, i], xy, atol=2e-5) and abs(ta[t, i] - alt) < 1e-5 and abs(tp[t, i] - prog) < 1e-5
            out[i] = (tx[t, i, 0], tx[t, i, 1], ta[t, i], tp[t, i])
        c, d, e, *_ = mo.waypoint_step(out, c, bounds, d, e, agent.STOP_THRESHOLD, t == agent.args.max_action_len - 1)
        assert np.array_equal(ended[t], e), t
    if steps < agent.args.max_action_len:
        assert e.all()                                   # the early exit happens once every sample has ended
    # ---- loss: the CPU reference rollout on OUR trunk features, cv2-exact attention maps ----
    batch = lr["batch"]
    frames = agent._ctx[3]["frames"].detach().cpu().view(B, steps, 512, 49)
    px = batch["corners_px"].cpu().numpy()
    sal_gt = torch.from_numpy(np.stack([np.stack([wo.warp_fixed_point(att, wo.inverse_homography(px[i, t]))[:, :, 0]
                                                  for t in range(steps)]) for i in range(B)]).astype(np.float64) / 255)
    sd = {k: v.detach().cpu() for k, v in agent.vln_model.used_parameters().items()}
    seq, lin = agent._lang_eval_forward(batch)           # no dropout: the train-mode pass computes the same
    sd_b = {k: v.detach().cpu().clone() for k, v in agent.lang_model.state_dict().items() if "position_ids" not in k}
    with torch.no_grad():
        oseq, _, _ = bo.custom_bert_forward(sd_b, batch["input_ids"].cpu(), batch["attention_mask"].cpu())
        _, olin, _ = bo.custom_bert_forward(sd_b, batch["cls_input_ids"].cpu(), batch["cls_attention_mask"].cpu())
    args = (frames, batch["directions"].cpu())
    tgt = (batch["gt_xy"].cpu(), batch["gt_alt"].cpu(), batch["gt_prog"].cpu())
    with torch.no_grad():
        r_ours = float(ref.rollout_loss(sd, *args, lin.cpu().float(), seq.cpu().float(), *tgt, gt_saliency=sal_gt,
                                        nss_w=0.1, train_ml=0.2))
        r_oracle = float(ref.rollout_loss(sd, *args, olin.float(), oseq.float(), *tgt, gt_saliency=sal_gt, nss_w=0.1,
                                          train_ml=0.2))
    assert abs(ours - r_ours) <= 1e-4 * abs(r_ours), (ours, r_ours)
    assert abs(ours - r_oracle) <= 1e-2 * abs(r_oracle), (ours, r_oracle)
    # ---- bookkeeping of the reference ----
    assert len(agent.logs["IL_loss"]) == n_log + 1 and abs(agent.il_losses()[-1] - ours) < 1e-9
    assert len(agent.losses) >= 1 and abs(float(agent.losses[-1]) - ours) < 1e-9
    assert len(traj) == B
    for i, tr in enumerate(traj):
        assert tr["instr_id"] == "m0__" + str(i) and tr["num_dia"] == 1
        assert len(tr["actions"]) == len(tr["gt_actions"]) == len(tr["gt_progress"]) == len(tr["progress"])
        assert 1 <= len(tr["actions"]) <= steps
        assert len(tr["path_corners"]) in (len(tr["actions"]), len(tr["actions"]) + 1)
        assert np.array_equal(tr["path_corners"][0][0], np.asarray(items[i]["gt_path_corners"][0]))
    for opt in agent.optimizers:                         # policy, trunk, BERT
        assert float(opt.g.abs().sum()) > 0


def test_bert_gradient_is_one_backward_of_the_collected_gradients(setup):
    agent, env, _, _ = setup
    _zero_lr(agent)
    agent.loss, agent.feedback = 0, "teacher"
    agent.rollout(train_ml=0.2, nss_w=0.1)
    lo = agent.lang_optimizer
    g_roll = lo.g.clone()
    eng = agent._ctx[2]
    B, L = eng.B, eng.L
    d_lang = torch.zeros((B, L, 768), device="cuda")
    d_cls = torch.zeros((B, 49), device="cuda")
    eng.backward(d_lang, d_cls)                          # the policy engine's summed d lang_feature / d cls_hidden
    lo.zero_grad()
    batch = agent._last_rollout["batch"]
    _, _, leng, leng2 = agent._lang_train_forward(batch)
    agent._lang_train_backward(leng, leng2, d_lang, d_cls)
    assert float(g_roll.abs().sum()) > 0
    assert _rel(lo.g, g_roll) < 1e-4, _rel(lo.g, g_roll)


def test_train_student_feedback(setup):
    agent, env, _, _ = setup
    _zero_lr(agent, 1e-5)
    p0 = [opt.p.clone() for opt in agent.optimizers]
    n_log = len(agent.logs["IL_loss"])
    agent.train([None], 1, feedback="student")           # the reference's loader fills env as a side effect
    assert len(agent.logs["IL_loss"]) == n_log + 2
    assert all(not torch.equal(opt.p, q) for opt, q in zip(agent.optimizers, p0))
    assert all(torch.isfinite(opt.p).all() for opt in agent.optimizers)
    # the teacher half carries no NSS term: with frozen weights its logged loss equals a teacher rollout with nss_w 0
    _zero_lr(agent)
    agent.train([None], 1, feedback="student")
    l_teacher_half = agent.il_losses()[-2]
    for nss_w in (0, 0.1):
        _zero_lr(agent)
        agent.feedback, agent.loss = "teacher", 0
        agent.rollout(train_ml=0.2, nss_w=nss_w)
        if nss_w == 0:
            assert abs(float(agent.loss) - l_teacher_half) <= 1e-6 * abs(l_teacher_half), (float(agent.loss), l_teacher_half)
        else:
            assert abs(float(agent.loss) - l_teacher_half) > 1e-6 * abs(l_teacher_half)


def test_test_loop(setup):
    agent, env, _, _ = setup
    B = env.batch_size
    T = agent.args.max_action_len
    res = agent.test([None], env_name="val_seen", feedback="student")
    assert sorted(res) == ["m0__%d" % i for i in range(B)]
    # the path corners are those of rollout_greedy on the same BERT features
    lb, _ = agent._language_batch(env.batch)
    seq, lin = agent._lang_eval_forward(lb)
    _, geo_h, tidx_h = env._gather_poses(None, 0)
    gb = dict(corners_gps=torch.from_numpy(np.stack([np.asarray(it["gt_path_corners"][0]) for it in env.batch])).cuda(),
              directions=torch.tensor([float(it["angle"]) for it in env.batch], dtype=torch.float64).cuda(),
              geo=torch.from_numpy(geo_h).cuda(), tile_idx=torch.from_numpy(tidx_h).cuda(),
              lang_feature=seq.float(), cls_hidden=lin.float())
    prev, agent.renderer = agent.renderer, env.renderer
    try:
        paths = agent.trajectories(agent.rollout_greedy(gb, max_action_len=T))
    finally:
        agent.renderer = prev
    for i in range(B):
        tr = res["m0__%d" % i]
        assert len(tr["path_corners"]) == len(paths[i])
        for (c1, _), (c2, _) in zip(tr["path_corners"], paths[i]):
            assert np.array_equal(np.asarray(c1), np.asarray(c2))
        assert len(tr["gt_progress"]) == len(tr["progress"]) >= 1
    avg, _ = env.eval_metrics(res)
    assert set(("sr", "spl", "gp", "iou")) <= set(avg) and np.isfinite(avg["gp"])
    # teacher feedback: the human-attention scores, equal to the host formula on the same h_sali
    res_t = agent.test([None], env_name="val_seen", feedback="teacher")
    assert any("nss" in tr for tr in res_t.values())
    avg_h, _ = env.eval_metrics(res_t, human_att_eval=True)
    assert set(("HA_precision", "HA_recall", "nss")) <= set(avg_h)
    eng, att_t = agent._ctx_eval
    Tn = att_t.shape[0]
    sal = _upsample(eng.h_sali.reshape(-1, 64).contiguous()).view(Tn, B, 224, 224)
    gt = att_t.double() / 255
    for i in range(B):
        want = [_host_scores(sal[t, i], gt[t, i], 0) for t in range(Tn) if float(gt[t, i].sum()) > 0]
        tr = res_t["m0__%d" % i]
        got = list(zip(tr.get("human_att_performance", []), tr.get("nss", [])))
        assert len(got) == len(want), i
        for (pr, nss), (p2, r2, n2) in zip(got, want):
            assert abs(pr[0] - p2) <= 1e-9 * max(abs(p2), 1e-12) and abs(pr[1] - r2) <= 1e-9 * max(abs(r2), 1e-12)
            assert abs(nss - n2) <= 1e-9 * max(abs(n2), 1e-12)


def test_checkpoints(setup, tmp_path):
    agent, env, _, _ = setup
    B, T = env.batch_size, agent.args.max_action_len
    _zero_lr(agent, 1e-4)
    agent.train([None], 1, feedback="student")          # moments and step counts that differ from a fresh agent
    path = str(tmp_path / "ckpt" / "lstm.pt")
    agent.save(3, path)
    fresh = _make_agent(seed=5, resume_optimizer=True)
    assert fresh.load(path) == 3
    for a, b in ((agent.vision_model, fresh.vision_model), (agent.vln_model, fresh.vln_model),
                 (agent.lang_model, fresh.lang_model)):
        sa, sb = a.state_dict(), b.state_dict()
        assert sa.keys() == sb.keys()
        for k in sa:
            assert torch.equal(sa[k], sb[k]), k          # parameters and BatchNorm buffers
    for o1, o2 in zip(agent.optimizers, fresh.optimizers):
        assert torch.equal(o1.m, o2.m) and torch.equal(o1.v, o2.v) and o1.step_count == o2.step_count > 0
    # a bit-equal greedy rollout
    g = torch.Generator().manual_seed(3)
    _, geo_h, tidx_h = env._gather_poses(None, 0)
    gb = dict(corners_gps=torch.from_numpy(np.stack([np.asarray(it["gt_path_corners"][0]) for it in env.batch])).cuda(),
              directions=torch.tensor([float(it["angle"]) for it in env.batch], dtype=torch.float64).cuda(),
              geo=torch.from_numpy(geo_h).cuda(), tile_idx=torch.from_numpy(tidx_h).cuda(),
              lang_feature=torch.randn(B, 9, 768, generator=g).cuda(), cls_hidden=torch.rand(B, 49, generator=g).cuda())
    outs = []
    for a in (agent, fresh):
        prev, a.renderer = a.renderer, env.renderer
        try:
            outs.append({k: v.clone() for k, v in a.rollout_greedy(gb, max_action_len=T).items()})
        finally:
            a.renderer = prev
    for k in ("output", "corners", "directions", "ended"):
        assert torch.equal(outs[0][k], outs[1][k]), k
    # a torch-format optimiser state cannot be resumed
    states = torch.load(path, map_location="cuda")
    states["vln_model"]["optimizer"] = {"state": {}, "param_groups": []}
    bad = str(tmp_path / "torch_optim.pt")
    torch.save(states, bad)
    with pytest.raises(ValueError):
        fresh.load(bad)
    # the reference's layout: a vln_model entry holding a plain ViT_LSTM.state_dict(), trunk keys included
    plain = str(tmp_path / "plain.pt")
    torch.save({"vln_model": {"epoch": 1, "state_dict": agent.vln_model.state_dict()}}, plain)
    other = _make_agent(seed=9)
    assert other.load(plain) == 0
    sa, sb = agent.vln_model.state_dict(), other.vln_model.state_dict()
    assert any(k.startswith("vision_model.") for k in sa)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
