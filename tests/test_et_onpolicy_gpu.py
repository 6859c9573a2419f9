"""GPU: the ET agent's on-policy student-feedback training rollout (``NavCMTAgent.student_rollout_step``, ``rollout``
with ``args.on_policy_student``): per step a train-mode trunk pass, the ET in train mode over the history, the step's
loss and backward, and the simulator moved by that same train-mode prediction (src/xview_et/agent.py:580-760).

The reference point is ``train_rollout_step`` replayed over the poses, targets and history lengths the on-policy
rollout recorded, with the same dropout seeds: it runs the same kernels in the same per-step order, so the per-step
outputs are equal bit for bit and the losses and gradients up to the order of atomic reductions."""
import os
import tempfile
import types

import numpy as np
import pytest
import torch

from oracle import model_oracle as mo
from oracle import teacher_oracle as to
from oracle import warp_oracle as wo
from test_agent_dropin_gpu import BL, SIZE, TR, _items, _Tok

pytestmark = pytest.mark.gpu

B, T, NSS_W, ML = 4, 4, 0.1, 0.2


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _zero_lr(agent, lr=0.0):
    for opt in agent.optimizers:
        opt.lr, opt.wd = lr, 0.0
        opt.zero_grad()


@pytest.fixture(scope="module")
def setup(built_lib):
    from transformers import BertConfig
    from avdn_b200.env import ANDHNavBatch
    from avdn_b200.models.bert import CustomBERTModel
    from avdn_b200.xview_et.agent import NavCMTAgent
    V = 400
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(mo.yolov3_trunk_cfg())
    args = types.SimpleNamespace(demb=768, encoder_heads=12, encoder_layers=2, dropout_transformer_encoder=0.1,
                                 num_input_actions=1, dropout_emb=0.0, darknet_model_file=f.name, darknet_weight_file=None,
                                 lr=1e-5, nss_w=NSS_W, nss_r=0, ml_weight=ML, teacher_weight=1.0, max_action_len=T,
                                 no_dropout=True, train_val_on_full=False, vision_only=False, no_direction=False,
                                 optim="adamW")
    torch.manual_seed(0)
    agent = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    agent.tokenizer = _Tok(V)
    agent.attach_lang_model(CustomBERTModel(BertConfig(num_hidden_layers=1, vocab_size=V, max_position_embeddings=64)))
    env = ANDHNavBatch(batch_size=B, device="cuda")
    env.map_batch["m0"] = wo.synthetic_tile(seed=4, size=SIZE)
    env.attention_map_batch["m0"] = wo.synthetic_attention_tile(seed=4, size=SIZE)
    env.batch = _items(B, 7)
    agent.env = env
    return agent, env


def _student_batch(agent, env):
    """``student_rollout_step``'s input for the environment's batch: the tokenised dialogs and the start poses."""
    items = env.batch
    env._sync_maps()
    lb, _ = agent._language_batch(items)
    _, geo_h, tidx_h = env._gather_poses(None, 0)
    batch = dict(lb, corners_gps=torch.from_numpy(np.stack([np.asarray(it["gt_path_corners"][0]) for it in items])).cuda(),
                 directions=torch.tensor([float(it["angle"]) for it in items], dtype=torch.float64).cuda(),
                 geo=torch.from_numpy(geo_h).cuda(), tile_idx=torch.from_numpy(tidx_h).cuda())
    return batch, [np.asarray(it["gt_path_corners"], dtype=np.float64) for it in items]


def _on_policy(agent, env):
    """One on-policy rollout on the environment's batch.  Returns (loss, per-step outputs, arena gradients, the
    dropout counters of the ET and BERT before the rollout)."""
    batch, gt_paths = _student_batch(agent, env)
    seeds = (getattr(agent.vln_model, "_drop_step", 0), getattr(agent.lang_model, "_drop_step", 0))
    prev, agent.renderer = agent.renderer, env.renderer
    try:
        _zero_lr(agent)
        outs = []
        loss = agent.student_rollout_step(batch, gt_paths, nss_w=NSS_W, train_ml=ML, step=False, sync_loss=True,
                                          collect=outs)
    finally:
        agent.renderer = prev
    return loss, outs, [o.g.clone() for o in agent.optimizers], seeds


def _replay(agent, env, seeds):
    """``train_rollout_step`` over the recorded batch of the last on-policy rollout with the same dropout seeds."""
    agent.vln_model._drop_step, agent.lang_model._drop_step = seeds
    prev, agent.renderer = agent.renderer, env.renderer
    try:
        _zero_lr(agent)
        outs = []
        loss = agent.train_rollout_step(agent._last_rollout["batch"], sync_loss=True, step=False, nss_w=NSS_W,
                                        train_ml=ML, bn_per_step=True, collect=outs)
    finally:
        agent.renderer = prev
    return loss, outs, [o.g.clone() for o in agent.optimizers]


def _check_replay(on, re):
    (loss, outs, g_on, _), (loss_r, outs_r, g_re) = on, re
    assert abs(loss - loss_r) <= 1e-6 * abs(loss_r), (loss, loss_r)
    assert len(outs) == len(outs_r)
    for t, (a, b) in enumerate(zip(outs, outs_r)):
        assert torch.equal(a, b), t
    # ET, trunk, BERT: equal up to the order of atomic reductions.  The BERT backward is the noisiest: two runs of
    # the same replay on the same inputs have been seen to differ by 2e-5 in its arena (B200), so it gets 1e-4.
    for k, tol in enumerate((1e-5, 1e-5, 1e-4)):
        assert float(g_re[k].abs().sum()) > 0 and float(g_on[k].abs().sum()) > 0, k
        assert _rel(g_on[k], g_re[k]) < tol, (k, _rel(g_on[k], g_re[k]))


@pytest.mark.parametrize("dropout", [False, True])
def test_on_policy_equals_teacher_forced_replay(setup, dropout):
    agent, env = setup
    agent.args.no_dropout = not dropout
    try:
        on = _on_policy(agent, env)
        lr = agent._last_rollout
        assert 1 <= lr["steps"] <= T
        assert torch.equal(torch.stack(on[1]), lr["output"])
        re = _replay(agent, env, on[3])
    finally:
        agent.args.no_dropout = True
    _check_replay(on, re)


def test_poses_are_the_train_mode_decisions(setup):
    """``rollout`` with ``on_policy_student``: the oracle simulator driven by the recorded train-mode outputs
    reproduces the visited poses and stop flags; ``lenths`` are the alive counts; the trajectory dicts log exactly
    those outputs and poses."""
    agent, env = setup
    agent.args.on_policy_student, agent.args.no_dropout = True, False
    try:
        _zero_lr(agent)
        agent.loss, agent.feedback, agent.env_name = 0, "student", "train"
        n_log = len(agent.logs["IL_loss"])
        traj = agent.rollout(train_ml=ML, nss_w=NSS_W)
    finally:
        agent.args.on_policy_student, agent.args.no_dropout = False, True
    lr = agent._last_rollout
    steps = lr["steps"]
    out = lr["output"].cpu().numpy()
    corners, dirs = lr["corners"].cpu().numpy(), lr["directions"].cpu().numpy()
    ended = lr["ended"].cpu().numpy().astype(bool)
    assert corners.shape == (steps + 1, B, 4, 2) and dirs.shape == (steps + 1, B) and out.shape == (steps, B, 4)
    c = np.stack([np.asarray(it["gt_path_corners"][0]) for it in env.batch])
    d = np.array([it["angle"] for it in env.batch], dtype=np.float64)
    e = np.zeros(B, dtype=bool)
    bounds = np.tile(np.concatenate([BL, TR]), (B, 1))
    for t in range(steps):
        assert np.allclose(corners[t], c, rtol=0, atol=1e-9) and np.allclose(dirs[t], d, rtol=0, atol=1e-9), t
        c, d, e, *_ = mo.waypoint_step(out[t], c, bounds, d, e, 0.5, t == T - 1)
        assert np.array_equal(ended[t], e), t
    assert np.allclose(corners[steps], c, rtol=0, atol=1e-9) and np.allclose(dirs[steps], d, rtol=0, atol=1e-9)
    if steps < T:
        assert e.all()                                   # the loop stopped after the step at which all had ended
    if steps > 1:
        assert not ended[steps - 2].all()
    alive = np.ones((steps, B), dtype=bool)
    alive[1:] = ~ended[:steps - 1]
    lenths = np.asarray(lr["lenths"])                    # [B, steps]
    assert np.array_equal(lenths, np.cumsum(alive, axis=0).T)
    assert np.array_equal(lenths, np.asarray(lr["batch"]["lenths"]))
    for t in range(steps):
        assert lenths[:, t].max() == t + 1 and lenths[:, t].min() >= 1
    assert len(agent.logs["IL_loss"]) == n_log + 1
    assert abs(float(agent.loss) - agent.il_losses()[-1]) < 1e-9
    for i, tr in enumerate(traj):
        steps_i = [t for t in range(steps) if alive[t, i]]
        assert len(tr["actions"]) == len(tr["progress"]) == len(tr["gt_actions"]) == len(steps_i)
        for k, t in enumerate(steps_i):
            o = out[t, i]
            m = max(abs(float(o[0])), abs(float(o[1])), 1.0)
            assert np.array_equal(tr["actions"][k][0], np.array([o[0] / m, o[1] / m], dtype=np.float32))
            assert tr["progress"][k] == float(o[3])
        moved = [t for t in range(steps) if not ended[t, i]]
        assert len(tr["path_corners"]) == 1 + len(moved)
        for (pc, pd), t in zip(tr["path_corners"][1:], moved):
            assert np.array_equal(pc, corners[t + 1, i]) and pd == float(dirs[t + 1, i])


def test_targets_are_the_teacher_at_the_visited_poses(setup):
    agent, env = setup
    agent.args.no_dropout = False
    try:
        _on_policy(agent, env)
    finally:
        agent.args.no_dropout = True
    lr = agent._last_rollout
    steps = lr["steps"]
    corners = lr["corners"][:steps]
    ended_before = torch.zeros((steps, B), dtype=torch.uint8, device="cuda")
    ended_before[1:] = lr["ended"][:steps - 1]
    gts = [np.asarray(it["gt_path_corners"], dtype=np.float64) for it in env.batch]
    xy, alt, prog = agent.teacher_action(corners.reshape(steps * B, 4, 2), [gts[k % B] for k in range(steps * B)],
                                         ended_before.reshape(-1), feedback="student")
    assert torch.equal(xy.view(steps, B, 2), lr["tgt_xy"])
    assert torch.equal(alt.view(steps, B), lr["tgt_alt"]) and torch.equal(prog.view(steps, B), lr["tgt_prog"])
    c, eb = corners.cpu().numpy(), ended_before.cpu().numpy()
    tx, ta, tp = lr["tgt_xy"].cpu().numpy(), lr["tgt_alt"].cpu().numpy(), lr["tgt_prog"].cpu().numpy()
    for t in range(steps):
        for i in range(B):
            x_o, a_o, p_o = to.teacher_action(c[t, i], env.batch[i]["gt_path_corners"], bool(eb[t, i]),
                                              feedback="student")
            assert np.allclose(tx[t, i], x_o, rtol=0, atol=1e-5), (t, i)
            assert abs(ta[t, i] - a_o) <= 1e-5 and abs(tp[t, i] - p_o) <= 1e-5, (t, i)
    b = lr["batch"]
    assert torch.equal(b["gt_xy"], lr["tgt_xy"].transpose(0, 1)) and torch.equal(b["gt_prog"], lr["tgt_prog"].t())


def test_early_exit_after_the_first_step(setup):
    agent, env = setup
    vm = agent.vision_model
    bias = agent.vln_model.decoder_2_action_full[6].bias
    nbt = [k for k in vm.state_dict() if k.endswith("num_batches_tracked")][0]
    with torch.no_grad():
        old = float(bias[3])
        bias[3] = 100.0                                  # progress far above 0.5: every sample stops at step 0
    try:
        n0 = int(vm.state_dict()[nbt])
        on = _on_policy(agent, env)
        n1 = int(vm.state_dict()[nbt])
        lr = agent._last_rollout
        re = _replay(agent, env, on[3])
    finally:
        with torch.no_grad():
            bias[3] = old
    assert lr["steps"] == 1 and len(on[1]) == 1
    assert n1 - n0 == 1                                  # exactly one trunk pass
    assert lr["ended"].shape[0] == 1 and bool(lr["ended"].all())
    assert lr["corners"].shape[0] == 2 and lr["batch"]["corners_px"].shape[1] == 1
    _check_replay(on, re)


def test_no_direction(setup):
    agent, env = setup
    agent.args.no_direction, agent.args.no_dropout = True, False
    try:
        on = _on_policy(agent, env)
        dirs = agent._last_rollout["batch"]["directions"]
        re = _replay(agent, env, on[3])
    finally:
        agent.args.no_direction, agent.args.no_dropout = False, True
    assert dirs.shape == (B, agent._last_rollout["steps"], 2) and not dirs.any()
    _check_replay(on, re)


def test_train_loop_on_policy(setup):
    agent, env = setup
    agent.args.on_policy_student = True
    try:
        _zero_lr(agent, 1e-5)
        p0 = [opt.p.clone() for opt in agent.optimizers]
        n_log = len(agent.logs["IL_loss"])
        agent.train([None], 1, feedback="student")
        assert len(agent.logs["IL_loss"]) == n_log + 2
        assert all(not torch.equal(opt.p, q) for opt, q in zip(agent.optimizers, p0))     # ET, trunk, BERT
        assert all(torch.isfinite(opt.p).all() for opt in agent.optimizers)
        assert all(np.isfinite(agent.il_losses()[-2:]))
        agent.args.bn_per_step = False
        with pytest.raises(ValueError):
            agent.train([None], 1, feedback="student")
        batch, gt_paths = _student_batch(agent, env)
        n_log = len(agent.logs["IL_loss"])
        with pytest.raises(ValueError):
            agent.student_rollout_step(batch, gt_paths)
        assert len(agent.logs["IL_loss"]) == n_log
    finally:
        agent.args.on_policy_student = False
        if hasattr(agent.args, "bn_per_step"):
            del agent.args.bn_per_step
