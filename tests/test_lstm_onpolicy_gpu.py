"""GPU: the LSTM agent's on-policy student-feedback training rollout (``NavCMTAgent.student_rollout_step``,
``rollout`` with ``args.on_policy_student``) and what it is built from -- ``avdn_add_dropout_f32_at`` and the
step-wise forward of ``ViT_LSTM``'s training engine (``begin`` / ``step`` / ``finish``, ``n_steps`` in ``loss`` /
``backward``)."""
import numpy as np
import pytest
import torch

from oracle import model_oracle as mo
from test_agent_dropin_gpu import BL, TR
from test_lstm_dropin_gpu import _env, _make_agent, _rel, _zero_lr
from test_lstm_train_gpu import _policy

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("with_b", [False, True])
def test_add_dropout_at_slices_match_the_whole_tensor(built_lib, p, with_b):
    from avdn_b200 import _lib
    T, n, seed, site = 7, 3 * 49 + 5, 987654321, 3000
    g = torch.Generator(device="cuda").manual_seed(4)
    a = torch.randn(T * n, device="cuda", generator=g)
    b = torch.randn(T * n, device="cuda", generator=g) if with_b else None
    whole = torch.full_like(a, float("nan"))
    _lib.call("avdn_add_dropout_f32", _lib.ptr(a), _lib.ptr(b), _lib.ptr(whole), T * n, p, seed, site)
    parts = torch.full_like(a, float("nan"))
    for t in range(T):
        _lib.call("avdn_add_dropout_f32_at", _lib.ptr(a[t * n:]), None if b is None else _lib.ptr(b[t * n:]),
                  _lib.ptr(parts[t * n:]), n, t * n, p, seed, site)
    assert torch.equal(whole, parts)
    s = a + (b if with_b else 0)
    if p == 0:
        assert torch.equal(whole, s)
    else:
        dropped = whole == 0
        assert 0.1 < float(dropped.float().mean()) < 0.3
        assert torch.allclose(whole[~dropped], s[~dropped] / (1 - p), rtol=1e-6, atol=0)


def test_add_dropout_at_rejects_bad_arguments(built_lib):
    from avdn_b200 import _lib
    h = _lib.lib()
    x = torch.zeros(64, device="cuda")
    assert h.avdn_add_dropout_f32_at(None, None, _lib.ptr(x), 4, 0, 0.2, 1, 3000, None) == -1
    assert "null" in _lib.last_error()
    assert h.avdn_add_dropout_f32_at(_lib.ptr(x), None, None, 4, 0, 0.2, 1, 3000, None) == -1
    assert h.avdn_add_dropout_f32_at(_lib.ptr(x), None, _lib.ptr(x), -1, 0, 0.2, 1, 3000, None) == -1
    assert h.avdn_add_dropout_f32_at(_lib.ptr(x), None, _lib.ptr(x), 4, -1, 0.2, 1, 3000, None) == -1
    assert h.avdn_add_dropout_f32_at(_lib.ptr(x), None, _lib.ptr(x), 4, 0, 1.0, 1, 3000, None) == -1
    assert h.avdn_add_dropout_f32_at(_lib.ptr(x), None, _lib.ptr(x), 0, 0, 0.2, 1, 3000, None) == 0


# ------------------------------------------------------------------------------------------------------ engine
# every buffer the backward reads, and the outputs
_FWD_BUFS = ("attn512", "wc", "e49", "e49_t", "e49d", "deg", "dir_emb", "gates_v", "gates_d", "c_v", "c_d", "cat2",
             "target", "attn", "act_in", "m0", "m1", "output", "s0", "h_sali")


def _inputs(B, T, L, seed):
    g = torch.Generator().manual_seed(seed)
    c = lambda x: x.cuda()
    frames = c(torch.randn(B, T, 512, 49, generator=g))
    deg = c(torch.randint(0, 360, (B, T), generator=g).float() + torch.rand(B, T, generator=g))
    cls = c(torch.relu(torch.randn(B, 49, generator=g)))
    lang = c(torch.randn(B, L, 768, generator=g))
    tgt = (c(torch.rand(T, B, 2, generator=g) * 2 - 1), c(torch.rand(T, B, generator=g)), c(torch.rand(T, B, generator=g)))
    att = torch.zeros(T, B, 224, 224, dtype=torch.uint8)
    att[:, ::2, 40:100, 60:140] = 255
    return frames, deg, cls, lang, tgt, c(att)


def _loss_backward(eng, tgt, att, n_steps, B, L):
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    k = n_steps if n_steps is not None else eng.T
    eng.loss(tgt[0][:k].contiguous(), tgt[1][:k].contiguous(), tgt[2][:k].contiguous(), att[:k].contiguous(), 0.1, 0,
             0.2 / B, loss, n_steps=n_steps)
    d_lang, d_cls = torch.zeros(B, L, 768, device="cuda"), torch.zeros(B, 49, device="cuda")
    d_frames = eng.backward(d_lang, d_cls, n_steps=n_steps)
    return float(loss), d_frames.clone(), d_lang, d_cls


@pytest.mark.parametrize("B", [4, 64])
@pytest.mark.parametrize("T", [1, 3, 10])
def test_stepwise_forward_matches_forward(built_lib, B, T):
    from avdn_b200.models.vln_model import _TrainEngine
    L, p, seed = 23, 0.2, 0x5EED1234
    m = _policy(train=True)
    frames, deg, cls, lang, tgt, att = _inputs(B, T, L, B + T)
    whole = _TrainEngine(m, B, L, T, "cuda", None)
    whole.forward(frames.view(B * T, 512, 49), deg, cls, lang, p, seed)
    steps = _TrainEngine(m, B, L, T, "cuda", None)
    steps.begin(cls, lang, p, seed)
    for t in range(T):
        out = steps.step(t, frames[:, t].contiguous(), deg[:, t].contiguous())
        assert torch.equal(out, whole.output[t]), t
    steps.finish()
    for name in _FWD_BUFS:
        assert torch.equal(getattr(steps, name), getattr(whole, name)), name
    assert torch.equal(steps._in[0], whole._in[0])                 # the frames the backward reads
    assert bool((whole.e49d == 0).any())                            # dropout was on
    r1, r2 = _loss_backward(whole, tgt, att, None, B, L), _loss_backward(steps, tgt, att, None, B, L)
    # the loss and the weight gradients of the frame attention are reduced with atomics: equal up to their order
    assert abs(r1[0] - r2[0]) <= 1e-12 * abs(r1[0])
    for a, b in zip(r1[1:], r2[1:]):
        assert _rel(b, a) <= 1e-6, _rel(b, a)
    for n in whole.G:
        assert _rel(steps.G[n], whole.G[n]) <= 1e-6, n


@pytest.mark.parametrize("B", [4, 64])
@pytest.mark.parametrize("T", [3, 10])
def test_loss_and_backward_over_a_prefix(built_lib, B, T):
    """``n_steps = k < T`` in an engine of T steps (forward over all T, or step-wise over k) equals an engine of k."""
    from avdn_b200.models.vln_model import _TrainEngine
    L, p, seed, k = 23, 0.2, 77, T // 2
    m = _policy(train=True)
    frames, deg, cls, lang, tgt, att = _inputs(B, T, L, 3 * B + T)
    short = _TrainEngine(m, B, L, k, "cuda", None)
    short.forward(frames[:, :k].reshape(B * k, 512, 49), deg[:, :k].contiguous(), cls, lang, p, seed)
    want = _loss_backward(short, tgt, att, None, B, L)
    full = _TrainEngine(m, B, L, T, "cuda", None)
    full.forward(frames.view(B * T, 512, 49), deg, cls, lang, p, seed)
    stepped = _TrainEngine(m, B, L, T, "cuda", None)
    stepped.begin(cls, lang, p, seed)
    for t in range(k):
        stepped.step(t, frames[:, t].contiguous(), deg[:, t].contiguous())
    stepped.finish()
    for eng in (full, stepped):
        loss, d_frames, d_lang, d_cls = _loss_backward(eng, tgt, att, k, B, L)
        assert abs(loss - want[0]) <= 1e-6 * abs(want[0]), (loss, want[0])
        d5 = d_frames.view(B, T, 512, 49)
        assert _rel(d5[:, :k], want[1].view(B, k, 512, 49)) <= 1e-6
        assert not d5[:, k:].any()
        assert _rel(d_lang, want[2]) <= 1e-6 and _rel(d_cls, want[3]) <= 1e-6
        for n in short.G:
            assert _rel(eng.G[n], short.G[n]) <= 1e-6, n


# ------------------------------------------------------------------------------------------------------- agent
@pytest.fixture(scope="module")
def setup(built_lib):
    agent = _make_agent()
    env, _, _ = _env()
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


def _on_policy_and_replay(agent, env):
    """The on-policy rollout, then ``train_rollout_step`` over the poses and targets it visited with the same dropout
    seeds.  Returns (on-policy loss, replay loss, gradients of both: policy, trunk, BERT)."""
    vln, lm = agent.vln_model, agent.lang_model
    batch, gt_paths = _student_batch(agent, env)
    prev, agent.renderer = agent.renderer, env.renderer
    try:
        _zero_lr(agent)
        s_v, s_l = getattr(vln, "_drop_step", 0), lm._drop_step
        loss = agent.student_rollout_step(batch, gt_paths, nss_w=0.1, train_ml=0.2, step=False, sync_loss=True)
        g_on = [o.g.clone() for o in agent.optimizers]
        vln._drop_step, lm._drop_step = s_v, s_l
        _zero_lr(agent)
        replay = agent.train_rollout_step(agent._last_rollout["batch"], sync_loss=True, step=False, nss_w=0.1,
                                          train_ml=0.2, bn_per_step=True)
        g_re = [o.g.clone() for o in agent.optimizers]
    finally:
        agent.renderer = prev
    return loss, replay, g_on, g_re


@pytest.mark.parametrize("dropout", [False, True])
def test_on_policy_equals_teacher_forced_replay(setup, dropout):
    agent, env = setup
    agent.args.no_dropout = not dropout
    try:
        loss, replay, g_on, g_re = _on_policy_and_replay(agent, env)
    finally:
        agent.args.no_dropout = True
    lr = agent._last_rollout
    assert 1 <= lr["steps"] <= agent.args.max_action_len
    assert abs(loss - replay) <= 1e-6 * abs(replay), (loss, replay)
    policy, trunk, bert = range(3)
    for k in (policy, bert):
        assert float(g_re[k].abs().sum()) > 0
        assert _rel(g_on[k], g_re[k]) < 1e-5, (k, _rel(g_on[k], g_re[k]))
    # the trunk: per-step passes over the same views, up to the order of the trunk backward's atomic reductions
    assert _rel(g_on[trunk], g_re[trunk]) < 1e-5, _rel(g_on[trunk], g_re[trunk])


def test_poses_are_the_train_mode_decisions(setup):
    """``rollout`` with ``on_policy_student``: the oracle simulator driven by the recorded train-mode outputs
    reproduces the visited poses and stop flags, and the trajectory dicts log exactly those outputs and poses."""
    agent, env = setup
    B, T = env.batch_size, agent.args.max_action_len
    agent.args.on_policy_student, agent.args.no_dropout = True, False
    try:
        _zero_lr(agent)
        agent.loss, agent.feedback, agent.env_name = 0, "student", "train"
        n_log = len(agent.logs["IL_loss"])
        traj = agent.rollout(train_ml=0.2, nss_w=0.1)
    finally:
        agent.args.on_policy_student, agent.args.no_dropout = False, True
    lr = agent._last_rollout
    steps = lr["steps"]
    out = lr["output"].cpu().numpy()
    corners, dirs = lr["corners"].cpu().numpy(), lr["directions"].cpu().numpy()
    ended = lr["ended"].cpu().numpy().astype(bool)
    c = np.stack([np.asarray(it["gt_path_corners"][0]) for it in env.batch])
    d = np.array([it["angle"] for it in env.batch], dtype=np.float64)
    e = np.zeros(B, dtype=bool)
    bounds = np.tile(np.concatenate([BL, TR]), (B, 1))
    for t in range(steps):
        assert np.allclose(corners[t], c, rtol=0, atol=1e-9) and np.allclose(dirs[t], d, rtol=0, atol=1e-9), t
        c, d, e, *_ = mo.waypoint_step(out[t], c, bounds, d, e, 0.25, t == T - 1)
        assert np.array_equal(ended[t], e), t
    assert np.allclose(corners[steps], c, rtol=0, atol=1e-9) and np.allclose(dirs[steps], d, rtol=0, atol=1e-9)
    if steps < T:
        assert e.all()
    assert len(agent.logs["IL_loss"]) == n_log + 1
    for i, tr in enumerate(traj):
        alive = [t for t in range(steps) if t == 0 or not ended[t - 1, i]]
        assert len(tr["actions"]) == len(tr["progress"]) == len(tr["gt_actions"]) == len(alive)
        for k, t in enumerate(alive):
            o = out[t, i]
            m = max(abs(float(o[0])), abs(float(o[1])), 1.0)
            assert np.array_equal(tr["actions"][k][0], np.array([o[0] / m, o[1] / m], dtype=np.float32))
            assert tr["progress"][k] == float(o[3])
        moved = [t for t in range(steps) if not ended[t, i]]
        assert len(tr["path_corners"]) == 1 + len(moved)
        for (pc, pd), t in zip(tr["path_corners"][1:], moved):
            assert np.array_equal(pc, corners[t + 1, i]) and pd == float(dirs[t + 1, i])


def test_early_exit_after_the_first_step(setup):
    agent, env = setup
    vm = agent.vision_model
    bias = agent.vln_model.decoder_2_action_full[6].bias
    nbt = [k for k in vm.state_dict() if k.endswith("num_batches_tracked")][0]
    with torch.no_grad():
        old = float(bias[3])
        bias[3] = 100.0                                  # progress far above 0.25: every sample stops at step 0
    try:
        n0 = int(vm.state_dict()[nbt])
        loss, replay, _, _ = _on_policy_and_replay(agent, env)
        steps = agent._last_rollout["steps"]
        n1 = int(vm.state_dict()[nbt])
    finally:
        with torch.no_grad():
            bias[3] = old
    assert steps == 1
    assert n1 - n0 == 2                                  # one trunk pass on-policy, then the replay's one
    assert agent._last_rollout["ended"].shape[0] == 1 and bool(agent._last_rollout["ended"].all())
    assert abs(loss - replay) <= 1e-6 * abs(replay), (loss, replay)


def test_train_loop_on_policy(setup):
    agent, env = setup
    agent.args.on_policy_student = True
    try:
        _zero_lr(agent, 1e-5)
        p0 = [opt.p.clone() for opt in agent.optimizers]
        n_log = len(agent.logs["IL_loss"])
        agent.train([None], 1, feedback="student")
        assert len(agent.logs["IL_loss"]) == n_log + 2
        assert all(not torch.equal(opt.p, q) for opt, q in zip(agent.optimizers, p0))     # policy, trunk, BERT
        assert all(torch.isfinite(opt.p).all() for opt in agent.optimizers)
        assert all(np.isfinite(agent.il_losses()[-2:]))
        agent.args.bn_per_step = False
        with pytest.raises(ValueError):
            agent.train([None], 1, feedback="student")
    finally:
        agent.args.on_policy_student = False
        if hasattr(agent.args, "bn_per_step"):
            del agent.args.bn_per_step
