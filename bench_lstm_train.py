"""Teacher-forced training rollout of the LSTM baseline (``run_lstm_haa.sh``: lr 1e-5, adamW, nss_w 0) on one GPU:
B = 64 episodes x T = 10 steps, 250-token dialog, views rendered from a 3000x3000 tile.  Prints one JSON line.

A rollout = render the 640 views -> Darknet trunk in train mode (one pass over B*T views) -> ViT_LSTM's 10 recurrent
steps with train-mode dropout and the loss of every step -> backward through time -> trunk backward -> clip + AdamW
on both models (``NavCMTAgent.train_rollout_step``).  Before every warm-up and timed rollout the weights, AdamW moments
and step counts, the trunk's BatchNorm statistics and the dropout counter are restored, so every rollout is the same
training step.  The stage breakdown comes from a separate rollout built from the same pieces with CUDA events between
them.  The stock-torch arm runs the policy part only (the CPU reference rollout with autograd, on CUDA tensors, i.e.
cuBLAS) on the features and dropout masks of our last rollout, and its loss is compared with ours.

    python bench_lstm_train.py [--steps 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import types

import numpy as np
import torch

B, T, L, SIZE = 64, 10, 250, 3000


def teacher_batch(dev, seed=0):
    """Poses along a straight ground-truth path from ``bench_rollout``'s start poses, random targets."""
    from bench_rollout import synthetic_rollout_batch
    sb = synthetic_rollout_batch(B, L, seed, size=SIZE)
    c0, geo = sb["corners_gps"].numpy(), sb["geo"].numpy()
    step = np.array([0.0002, -0.00015])
    poses = np.stack([c0 + k * step for k in range(T)], 1)                            # [B,T,4,2] (lat, lng)
    g = geo[:, None, None, :]
    px = np.stack([np.rint((poses[..., 1] - g[..., 1]) / g[..., 4]), np.rint((g[..., 2] - poses[..., 0]) / g[..., 4])], -1)
    gen = torch.Generator().manual_seed(seed)
    deg = (sb["directions"].float()[:, None] + torch.arange(T).float() * 5) % 360
    return dict(corners_px=torch.from_numpy(px.astype(np.int32)).to(dev), tile_idx=None,
                lang_feature=sb["lang_feature"].to(dev), cls_hidden=sb["cls_hidden"].to(dev), directions=deg.to(dev),
                gt_xy=(torch.rand(B, T, 2, generator=gen) * 2 - 1).to(dev), gt_alt=torch.rand(B, T, generator=gen).to(dev),
                gt_prog=torch.rand(B, T, generator=gen).to(dev))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:                          # the measurement stands; the card is then reported as unknown
        return torch.cuda.get_device_name(0), f"unknown ({type(e).__name__})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lstm_train.py needs a CUDA device")
    from avdn_b200 import _lib
    from avdn_b200 import agent_common as ac
    from avdn_b200.utils import synthetic as syn
    from avdn_b200.xview_lstm.agent import NavCMTAgent
    dev = "cuda"
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(syn.yolov3_trunk_cfg())
    torch.manual_seed(0)
    agent = NavCMTAgent(types.SimpleNamespace(darknet_model_file=f.name, darknet_weight_file=None, max_action_len=T,
                                              lr=1e-5, nss_w=0.0, nss_r=0, ml_weight=0.2), device=dev)
    os.unlink(f.name)
    agent.renderer.add_map("tile", syn.synthetic_tile(seed=0, size=SIZE), None)
    batch = teacher_batch(dev)
    state = [t for o in agent.optimizers for t in (o.p, o.m, o.v)] + list(agent.vision_model.buffers())
    snap = ([t.clone() for t in state], [o.step_count for o in agent.optimizers],
            getattr(agent.vln_model, "_drop_step", 0))

    def restore():
        for t, t0 in zip(state, snap[0]):
            t.copy_(t0)
        for o, n in zip(agent.optimizers, snap[1]):
            o.step_count = n
        agent.vln_model._drop_step = snap[2]

    for _ in range(a.warmup):
        restore()
        agent.train_rollout_step(batch)
    torch.cuda.synchronize()
    times = []
    for _ in range(a.steps):
        restore()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        agent.train_rollout_step(batch)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ours_loss = float(agent.loss_total.item())
    teng, tengs, eng, tb = agent._ctx
    frames = tb["frames"].view(B, T, 512, 49).clone()
    p, seed = eng.p, eng.seed

    # ---- stage breakdown: one more rollout, the same pieces with events between them ----
    restore()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
    vln, vm = agent.vln_model, agent.vision_model
    deg, lang, cls = batch["directions"], batch["lang_feature"], batch["cls_hidden"]
    tr = lambda x: x.float().transpose(0, 1).contiguous()
    for o in agent.optimizers:
        o.zero_grad()
    ev[0].record()
    x, _, _ = ac.render_rollout_views(agent, batch, B * T, tb["x"], tb["att"])
    ev[1].record()
    vln.train()
    vm.train()
    teng, tengs, l0, _ = ac.rollout_trunk_forward(agent, x, B, T, tb["frames"], False)
    ev[2].record()
    eng.forward(tb["frames"].view(B * T, 512, 49), deg, cls, lang, *vln.dropout_config())
    agent.loss_total.zero_()
    eng.loss(tr(batch["gt_xy"]), tr(batch["gt_alt"]), tr(batch["gt_prog"]), None, 0.0, 0, 0.2 / B, agent.loss_total)
    ev[3].record()
    eng.backward()
    ev[4].record()
    ac.rollout_trunk_backward(agent, teng, tengs, l0, eng.d_frames, B, T)
    ev[5].record()
    for o in agent.optimizers:
        o.step()
    ev[6].record()
    torch.cuda.synchronize()
    names = ["render", "trunk_forward", "policy_forward_and_loss", "backward_through_time", "trunk_backward",
             "optimiser"]
    breakdown = {n: round(ev[i].elapsed_time(ev[i + 1]), 3) for i, n in enumerate(names)}

    # ---- stock torch, policy part only: the reference rollout with autograd on CUDA tensors ----
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests"))
    import lstm_rollout_reference as ref
    from avdn_b200.models.vln_model import SITE_INPUT, SITE_FC, SITE_DEC

    def keep(n, site):
        out = torch.empty(n, device=dev)
        _lib.call("avdn_dropout_keep_scale", _lib.ptr(out), n, p, seed, site)
        return out

    inp, fc = keep(T * B * 49, SITE_INPUT).view(T, B, 49), keep(T * B * 128, SITE_FC).view(T, B, 128)
    drop = [dict(input=inp[t], fc=fc[t], h0=keep(B * 256, SITE_DEC + 2 * t).view(B, 256),
                 h1=keep(B * 32, SITE_DEC + 2 * t + 1).view(B, 32)) for t in range(T)]
    restore()
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in agent.vln_model.used_parameters().items()}
    torch_ms = []
    for i in range(2):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        tot = ref.rollout_loss(sd, frames, deg, cls, lang, batch["gt_xy"], batch["gt_alt"], batch["gt_prog"],
                               train_ml=0.2, drop=drop)
        tot.backward()
        s1.record()
        s1.synchronize()
        torch_ms.append(s0.elapsed_time(s1))
    torch_loss = float(tot.detach())
    name, power = card()
    ms = float(np.median(times))
    print(json.dumps({
        "workload": "lstm_haa teacher-forced training rollout, B=64 x T=10 steps, L=250, views rendered from a "
                    "3000x3000 tile, train-mode trunk over 640 views, dropout 0.2, clip 40 + AdamW",
        "gpu": name, "power_limit": power, "steps": a.steps, "warmup": a.warmup,
        "ms_per_rollout": round(ms, 3), "ms_per_rollout_all": [round(t, 3) for t in times],
        "episodes_per_s": round(B / ms * 1e3, 2), "breakdown_ms": breakdown,
        "policy_ms": round(breakdown["policy_forward_and_loss"] + breakdown["backward_through_time"], 3),
        "stock_torch_policy_ms": round(torch_ms[-1], 3), "loss": ours_loss, "stock_torch_loss": torch_loss,
        "loss_rel_diff": abs(ours_loss - torch_loss) / max(abs(torch_loss), 1e-30)}))


if __name__ == "__main__":
    main()
