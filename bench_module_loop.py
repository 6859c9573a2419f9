"""The LSTM baseline's training iteration written with module calls only -- the reference's loop shape: T = 10 steps of
``ViT_LSTM.forward`` on a ``Darknet`` (one train-mode trunk pass per step, every pass pending until the single
backward), the loss in torch, one ``backward()`` -- against the agent's fused ``train_rollout_step(bn_per_step=True)``
on the same batch.  B = 4 and B = 64 episodes, 250-token dialogs, random views, fixation maps on half the samples,
dropout on in both.  Neither arm takes the optimiser step; both zero the gradient arenas first.

Per batch size and arm: the median, min and max of the synchronised iteration time, the growth of
``torch.cuda.memory_allocated`` over the arm's first iterations (the engines it creates), and
``torch.cuda.max_memory_allocated`` over the timed iterations of both arms.  The arms alternate, each warmed up
first.  Prints one JSON line with the GPU name and power limit.

    python bench_module_loop.py [--steps 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import json
import os
import tempfile
import time
import types

import numpy as np
import torch

from bench_lstm_loop import card

T, L = 10, 250
ARMS = ("module_loop", "agent_fused")
PI_REF = 3.14159


def _ang(v0, v1):
    return ((torch.atan2(v0, v1) / PI_REF + 2) / 2) % 1


def step_loss(out, pred, gt_xy, gt_alt, gt_prog, att, nss_w, train_ml):
    """The reference's loss of one step over the batch (src/xview_lstm/agent.py:636,663-685,883-885, jitter 0) in
    torch: the MSE terms and the angular term of every sample, nss_w x NSS of the samples with fixations."""
    B = out.shape[0]
    ml = ((out[:, :2] - gt_xy) ** 2).sum() + ((_ang(out[:, 0], out[:, 1]) - _ang(gt_xy[:, 0], gt_xy[:, 1])) ** 2).sum()
    ml = ml + ((out[:, 2] - gt_alt) ** 2).sum() + ((out[:, 3] - gt_prog) ** 2).sum()
    s = pred.view(B, -1)
    fix = att.view(B, -1).float() / 255
    has = fix.sum(1) > 0
    n_sal = (s - s.mean(1, keepdim=True)) / s.std(1, keepdim=True)
    nss = -(n_sal * fix).sum(1) / (fix.sum(1) + 0.001)
    ml = ml + nss_w * torch.where(has, nss, torch.zeros_like(nss)).sum()
    return ml * train_ml / B


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, nargs="+", default=[4, 64])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_module_loop.py needs a CUDA device")
    from avdn_b200.utils import synthetic as syn
    from avdn_b200.xview_lstm.agent import NavCMTAgent
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(syn.yolov3_trunk_cfg())
    args = types.SimpleNamespace(darknet_model_file=f.name, darknet_weight_file=None, max_action_len=T, lr=1e-5,
                                 nss_w=1.0, nss_r=0, ml_weight=0.2, optim="adamW", bn_per_step=True)
    torch.manual_seed(0)
    agent = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    vln = agent.vln_model
    out = {"workload": f"lstm training iteration without the optimiser step: T={T} steps, L={L} tokens, per-step "
                       "train-mode trunk passes, dropout on; module calls + torch loss + one backward vs the agent's "
                       "fused train_rollout_step(bn_per_step=True); alternated",
           "steps": a.steps, "warmup": a.warmup}
    for B in a.batch:
        g = torch.Generator(device="cuda").manual_seed(B)
        dev = "cuda"
        x = torch.zeros(B * T, 224, 224, 4, device=dev)
        x[..., :3] = torch.randn(B * T, 224, 224, 3, device=dev, generator=g)
        x = x.to(torch.bfloat16)
        att = torch.zeros(B * T, 224, 224, dtype=torch.uint8, device=dev)
        att.view(B, T, 224, 224)[::2, :, 40:100, 60:140] = 255
        batch = dict(images=x, att=att, lang_feature=torch.randn(B, L, 768, device=dev, generator=g),
                     cls_hidden=torch.relu(torch.randn(B, 49, device=dev, generator=g)),
                     directions=torch.randint(0, 360, (B, T), device=dev, generator=g).float(),
                     gt_xy=torch.rand(B, T, 2, device=dev, generator=g) * 2 - 1,
                     gt_alt=torch.rand(B, T, device=dev, generator=g), gt_prog=torch.rand(B, T, device=dev, generator=g))
        x5, att5 = x.view(B, T, 224, 224, 4), att.view(B, T, 224, 224)
        ims = [x5[:, t, ..., :3].permute(0, 3, 1, 2).float().contiguous() for t in range(T)]

        def module_loop():
            for opt in agent.optimizers:
                opt.zero_grad()
            vln.train()
            state, total = (None,) * 4, 0
            for t in range(T):
                h, c, hh, cc, o, pred = vln(batch["directions"][:, t:t + 1], ims[t], None, batch["cls_hidden"],
                                            batch["lang_feature"], *state)
                state = (h, c, hh, cc)
                total = total + step_loss(o, pred, batch["gt_xy"][:, t], batch["gt_alt"][:, t],
                                          batch["gt_prog"][:, t], att5[:, t], args.nss_w, args.ml_weight)
            total.backward()

        def agent_fused():
            agent.train_rollout_step(batch, step=False, bn_per_step=True)

        fns = dict(module_loop=module_loop, agent_fused=agent_fused)

        def timed(fn):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3

        grown = {}
        for arm in ARMS:
            torch.cuda.synchronize()
            m0 = torch.cuda.memory_allocated()
            for _ in range(a.warmup):
                fns[arm]()
            torch.cuda.synchronize()
            grown[arm] = torch.cuda.memory_allocated() - m0
        torch.cuda.reset_peak_memory_stats()
        ms = {arm: [] for arm in ARMS}
        for i in range(a.steps):
            for arm in (ARMS if i % 2 == 0 else ARMS[::-1]):
                ms[arm].append(timed(fns[arm]))
        out[f"B{B}_max_memory_allocated_mb"] = round(torch.cuda.max_memory_allocated() / 2 ** 20, 1)
        for arm in ARMS:
            v = np.array(ms[arm])
            out[f"B{B}_{arm}_ms"] = round(float(np.median(v)), 3)
            out[f"B{B}_{arm}_ms_min_max"] = [round(float(v.min()), 3), round(float(v.max()), 3)]
            out[f"B{B}_{arm}_engine_memory_mb"] = round(grown[arm] / 2 ** 20, 1)
    out["gpu"], out["power_limit"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
