"""The ET agent's student-feedback training two ways, alternated in one process: the default two-pass path (a no-grad
eval-mode greedy rollout fixes the poses -- CUDA-graph trunk, incremental decoder -- then a teacher-forced training
rollout over them) and the on-policy path (``args.on_policy_student``: one train-mode pass whose predictions move the
simulator, ``student_rollout_step``).  Workload: B = 64 episodes, ``max_action_len`` 10, a 2-layer, 12-head,
768-wide ET with encoder dropout 0.1, BERT-base trained in the loop, dialogs of about 250 tokens, views rendered from a
3000x3000 synthetic tile, ``bn_per_step`` and ``nss_w`` 1.0.  Prints one JSON line.

* ``student_rollout_ms``: one ``rollout(train_ml=0.2, nss_w=args.nss_w)`` under student feedback (forward, loss and
  backward of the student half; no optimiser step).
* ``train_iteration_ms``: one ``train(loader, 1, 'student')`` iteration (teacher half + student half + AdamW).
Every timing is synchronised at both ends; the arms alternate, each warmed up first.  Per arm: the median, min and max,
the rollout's step count and its host reads of the stop flags inside the step loop.

    python bench_et_onpolicy.py [--steps 5] [--warmup 2]
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

from bench_lstm_loop import SIZE, T, WordHashTokenizer, card, items

ARMS = ("two_pass", "on_policy")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_et_onpolicy.py needs a CUDA device")
    from avdn_b200.env import ANDHNavBatch
    from avdn_b200.utils import synthetic as syn
    from avdn_b200.xview_et.agent import NavCMTAgent
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(syn.yolov3_trunk_cfg())
    args = types.SimpleNamespace(demb=768, encoder_heads=12, encoder_layers=2, dropout_transformer_encoder=0.1,
                                 num_input_actions=1, dropout_emb=0.0, darknet_model_file=f.name,
                                 darknet_weight_file=None, max_action_len=T, lr=1e-5, nss_w=1.0, nss_r=0,
                                 ml_weight=0.2, teacher_weight=1.0, train_val_on_full=False, vision_only=False,
                                 no_direction=False, optim="adamW", bn_per_step=True, on_policy_student=False)
    torch.manual_seed(0)
    agent = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    agent.tokenizer = WordHashTokenizer()
    agent.attach_lang_model()
    env = ANDHNavBatch(batch_size=len(items()), device="cuda")
    env.map_batch["tile"] = syn.synthetic_tile(seed=0, size=SIZE)
    env.attention_map_batch["tile"] = syn.synthetic_attention_tile(seed=0, size=SIZE)
    env.batch = items()
    agent.env = env
    loader = [None]                                  # the reference's loader fills env as a side effect

    def student_rollout():
        agent.vision_model.train(); agent.vln_model.train(); agent.lang_model.train()
        agent.feedback, agent.loss = "student", 0
        agent.rollout(train_ml=0.2, nss_w=float(args.nss_w))

    def train_iteration():
        agent.train(loader, 1, feedback="student")

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    res = {arm: dict(student_rollout_ms=[], train_iteration_ms=[], steps=[]) for arm in ARMS}
    for arm in ARMS:
        args.on_policy_student = arm == "on_policy"
        for _ in range(a.warmup):
            student_rollout()
            train_iteration()
    for i in range(a.steps):
        for arm in (ARMS if i % 2 == 0 else ARMS[::-1]):
            args.on_policy_student = arm == "on_policy"
            res[arm]["student_rollout_ms"].append(timed(student_rollout))
            res[arm]["steps"].append(int(agent._last_rollout["steps"]))
            res[arm]["train_iteration_ms"].append(timed(train_iteration))
    name, power = card()
    out = {"workload": "et_haa student-feedback training: B=64 episodes, max_action_len 10, 2-layer 12-head ET "
                       "(encoder dropout 0.1), BERT-base trained in the loop, ~250-token dialogs, 3000x3000 synthetic "
                       "tile, bn_per_step, nss_w 1.0; two-pass vs on-policy, alternated",
           "gpu": name, "power_limit": power, "steps": a.steps, "warmup": a.warmup}
    for arm in ARMS:
        r = res[arm]
        for k in ("student_rollout_ms", "train_iteration_ms"):
            x = np.array(r[k])
            out[f"{arm}_{k}"] = round(float(np.median(x)), 3)
            out[f"{arm}_{k}_min_max"] = [round(float(x.min()), 3), round(float(x.max()), 3)]
        out[f"{arm}_rollout_steps"] = r["steps"]
        # the greedy loop reads the B stop flags after every step; the on-policy loop after every step but the last
        out[f"{arm}_stop_flag_reads_in_loop"] = [min(s, T - 1) if arm == "on_policy" else s for s in r["steps"]]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
