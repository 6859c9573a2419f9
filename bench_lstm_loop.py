"""The LSTM baseline's agent loop on one GPU, with the reference's signatures: ``NavCMTAgent.train(loader, 1,
'student')`` and ``test(loader, feedback=...)`` over an ``ANDHNavBatch`` of B = 64 episodes, ``max_action_len`` 10,
BERT-base (``CustomBERTModel()``) trained in the loop, dialogs of about 250 tokens (a tokenizer stand-in: words hash to
ids), views rendered from a 3000x3000 synthetic tile.  Prints one JSON line.

* ``ms_per_train_iteration``: one ``train`` iteration = a teacher-feedback training rollout (no NSS term) + a
  student-feedback one (greedy rollout, then training on its poses) + clip + AdamW on policy, trunk and BERT.
* ``ms_per_test_batch_student`` / ``_teacher``: one ``test`` batch (greedy rollout / teacher poses with the
  human-attention validation scores).
Each is timed over several iterations after warm-up, with a synchronise at the end of each.

The scoring of the teacher-feedback validation (precision, recall, NSS of every step and sample) is also timed on the
T*B rows of the last teacher test batch, through ``avdn_saliency_metrics`` (one launch) and through the ET agent's
per-sample torch loop (``xview_et.agent.NavCMTAgent._eval_rollout``), with the largest difference between the two.

    python bench_lstm_loop.py [--steps 3] [--warmup 1]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import tempfile
import time
import types

import numpy as np
import torch

B, T, SIZE, WORDS = 64, 10, 3000, 250
BL, TR = np.array([40.0, -75.0]), np.array([40.03, -74.97])
LAT_RATIO = 0.03 / SIZE


class WordHashTokenizer:
    """Stand-in for BertTokenizerFast (no vocabulary offline): one id per word, [CLS] = 101 first, [SEP] = 102 last,
    padding 0 -- the reference's token counts for dialogs of the same number of words."""

    def __init__(self, vocab=30522):
        self.vocab = vocab

    def __call__(self, texts, padding=True, return_tensors="pt"):
        word_id = lambda w: 1000 + sum(ord(c) * (k + 1) for k, c in enumerate(w)) % (self.vocab - 1000)
        rows = [[101] + [word_id(w) for w in t.split()] + [102] for t in texts]
        n = max(len(r) for r in rows)
        ids = torch.zeros(len(rows), n, dtype=torch.long)
        mask = torch.zeros(len(rows), n, dtype=torch.long)
        for i, r in enumerate(rows):
            ids[i, :len(r)] = torch.tensor(r)
            mask[i, :len(r)] = 1
        return {"input_ids": ids, "attention_mask": mask}


def items(seed=0):
    """B episodes on one map: rotated-square views (40-80 m) with a 2-5 step straight ground-truth path, and a dialog
    of WORDS words (about 250 tokens; 50 of them in pre_dialogs)."""
    rng = np.random.default_rng(seed)
    words = ["fly", "towards", "the", "red", "building", "turn", "left", "right", "stop", "near", "road", "tree",
             "[que]", "[ins]", "where", "should", "i", "go", "after", "parking", "lot", "house", "roof", "river"]
    out = []
    for i in range(B):
        ctr = (BL + TR) / 2 + rng.uniform(-0.009, 0.009, size=2)
        half = rng.uniform(0.0002, 0.0004)
        th = rng.uniform(0, 2 * np.pi)
        R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        sq = (np.array([[1, -1], [1, 1], [-1, 1], [-1, -1]]) * half) @ R.T
        step = rng.uniform(-0.0004, 0.0004, size=2)
        path = [ctr + sq + k * step for k in range(int(rng.integers(2, 6)))]
        v = path[0][0] / 2 + path[0][1] / 2 - np.mean(path[0], axis=0)
        ang = (np.degrees(np.arctan2(v[1], v[0])) + 360) % 360
        text = " ".join(rng.choice(words, size=WORDS))
        out.append(dict(map_name="tile", route_index=str(i), gps_botm_left=BL.copy(), gps_top_right=TR.copy(),
                        lng_ratio=LAT_RATIO, lat_ratio=LAT_RATIO, angle=float(round(ang) % 360),
                        gt_path_corners=[np.asarray(p) for p in path], pre_dialogs=" ".join(text.split()[:50]) + " ",
                        instructions=" ".join(text.split()[50:])))
    return out


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:                          # the measurement stands; the card is then reported as unknown
        return torch.cuda.get_device_name(0), f"unknown ({type(e).__name__})"


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
    return ms


def et_host_scores(args, h_sali, att_t):
    """The per-sample scoring loop of ``xview_et.agent.NavCMTAgent._eval_rollout`` over [T,B] rows: per step one
    upsample launch, then per sample the torch NSS / clip / sums.  Returns [T,B,4] (precision, recall, nss, fixation
    sum; rows without fixations hold zeros)."""
    from avdn_b200 import _lib
    from avdn_b200.xview_et.agent import NavCMTAgent as ET
    et = types.SimpleNamespace(args=args)
    Tn, Bn = att_t.shape[:2]
    out = np.zeros((Tn, Bn, 4))
    for t in range(Tn):
        sal = torch.empty((Bn, 224, 224), dtype=torch.float32, device="cuda")
        _lib.call("avdn_upsample_saliency", _lib.ptr(h_sali[t].contiguous()), Bn, _lib.ptr(sal))
        gt = att_t[t].double() / 255
        for i in range(Bn):
            fs = float(gt[i].sum())
            if fs > 0:
                nss = ET.NSS(et, sal[i].double(), gt[i])
                p = sal[i].clip(0, 1).double()
                tp, sp = float((p * gt[i]).sum()), float(p.sum())
                out[t, i] = (tp / sp if sp != 0 else 0.0, tp / fs, float(nss), fs)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lstm_loop.py needs a CUDA device")
    from avdn_b200 import _lib
    from avdn_b200.env import ANDHNavBatch
    from avdn_b200.utils import synthetic as syn
    from avdn_b200.xview_lstm.agent import NavCMTAgent
    with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
        f.write(syn.yolov3_trunk_cfg())
    args = types.SimpleNamespace(darknet_model_file=f.name, darknet_weight_file=None, max_action_len=T, lr=1e-5,
                                 nss_w=1.0, nss_r=0, ml_weight=0.2, teacher_weight=1.0, train_val_on_full=False,
                                 vision_only=False, optim="adamW")
    torch.manual_seed(0)
    agent = NavCMTAgent(args, device="cuda")
    os.unlink(f.name)
    agent.tokenizer = WordHashTokenizer()
    agent.attach_lang_model()
    env = ANDHNavBatch(batch_size=B, device="cuda")
    env.map_batch["tile"] = syn.synthetic_tile(seed=0, size=SIZE)
    env.attention_map_batch["tile"] = syn.synthetic_attention_tile(seed=0, size=SIZE)
    env.batch = items()
    agent.env = env
    loader = [None]                                  # the reference's loader fills env as a side effect
    n_tok = int(agent._language_batch(env.batch)[0]["cls_attention_mask"].sum(1).float().mean())

    train_ms = timed(lambda: agent.train(loader, 1, feedback="student"), a.steps, a.warmup)
    student_ms = timed(lambda: agent.test(loader, env_name="val_seen", feedback="student"), a.steps, a.warmup)
    teacher_ms = timed(lambda: agent.test(loader, env_name="val_seen", feedback="teacher"), a.steps, a.warmup)

    # ---- the teacher-feedback scoring of the last test batch's rows: kernel vs the ET agent's per-sample loop ----
    eng, att_t = agent._ctx_eval
    Tn = att_t.shape[0]
    h = eng.h_sali.contiguous()
    dev_out = torch.empty((Tn, B, 4), dtype=torch.float64, device="cuda")
    kern = lambda: _lib.call("avdn_saliency_metrics", _lib.ptr(h), _lib.ptr(att_t), Tn * B, 0, _lib.ptr(dev_out))
    kern()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        kern()
    e1.record()
    e1.synchronize()
    kernel_ms = e0.elapsed_time(e1) / 20
    et_host_scores(args, h, att_t)                   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host = et_host_scores(args, h, att_t)
    host_ms = (time.perf_counter() - t0) * 1e3
    k = dev_out.cpu().numpy()
    rows = host[..., 3] > 0
    rel = np.abs(k[..., :3] - host[..., :3]) / np.maximum(np.abs(host[..., :3]), 1e-12)
    name, power = card()
    med = lambda x: round(float(np.median(x)), 3)
    print(json.dumps({
        "workload": "lstm_haa agent loop: B=64 episodes, max_action_len 10, BERT-base trained in the loop, "
                    f"~{n_tok}-token dialogs, views rendered from a 3000x3000 synthetic tile",
        "gpu": name, "power_limit": power, "steps": a.steps, "warmup": a.warmup,
        "ms_per_train_iteration": med(train_ms), "ms_per_train_iteration_all": [round(x, 3) for x in train_ms],
        "ms_per_test_batch_student": med(student_ms), "ms_per_test_batch_teacher": med(teacher_ms),
        "scoring_rows": int(Tn * B), "scoring_rows_with_fixations": int(rows.sum()),
        "scoring_kernel_ms": round(kernel_ms, 4), "scoring_et_host_loop_ms": round(host_ms, 3),
        "scoring_max_rel_diff": float(rel[rows].max()) if rows.any() else 0.0,
        "scoring_fixation_rows_agree": bool(np.array_equal(k[..., 3] > 0, rows))}))


if __name__ == "__main__":
    main()
