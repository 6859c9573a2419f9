"""Training workload of bench.py: BASELINE.json configs[1] (and configs[3] under
torchrun): et_haa training step, bf16 tensor-core path, batch 64 per GPU,
synthetic ANDH shape (250-token dialog history, 10 views of 224x224 per
episode), Darknet features + transformer + both heads, loss, backward, AdamW.

A step = render the 640 views of the batch from the synthetic 3000x3000 tile,
Darknet trunk forward (train-mode BatchNorm), ET forward, fused loss, ET
backward, Darknet backward, (gradient all-reduce), clip + AdamW on both models.
"""
from __future__ import annotations

import math
import json
import os
import time
import types

import numpy as np
import torch

L_LANG, T_STEPS, SIZE = 250, 10, 3000
DARKNET_GFLOP_IMG = 15.295          # forward, per 224x224 image (SURVEY.md §8a D2)


def et_flops_fwd(S=270, d=768, layers=2):
    # per layer: qkv 3d^2 + out d^2 + ffn 2d^2 = 6 d^2 MACs per token; attention 2 S d MACs per token
    return layers * (2 * S * d * 6 * d + 4 * S * S * d)


def make_args(cfg_path):
    return types.SimpleNamespace(demb=768, encoder_heads=12, encoder_layers=2, dropout_transformer_encoder=0.1,
                                 num_input_actions=1, dropout_emb=0.0, darknet_model_file=cfg_path,
                                 darknet_weight_file=None, lr=1e-5, nss_w=0.1, nss_r=0, ml_weight=0.2)


def synthetic_batch(B, T, L, seed, tile_size=SIZE):
    """Host (numpy / torch CPU) episode tensors of the ANDH shape (SURVEY.md §8d)."""
    from avdn_b200.utils import synthetic as wo   # synthetic inputs (product-side generators)
    g = torch.Generator().manual_seed(seed)
    rng = np.random.default_rng(seed)
    corners = wo.synthetic_pose_corners(B * T, seed=seed, size=tile_size, edge_frac=0.05).reshape(B, T, 4, 2)
    deg = torch.from_numpy(rng.integers(0, 360, size=(B, T)).astype(np.float32))
    dirs = torch.stack([torch.sin(deg / 180 * 3.14159), torch.cos(deg / 180 * 3.14159)], -1)
    xy = torch.from_numpy(rng.uniform(-1, 1, size=(B, 2)).astype(np.float32))
    xy = xy / torch.clamp(xy.abs().max(dim=1, keepdim=True).values, min=1.0)
    return dict(
        corners_px=torch.from_numpy(corners.astype(np.int32)),
        lang=torch.randn(B, L, 768, generator=g),
        lang_cls=torch.relu(torch.randn(B, 49, generator=g)),
        directions=dirs.contiguous(),
        gt_xy=xy.contiguous(),
        gt_alt=torch.from_numpy(rng.uniform(0, 1, size=B).astype(np.float32)),
        gt_prog=torch.from_numpy(rng.uniform(0, 1, size=B).astype(np.float32)),
        lenths=[T] * B,
    )


class TrainWorkload:
    name = "train_cfg2"
    metric = "HAA-Transformer train episodes/s"
    unit = "episodes/s"
    dtype = "bf16"
    B = 64
    CPU_SAMPLE = 4                    # episodes per CPU step = BASELINE configs[0] (batch 4)

    def __init__(self, rank, world):
        self.rank, self.world = rank, world
        self.B = int(os.environ.get("AVDN_BENCH_BATCH", self.B))

    def units_per_step(self):
        return self.B

    def config(self):
        return {"workload": "et_haa training step bf16, batch 64/GPU, synthetic ANDH shape: 250-token dialog, "
                            "10 views 224x224/episode rendered from a 3000x3000 tile, Darknet(57 conv, train-mode BN) "
                            "+ ET(2x768, 12 heads) + waypoint & human-attention heads, loss, backward, clip, AdamW "
                            "(BASELINE configs[1]; configs[3] under torchrun)",
                "global_batch": self.B * self.world, "per_gpu_batch": self.B, "views_per_step_per_gpu": self.B * T_STEPS,
                "seq_len": L_LANG + 2 * T_STEPS, "dropout": "train mode: 0.1 at the 4 sites of each encoder layer, 0.2 in the heads (stateless hash masks)",
                "cache": "per-step working set (~40 GB of activations) far exceeds L2; L2 is also flushed between steps",
                "parity_mode": "ET logits / loss / every gradient vs the fp32 oracle at the configs[0] shape (1e-2 / 5e-2); "
                               "trunk per block 1e-2 forward, 8e-2 backward (teacher-forced); trunk END TO END only by the "
                               "bf16-storage envelope (the random-init 57-block train-mode-BN chain amplifies a "
                               "perturbation ~100x, so no bf16 pipeline sits within 1e-2 of fp32 there); fused step loss "
                               "1e-2 at B=4, T=10, L=250 on conditioned weights (tests/test_agent_gpu.py)",
                "parallelism": f"dp{self.world} by episode, NCCL all-reduce of gradients" if self.world > 1 else "dp1"}

    cpu_dtype = "fp32"

    def cpu_config(self):
        """What the CPU leg (``--impl reference`` / ``cpu_baseline``) actually runs: BASELINE configs[0]."""
        return {"workload": "et_haa forward + loss + backward + clip + AdamW on the host cores, fp32, batch 4 "
                            "(BASELINE configs[0]): 40 views rendered with cv2.warpPerspective, Darknet (train-mode BN) "
                            "+ ET + both heads; torch CPU restatement pinned to the reference modules",
                "global_batch": self.CPU_SAMPLE, "per_gpu_batch": self.CPU_SAMPLE,
                "views_per_step_per_gpu": self.CPU_SAMPLE * T_STEPS, "dropout": "off (oracle arithmetic)",
                "cache": "n/a (host)", "parallelism": "none (one process, all host threads)"}

    # --------------------------------------------------------------------- GPU
    def setup_gpu(self, dev):
        import tempfile
        from avdn_b200.utils import synthetic as mo
        from avdn_b200.utils import synthetic as wo
        from avdn_b200.xview_et.agent import NavCMTAgent
        self.dev = dev
        with tempfile.NamedTemporaryFile("w", suffix=".cfg", delete=False) as f:
            f.write(mo.yolov3_trunk_cfg())
        torch.manual_seed(0)
        self.agent = NavCMTAgent(make_args(f.name), rank=self.rank, world_size=self.world, device=dev)
        os.unlink(f.name)
        tile = wo.synthetic_tile(seed=0, size=SIZE)
        att = wo.synthetic_attention_tile(seed=0, size=SIZE)
        self.agent.renderer.add_map("tile", tile, att)
        self.host = synthetic_batch(self.B, T_STEPS, L_LANG, seed=self.rank)
        self.pinned = {k: v.pin_memory() for k, v in self.host.items() if torch.is_tensor(v)}
        self.batch = {k: v.to(dev) for k, v in self.host.items() if torch.is_tensor(v)}
        self.batch["lenths"] = self.host["lenths"]
        self.loss_host = torch.zeros(1, dtype=torch.float64).pin_memory()
        self.profile = None
        self.last_loss = None
        self._start_state = None

    def _state_tensors(self):
        ag = self.agent
        return [t for o in ag.optimizers for t in (o.p, o.m, o.v)] + list(ag.vision_model.buffers())

    def _dropout_modules(self):
        ag = self.agent
        return [m for model in (ag.vision_model, ag.vln_model, ag.lang_model) if model is not None
                for m in model.modules() if hasattr(type(m), "dropout_config")]

    def snapshot(self):
        """Everything a training step reads and updates besides the batch: weights, AdamW moments and step counts,
        the trunk's BatchNorm running statistics and the dropout step counters (the masks derive from them)."""
        return ([t.clone() for t in self._state_tensors()], [o.step_count for o in self.agent.optimizers],
                [getattr(m, "_drop_step", 0) for m in self._dropout_modules()])

    def restore(self, snap):
        tensors, counts, drop = snap
        for t, t0 in zip(self._state_tensors(), tensors):
            t.copy_(t0)
        for o, n in zip(self.agent.optimizers, counts):
            o.step_count = n
        for m, n in zip(self._dropout_modules(), drop):
            m._drop_step = n

    def before_step(self):
        """Untimed, before every warm-up and timed step: put back the state the first step started from
        (``snapshot``), so that every step computes the same training step from the same state on the same batch.
        Without it each step trains on from the previous one, and the order of atomic reductions -- which is not
        fixed -- makes two runs of one command drift apart step by step (AdamW's first updates are nearly
        sign(grad), and the random-init train-mode trunk amplifies small differences)."""
        if self._start_state is None:
            self._start_state = self.snapshot()
        else:
            self.restore(self._start_state)

    def step(self):
        l0 = self.agent.launches
        self.agent.train_step(self.batch)
        return self.agent.launches - l0

    def after_step(self, timed):
        pass

    def outputs(self):
        """What the last ``step()`` produced (``bench.py --dump-outputs``): the step loss ``train_step`` returns and
        the state the step leaves -- the trunk's BatchNorm running statistics and, per model, the gradients and the
        updated parameters, concatenated in sorted parameter-name order so that they do not depend on the layout of
        the optimiser arenas.  ``before_step`` makes the last step start from the same state in every run."""
        ag = self.agent
        out = {"loss": ag.loss_total,
               "trunk_bn_running": torch.cat([b.flatten().float() for n, b in sorted(ag.vision_model.named_buffers())
                                              if "running" in n])}
        for model, opt in zip(("et", "trunk", "lang"), ag.optimizers):
            names = sorted(opt.params)
            out[f"{model}_grad"] = torch.cat([opt.grads[n].flatten() for n in names])
            out[f"{model}_param"] = torch.cat([opt.params[n].detach().flatten() for n in names])
        return out

    def step_e2e(self):
        h2d = 0
        b = {}
        for k, v in self.pinned.items():
            b[k] = v.to(self.dev, non_blocking=True)
            h2d += v.numel() * v.element_size()
        b["lenths"] = self.host["lenths"]
        loss = self.agent.train_step(b)
        self.loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last_loss = float(self.loss_host.item())
        return h2d, 8

    def profile_step(self):
        """One instrumented step (outside the timed region): per-kernel CUDA-event times."""
        from avdn_b200 import _lib
        _lib.PROFILE = []
        self.agent.train_step(self.batch)
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1, fl, nb in _lib.PROFILE:
            a = agg.setdefault(name, [0, 0.0, 0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += fl
        _lib.PROFILE = None
        self.profile = agg
        return agg

    def prepare_roofline(self):
        """Called on EVERY rank: the instrumented step is a full data-parallel step (all-reduce inside)."""
        if self.profile is None:
            self.profile_step()

    def flops_per_step(self):
        return (DARKNET_GFLOP_IMG * 1e9 * self.B * T_STEPS + et_flops_fwd() * self.B) * 3

    def roofline(self, peaks, ms_per_step=None):
        if self.profile is None:
            self.profile_step()
        g = {k: v for k, v in self.profile.items() if k.startswith("gemm") or k.startswith("avdn_conv3x3_thin")}
        g_ms = sum(v[1] for v in g.values())
        g_fl = sum(v[2] for v in g.values())
        g_n = sum(v[0] for v in g.values())
        tot = sum(v[1] for v in self.profile.values())
        ach = g_fl / (g_ms * 1e-3) / 1e12 if g_ms else None
        peak = peaks["bf16_sustained"]
        self._peak = peak
        top = sorted(self.profile.items(), key=lambda kv: -kv[1][1])[:14]
        # DRAM traffic is not measurable from inside the run (it needs ncu): null here; the ncu capture of this
        # command is summarised under profiles/ (r02_*).
        traffic, traffic_src = None, "not measured in-run (ncu summaries under profiles/)"
        return {"kernel": "gemm_kernel + conv3_halo_kernel (tcgen05 conv fwd/dgrad/wgrad + transformer GEMMs)",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": (ach / peak) if ach else None, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peaks["source"] + " (sustained bf16 cuBLAS; kernel timed inside a long step)",
                "algorithmic_flops_per_step": g_fl, "gemm_launches_per_step": g_n, "gemm_ms_per_step": g_ms,
                "gemm_share_of_kernel_time": g_ms / tot if tot else None,
                "kernel_ms_breakdown": {k: {"n": v[0], "ms": round(v[1], 3)} for k, v in top}}

    def extra(self, ms_per_step=None):
        out = {"last_loss": self.last_loss}
        if ms_per_step:
            fl = self.flops_per_step()
            out["step_tflops_algorithmic"] = fl / 1e12
            out["step_tflops_per_s"] = fl / (ms_per_step * 1e-3) / 1e12
            out["mfu_vs_sustained_bf16"] = out["step_tflops_per_s"] / self._peak if getattr(self, "_peak", None) else None
        return out

    # ------------------------------------------------------------ multi-GPU proofs
    def multi_gpu_checks(self, dist):
        """Under torchrun, on every rank, after the timed steps: (1) the replicas hold bit-identical parameters
        (all-reduce MAX and MIN of per-arena checksums agree), (2) how long the optimiser waited for the last
        gradient bucket (CUDA events around the wait on the communication stream, mean over instrumented steps)."""
        ag = self.agent
        sums = []
        for opt in ag.optimizers:
            p = opt.p
            sums += [p.double().sum(), p.double().abs().sum(), p.view(torch.int32).double().sum()]
        v = torch.stack(sums)
        hi, lo = v.clone(), v.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        in_sync = bool(torch.equal(hi, lo))
        ag.exposed_events = []
        for _ in range(3):
            ag.train_step(self.batch)
        torch.cuda.synchronize()
        ex = [a.elapsed_time(b) for a, b in ag.exposed_events]
        ag.exposed_events = None
        t = torch.tensor([float(np.mean(ex)) if ex else 0.0], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # (3) the same step with the collective switched off (every rank an independent replica, state snapshotted
        # and restored around it): max over ranks = what the slowest GPU of this box does on its own, the floor a
        # synchronous step cannot beat; the distance from ms_per_step to it is what data parallelism costs
        k = 8

        def back_to_back():
            for _ in range(2):
                ag.train_step(self.batch)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k):
                ag.train_step(self.batch)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k

        synced = back_to_back()                       # same loop with the all-reduce on, for a like-for-like pair
        snap = self.snapshot()
        world, ag.world = ag.world, 1
        try:
            solo = back_to_back()
        finally:
            ag.world = world
        self.restore(snap)
        per = [torch.zeros(2, dtype=torch.float64, device=self.dev) for _ in range(world)]
        dist.all_gather(per, torch.tensor([solo, synced], dtype=torch.float64, device=self.dev))
        synced = max(float(x[1].item()) for x in per)
        per = [round(float(x[0].item()), 3) for x in per]
        return {"replicas_in_sync": in_sync, "allreduce_exposed_ms": float(t.item()),
                "replica_ms_per_step_without_allreduce": {"per_rank": per, "max": max(per), "min": min(per),
                                                          "steps": k, "same_loop_with_allreduce": round(synced, 3),
                                                          "note": "back-to-back steps, no L2 flush between them"},
                "allreduce": {"bytes_per_step": int(sum(o.n for o in ag.optimizers) * (2 if ag._ar_bf16 else 4)),
                              "dtype": "bf16" if ag._ar_bf16 else "fp32", "buckets": 1 + len(ag._buckets or [])}}

    # ---------------------------------------------------------------- library bar
    def library_bar(self, ours_ms):
        """The same B = 64 step on stock torch 2.x kernels (cuDNN convolutions / BatchNorm, cuBLAS GEMMs, SDPA inside
        nn.TransformerEncoderLayer, fused AdamW): nn modules of the reference's architecture (random init), bf16
        autocast, channels-last, cudnn.benchmark -- the best stock configuration.  Test infrastructure like the CPU
        leg: nothing of it is on the product path.  View rendering is NOT included (the reference renders on the
        host), so the comparison favours the library side by the ~0.3 ms the renderer takes."""
        import torch.nn as nn
        import torch.nn.functional as F
        from avdn_b200.utils import synthetic as syn
        dev = self.dev
        B, T, L = self.B, T_STEPS, L_LANG

        class Trunk(nn.Module):
            def __init__(s_, cfg_text):
                super().__init__()
                s_.defs = []
                cur = None
                for line in cfg_text.split("\n"):
                    line = line.strip()
                    if line.startswith("["):
                        cur = {"type": line[1:-1]}
                        s_.defs.append(cur)
                    elif "=" in line and cur is not None:
                        k, v = line.split("=")
                        cur[k.strip()] = v.strip()
                s_.defs = s_.defs[1:]
                s_.mods = nn.ModuleList()
                ch = [3]
                for d in s_.defs:
                    if d["type"] == "convolutional":
                        f, k, st = int(d["filters"]), int(d["size"]), int(d["stride"])
                        s_.mods.append(nn.Sequential(nn.Conv2d(ch[-1], f, k, st, (k - 1) // 2, bias=False),
                                                     nn.BatchNorm2d(f), nn.LeakyReLU(0.01)))
                        ch.append(f)
                    else:
                        s_.mods.append(nn.Identity())
                        ch.append(ch[int(d["from"])])

            def forward(s_, x):
                outs = []
                for d, m in zip(s_.defs, s_.mods):
                    x = m(x) if d["type"] == "convolutional" else outs[-1] + outs[int(d["from"])]
                    outs.append(x)
                return x

        class ETLike(nn.Module):
            def __init__(s_):
                super().__init__()
                s_.w_in = nn.Linear(49, 49, bias=False); s_.w_out = nn.Linear(98, 49, bias=False)
                s_.fc2 = nn.Linear(49, 768); s_.demb = nn.Linear(2, 768); s_.ln = nn.LayerNorm(768)
                s_.enc = nn.TransformerEncoder(nn.TransformerEncoderLayer(768, 12, 768, 0.1), 2,
                                               enable_nested_tensor=False)
                s_.head = nn.Sequential(nn.Linear(768, 256), nn.ReLU(), nn.Dropout(0.2), nn.Linear(256, 32), nn.ReLU(),
                                        nn.Dropout(0.2), nn.Linear(32, 4))
                s_.fc = nn.Sequential(nn.Linear(768, 64), nn.Dropout(0.2), nn.ReLU())

            def forward(s_, frames, lang, lang_cls, dirs, mask, pe):
                Bq, Tq = dirs.shape[:2]
                ctx = frames.view(Bq, Tq, 512, 49)
                tgt = s_.w_in(lang_cls)                                                   # SoftDotAttention(49)
                attn = torch.softmax(torch.einsum("btcp,bp->btc", ctx, tgt), dim=2)
                wc = torch.einsum("btc,btcp->btp", attn, ctx)
                h = torch.tanh(s_.w_out(torch.cat((wc, lang_cls[:, None].expand(-1, Tq, -1)), -1)))
                x = torch.cat((lang + pe[:L], s_.fc2(h) + pe[L:L + Tq], s_.demb(dirs) + pe[L:L + Tq]), 1)
                x = s_.enc(s_.ln(x).transpose(0, 1), mask=mask).transpose(0, 1)
                out = s_.head(x[:, L + 2 * Tq - 1])
                sal = F.interpolate(s_.fc(x[:, L + Tq - 1]).view(-1, 1, 8, 8), size=(224, 224), mode="bilinear",
                                    align_corners=False)
                return out, sal

        prev = torch.backends.cudnn.benchmark
        torch.backends.cudnn.benchmark = True
        try:
            torch.manual_seed(0)
            trunk = Trunk(syn.yolov3_trunk_cfg()).to(dev).to(memory_format=torch.channels_last).train()
            et = ETLike().to(dev).train()
            opt_t = torch.optim.AdamW(trunk.parameters(), lr=1e-5, fused=True)
            opt_e = torch.optim.AdamW(et.parameters(), lr=1e-5, fused=True)
            images = torch.randn(B * T, 3, 224, 224, device=dev).contiguous(memory_format=torch.channels_last)
            S = L + 2 * T
            mask = torch.zeros(S, S, device=dev)
            mask[:L, L:] = float("-inf")
            tri = torch.triu(torch.full((T, T), float("-inf"), device=dev), 1)
            mask[L:L + T, L:L + T] = tri; mask[L:L + T, L + T:] = tri
            mask[L + T:, L:L + T] = tri; mask[L + T:, L + T:] = tri
            pe = torch.randn(S, 768, device=dev) * 0.02
            bt = self.batch
            fix = torch.zeros(B, 1, 224, 224, device=dev)
            fix[:, :, 60:120, 80:160] = 1.0

            def step():
                opt_t.zero_grad(set_to_none=True)
                opt_e.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    feats = trunk(images)
                    out, sal = et(feats.float().reshape(B * T, 512, 49), bt["lang"], bt["lang_cls"], bt["directions"],
                                  mask, pe)
                out, sal = out.float(), sal.float()
                loss = ((out[:, :2] - bt["gt_xy"]) ** 2).sum() + ((out[:, 2] - bt["gt_alt"]) ** 2).sum() + \
                       ((out[:, 3] - bt["gt_prog"]) ** 2).sum()
                m, sd_ = sal.mean((1, 2, 3), keepdim=True), sal.std((1, 2, 3), keepdim=True)
                loss = loss - 0.1 * ((((sal - m) / sd_) * fix).sum((1, 2, 3)) / (fix.sum((1, 2, 3)) + 1e-3)).sum()
                (loss * 0.2 / B).backward()
                torch.nn.utils.clip_grad_norm_(et.parameters(), 40.0)
                opt_t.step()
                opt_e.step()

            for _ in range(3):
                step()
            torch.cuda.synchronize()
            n = 5
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
            for a, b in evs:
                a.record(); step(); b.record()
            torch.cuda.synchronize()
            ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
        finally:
            torch.backends.cudnn.benchmark = prev
        del trunk, et, opt_t, opt_e, images
        torch.cuda.empty_cache()
        return {"what": "stock torch " + torch.__version__ + " modules of the same architecture (nn.Conv2d + "
                        "nn.BatchNorm2d(train) + nn.LeakyReLU x57 with shortcuts; SoftDotAttention + nn.TransformerEncoder "
                        "(2 x 768, 12 heads, ff 768) + both heads, upsample + NSS-style loss), bf16 autocast, channels-last, "
                        "cudnn.benchmark, fused AdamW on both models, clip on ET; batch 64 x 10 views; view rendering "
                        "excluded",
                "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": "episodes/s", "steps": n, "warmup": 3,
                "ours_ms_per_step": ours_ms, "ours_over_library_speedup": ms / ours_ms}

    # --------------------------------------------------------------------- CPU
    def _cpu_setup(self):
        if getattr(self, "_cpu", None) is not None:
            return self._cpu
        from oracle import model_oracle as mo
        torch.manual_seed(0)
        B, T, L = self.CPU_SAMPLE, T_STEPS, L_LANG
        cfg = mo.yolov3_trunk_cfg()
        sd = mo.random_trunk_state(cfg, seed=0)
        et_sd = mo.random_et_state(seed=0)
        for d in (sd, et_sd):
            for k, v in d.items():
                if v.is_floating_point() and "running" not in k and not k.endswith(".pe"):
                    v.requires_grad_(True)
        hb = synthetic_batch(B, T, L, seed=0)
        from avdn_b200.utils import synthetic as syn
        tile = syn.synthetic_tile(seed=0, size=SIZE)
        att = syn.synthetic_attention_tile(seed=0, size=SIZE)
        opt_t = torch.optim.AdamW([v for v in sd.values() if v.requires_grad], lr=1e-5)
        opt_e = torch.optim.AdamW([v for v in et_sd.values() if v.requires_grad], lr=1e-5)
        self._cpu = (mo, cfg, sd, et_sd, hb, tile, att, opt_t, opt_e)
        return self._cpu

    def cpu_step(self, n):
        """The oracle's restatement of the reference step (torch CPU fp32 autograd: Darknet
        train-mode forward, ET forward, loss, backward) on ``CPU_SAMPLE`` episodes."""
        import cv2
        mo, cfg, sd, et_sd, hb, tile, att, opt_t, opt_e = self._cpu_setup()
        B, T = self.CPU_SAMPLE, T_STEPS
        dst = np.array([[0, 0], [223, 0], [223, 223], [0, 223]], dtype=np.float32)
        mean = np.array([60.134, 49.697, 40.746], dtype=np.float32).reshape(3, 1, 1)       # agent.py:115-116
        std = np.array([29.99, 24.498, 22.046], dtype=np.float32).reshape(3, 1, 1)
        done = 0
        while done < n:
            opt_t.zero_grad(set_to_none=True)
            opt_e.zero_grad(set_to_none=True)
            # the observations: cv2 calls of src/env.py:287-293, normalisation of agent.py:586-592
            views, sal = [], []
            cpx = hb["corners_px"].numpy().astype(np.float32)
            for b in range(B):
                for t in range(T):
                    M = cv2.getPerspectiveTransform(cpx[b, t], dst)
                    views.append(cv2.warpPerspective(tile, M, (224, 224)))
                    if t == T - 1:
                        sal.append(cv2.warpPerspective(att, M, (224, 224))[:, :, 0].astype(np.float64) / 255)
            images = np.ascontiguousarray(np.stack(views)[:, :, :, ::-1].transpose(0, 3, 1, 2), dtype=np.float32)
            images -= mean
            images /= std
            gt_sal = torch.from_numpy(np.stack(sal))
            feats = mo.darknet_forward(torch.from_numpy(images), sd, cfg, train=True).view(B, T, 512, 49)
            out, sal_p, _ = mo.et_forward(et_sd, hb["directions"], feats, hb["lenths"], hb["lang"], hb["lang_cls"])
            loss = mo.step_loss(mo.et_loss(out, sal_p, hb["gt_xy"], hb["gt_alt"], hb["gt_prog"], gt_sal, 0.1), 0.2, B)
            loss.backward()
            torch.nn.utils.clip_grad_norm_([v for v in et_sd.values() if v.requires_grad], 40.0)      # agent.py:247
            opt_t.step()
            opt_e.step()
            done += B
        return done

    def cpu_info(self):
        return {"kind": "port", "cores": int(torch.get_num_threads()),
                "what": "cv2 view rendering + oracle/model_oracle.py (torch CPU fp32 restatement of Darknet + ET + loss, "
                        "fwd+bwd) + clip_grad_norm_ + AdamW, BASELINE configs[0] shape (batch 4, 10 views, 250 tokens)"}


class TrainRolloutWorkload(TrainWorkload):
    """The teacher-forced training rollout (src/xview_et/agent.py:580-760): the loss at every one of the 10 steps on
    the growing history -- views and trunk once over the 640 poses, then the reference's 10 encoder calls (history
    1..10), each with its loss and backward -- one optimiser step."""
    name = "train_rollout"
    metric = "HAA-Transformer train rollout episodes/s"

    def config(self):
        c = super().config()
        c["workload"] = c["workload"].replace("et_haa training step bf16", "et_haa teacher-forced training rollout "
                                              "(loss at each of the 10 steps on the history so far; 10 encoder "
                                              "forward+backward passes per step), bf16")
        return c

    def setup_gpu(self, dev):
        super().setup_gpu(dev)
        rng = np.random.default_rng(200 + self.rank)
        B, T = self.B, T_STEPS
        xy = torch.from_numpy(rng.uniform(-1, 1, size=(B, T, 2)).astype(np.float32))
        self.host.update(gt_xy=(xy / torch.clamp(xy.abs().amax(dim=2, keepdim=True), min=1.0)).contiguous(),
                         gt_alt=torch.from_numpy(rng.uniform(0, 1, size=(B, T)).astype(np.float32)),
                         gt_prog=torch.from_numpy(rng.uniform(0, 1, size=(B, T)).astype(np.float32)))
        self.host.pop("lenths")
        self.pinned = {k: v.pin_memory() for k, v in self.host.items() if torch.is_tensor(v)}
        self.batch = {k: v.to(dev) for k, v in self.host.items() if torch.is_tensor(v)}

    def step(self):
        l0 = self.agent.launches
        self.agent.train_rollout_step(self.batch)
        return self.agent.launches - l0

    def step_e2e(self):
        h2d = 0
        b = {}
        for k, v in self.pinned.items():
            b[k] = v.to(self.dev, non_blocking=True)
            h2d += v.numel() * v.element_size()
        loss = self.agent.train_rollout_step(b)
        self.loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last_loss = float(self.loss_host.item())
        return h2d, 8

    def profile_step(self):
        from avdn_b200 import _lib
        _lib.PROFILE = []
        self.agent.train_rollout_step(self.batch)
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1, fl, nb in _lib.PROFILE:
            a = agg.setdefault(name, [0, 0.0, 0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += fl
        _lib.PROFILE = None
        self.profile = agg
        return agg

    def flops_per_step(self):
        et = sum(et_flops_fwd(S=L_LANG + 2 * t) for t in range(1, T_STEPS + 1))
        return (DARKNET_GFLOP_IMG * 1e9 * self.B * T_STEPS + et * self.B) * 3

    def roofline(self, peaks, ms_per_step=None):
        r = super().roofline(peaks, ms_per_step)
        r["traffic"], r["traffic_source"] = None, None
        return r

    def cpu_step(self, n):
        raise SystemExit("the train_rollout workload has no CPU leg: use --no-cpu-baseline")


class TrainBertWorkload(TrainWorkload):
    """The training step with the language encoder in the loop (src/xview_et/agent.py:125-126,155,249,527-543):
    token ids in, BERT-base forward + backward + AdamW inside the step."""
    name = "train_bert"
    metric = "HAA-Transformer + BERT train episodes/s"

    def config(self):
        c = super().config()
        c["workload"] = c["workload"].replace("et_haa training step bf16", "et_haa training step with the language "
                                              "encoder (CustomBERTModel, bert-base, 250 tokens) trained in the loop, bf16")
        return c

    def setup_gpu(self, dev):
        super().setup_gpu(dev)
        self.agent.attach_lang_model()
        g = torch.Generator().manual_seed(100 + self.rank)
        ids = torch.randint(0, 30522, (self.B, L_LANG), generator=g)
        lens = torch.randint(L_LANG // 3, L_LANG + 1, (self.B,), generator=g)
        lens[0] = L_LANG
        mask = (torch.arange(L_LANG)[None] < lens[:, None]).long()
        for d in (self.host, ):
            d.pop("lang"); d.pop("lang_cls")
            d["input_ids"], d["attention_mask"] = ids, mask
        self.pinned = {k: v.pin_memory() for k, v in self.host.items() if torch.is_tensor(v)}
        self.batch = {k: v.to(dev) for k, v in self.host.items() if torch.is_tensor(v)}
        self.batch["lenths"] = self.host["lenths"]

    def flops_per_step(self):
        from bench_bert import bert_flops_fwd
        return super().flops_per_step() + 3 * bert_flops_fwd(self.B, L_LANG)

    def roofline(self, peaks, ms_per_step=None):
        r = super().roofline(peaks, ms_per_step)
        r["traffic"], r["traffic_source"] = None, None
        return r

    def cpu_step(self, n):
        raise SystemExit("the train_bert workload has no CPU leg: use --no-cpu-baseline (train and bert have one each)")
