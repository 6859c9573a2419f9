"""What the two agents (``xview_et.agent`` and ``xview_lstm.agent``, twins in the reference) share for training:
the batch-level training API (``RolloutTrainer``: loss weights, ``train_rollout_step``, ``train_iteration``, the
loss log, ``teacher_action``), the views and trunk passes of a teacher-forced training rollout, and the targets of
a student-feedback rollout.  Each agent supplies ``_train_rollout_step`` (its policy's forward, loss and backward)."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .models import dark_net as DN


class RolloutTrainer:
    """Mixin of the agents.  Needs ``args``, ``device``, ``launches``, ``loss_total``, ``logs`` and
    ``_train_rollout_step(batch, sync_loss, zero, step, collect, bn_per_step)``."""

    @property
    def nss_w(self):
        ov = getattr(self, "_nss_w_override", None)
        return float(ov if ov is not None else getattr(self.args, "nss_w", 1.0))        # parser.py:38 default 1

    @property
    def train_ml(self):
        ov = getattr(self, "_train_ml_override", None)
        return float(ov if ov is not None else getattr(self.args, "ml_weight", 0.2))     # parser.py:54

    class _Weights:
        """``with agent._weights(nss_w, train_ml):`` -- the per-rollout loss weights the reference passes to
        ``rollout(train_ml=..., nss_w=...)`` (agent.py:229-235); ``None`` keeps the value from ``args``."""

        def __init__(self, agent, nss_w, train_ml):
            self.a, self.v = agent, (nss_w, train_ml)

        def __enter__(self):
            self.old = (getattr(self.a, "_nss_w_override", None), getattr(self.a, "_train_ml_override", None))
            self.a._nss_w_override, self.a._train_ml_override = self.v

        def __exit__(self, *exc):
            self.a._nss_w_override, self.a._train_ml_override = self.old

    def _weights(self, nss_w=None, train_ml=None):
        return RolloutTrainer._Weights(self, nss_w, train_ml)

    LOG_KEEP = 4096

    def _log_loss(self):
        """``self.logs['IL_loss']`` (agent.py:885): one entry per rollout.  Device scalars (a copy: ``loss_total`` is
        rewritten every step), converted lazily by ``il_losses()``; bounded."""
        log = self.logs["IL_loss"]
        log.append(self.loss_total.clone())
        if len(log) > self.LOG_KEEP:
            del log[: len(log) - self.LOG_KEEP]

    def il_losses(self):
        """The logged losses as host floats (one synchronisation)."""
        log = self.logs["IL_loss"]
        return torch.stack([x.reshape(()) for x in log]).cpu().tolist() if log else []

    def train_iteration(self, teacher_batch, student_batch=None, sync_loss=False, feedback="student",
                        nss_w_weighting=1):
        """One iteration of ``train`` (agent.py:225-251).  ``feedback='student'`` (the reference's recipe): the
        teacher-feedback rollout with ``train_ml = args.ml_weight`` and **nss_w = 0** (agent.py:232), then the
        student-feedback rollout with ``nss_w = args.nss_w * nss_w_weighting`` (agent.py:235); the two add their
        losses, ONE backward's worth of gradients (accumulated over both), clip, one step of every optimiser.
        ``feedback='teacher'``: the teacher rollout alone with ``train_ml = args.teacher_weight`` and the NSS term
        (agent.py:229).  ``student_batch`` comes from ``student_batch()``.  Returns the summed loss."""
        nss = float(getattr(self.args, "nss_w", 1.0)) * nss_w_weighting
        if feedback == "teacher":
            tot = self.train_rollout_step(teacher_batch, nss_w=nss,
                                          train_ml=float(getattr(self.args, "teacher_weight", 1.0))).clone()
        elif feedback == "student":
            l1 = self.train_rollout_step(teacher_batch, step=False, nss_w=0.0).clone()
            tot = l1 + self.train_rollout_step(student_batch, zero=False, nss_w=nss)
        else:
            raise ValueError("Invalid feedback option")
        return float(tot.item()) if sync_loss else tot

    def train_rollout_step(self, batch, sync_loss=False, zero=True, step=True, nss_w=None, train_ml=None,
                           collect=None, bn_per_step=None):
        with self._weights(nss_w, train_ml):
            return self._train_rollout_step(batch, sync_loss, zero, step, collect, bn_per_step)

    def teacher_action(self, corners, gt_path_corners, ended, feedback=None):
        """``teacher_action`` (agent.py:386-507) for the whole batch on the device; ``feedback`` 'student' /
        'teacher' (default ``self.feedback`` or 'student').
        ``corners`` [B,4,2] f64 (lat,lng); ``gt_path_corners``: list (len B) of ``[n_i,4,2]`` arrays or a padded
        ``[B,Pmax,4,2]`` tensor with ``gt_len``; ``ended`` [B].  Returns device tensors
        ``(next_pos_ratio [B,2] f32, altitude [B] f32, progress [B] f32)`` -- the targets of ``output[:,0:2]``,
        ``output[:,2]`` and ``output[:,3]`` (agent.py:655-671)."""
        dev = self.device
        c = torch.as_tensor(np.asarray(corners) if not torch.is_tensor(corners) else corners).to(dev, torch.float64).contiguous()
        B = c.shape[0]
        packed = isinstance(gt_path_corners, tuple) and len(gt_path_corners) == 2 and torch.is_tensor(gt_path_corners[0])
        if isinstance(gt_path_corners, (list, tuple)) and not packed:
            lens = [len(g) for g in gt_path_corners]
            pmax = max(lens)
            gt = np.zeros((B, pmax, 4, 2), dtype=np.float64)
            for i, g in enumerate(gt_path_corners):
                gt[i, :lens[i]] = np.asarray(g, dtype=np.float64)
            gt_t = torch.from_numpy(gt).to(dev)
            len_t = torch.tensor(lens, dtype=torch.int32, device=dev)
        else:
            gt_t, len_t = gt_path_corners
            gt_t = gt_t.to(dev, torch.float64).contiguous()
            len_t = len_t.to(dev, torch.int32).contiguous()
            pmax = gt_t.shape[1]
        e = torch.as_tensor(np.asarray(ended, dtype=np.uint8) if not torch.is_tensor(ended) else ended).to(dev, torch.uint8).contiguous()
        ratio = torch.empty((B, 2), dtype=torch.float32, device=dev)
        alt = torch.empty(B, dtype=torch.float32, device=dev)
        prog = torch.empty(B, dtype=torch.float32, device=dev)
        fb = feedback if feedback is not None else getattr(self, "feedback", "student")
        if fb not in ("student", "teacher"):
            raise ValueError("Invalid feedback option")
        _lib.call("avdn_teacher_action", _lib.ptr(c), _lib.ptr(gt_t), int(pmax), _lib.ptr(len_t), _lib.ptr(e), B,
                  int(fb == "teacher"), _lib.ptr(ratio), _lib.ptr(alt), _lib.ptr(prog))
        self.launches += 1
        return ratio, alt, prog


def render_rollout_views(agent, batch, BT, x_out, att_out):
    """The B*T views of a training rollout: ``batch['images']`` as given, or rendered from ``corners_px`` [B,T,4,2]
    (``tile_idx`` [B,T] or None) into ``x_out``; the human-attention maps (``batch['att']``, else rendered into
    ``att_out`` when ``agent.nss_w != 0``, else None).  Returns (views, att, launches)."""
    att = batch.get("att")
    if "images" in batch:
        return batch["images"], att, 0
    r = agent.renderer
    ti = batch.get("tile_idx")
    ti = None if ti is None else ti.reshape(-1)
    minv = r.homography(batch["corners_px"].view(BT, 4, 2))
    r.render(None, ti, views=False, norm_nhwc=True, minv=minv, out={"norm_nhwc": x_out})
    n = 2
    if att is None and agent.nss_w != 0:
        r.render(None, ti, views=False, att=True, minv=minv, out={"att": att_out})
        att = att_out
        n += 1
    return x_out, att, n


def rollout_trunk_forward(agent, x, B, T, frames_out, bn_per_step=None):
    """Train-mode trunk pass of a rollout's views ``x`` [B*T,224,224,4] into ``frames_out`` [B*T,512,7,7].
    ``bn_per_step`` (default ``args.bn_per_step``, false): the reference's BatchNorm semantics -- one pass per time
    step over that step's B views (its own batch statistics, one running-statistics update per step,
    agent.py:593), each kept for its own backward -- instead of one pass over all B*T views (DESIGN.md §8).
    Returns (engine, per-step engines or None, launch count before the passes, launches)."""
    vm, dev = agent.vision_model, agent.device
    if bn_per_step is None:
        bn_per_step = bool(getattr(agent.args, "bn_per_step", False))
    if not bn_per_step:
        teng = vm.engine(B * T, 224, 224, dev)
        l0 = teng.launches
        DN._trunk_forward(vm, teng, x, True, out=frames_out)
        return teng, None, l0, 0
    key = ("rollout_steps", B, T)
    sb = agent._bufs.get(key)
    if sb is None:
        sb = dict(x=[torch.empty((B, 224, 224, 4), dtype=torch.bfloat16, device=dev) for _ in range(T)],
                  f=torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev),
                  df=torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev))
        agent._bufs[key] = sb
    tengs = [vm.engine(B, 224, 224, dev, slot=1 + t) for t in range(T)]
    l0 = sum(e.launches for e in tengs)
    x5 = x.view(B, T, 224, 224, 4)
    f5 = frames_out.view(B, T, 512, 49)
    for t in range(T):
        sb["x"][t].copy_(x5[:, t])
        DN._trunk_forward(vm, tengs[t], sb["x"][t], True, out=sb["f"])
        f5[:, t].copy_(sb["f"].view(B, 512, 49))
    return tengs[0], tengs, l0, 2 * T


def rollout_trunk_backward(agent, teng, tengs, l0, d_frames, B, T, after_layer=None, flush_layers=None):
    """Backward of ``rollout_trunk_forward`` from ``d_frames`` [B*T,512,49]; parameter gradients accumulate into
    the trunk's arena.  With per-step passes every pass runs back through its own activations and the last one
    (step 0) carries ``after_layer`` / ``flush_layers`` (the data-parallel buckets).  Returns the launches."""
    vm = agent.vision_model
    if tengs is None:
        DN._trunk_backward(vm, teng, d_frames.view(-1, 512, 7, 7), after_layer=after_layer, flush_layers=flush_layers)
        return teng.launches - l0
    sb = agent._bufs[("rollout_steps", B, T)]
    d5 = d_frames.view(B, T, 512, 49)
    for t in reversed(range(T)):
        sb["df"].view(B, 512, 49).copy_(d5[:, t])
        last = (t == 0)
        DN._trunk_backward(vm, tengs[t], sb["df"], after_layer=after_layer if last else None,
                           flush_layers=flush_layers if last else None)
    return T + sum(e.launches for e in tengs) - l0


def student_rollout_targets(agent, batch, res, gt_path_corners):
    """Training targets of a no-grad greedy rollout ``res`` (``rollout_greedy``'s result for ``batch``): the
    ``teacher_action`` target of every step in one launch (student feedback, agent.py:655-661) and the pixel corners
    of every pose.  Returns (dict of [B,T,...] tensors ``corners_px``, ``tile_idx``, ``gt_xy``, ``gt_alt``,
    ``gt_prog``; ``ended_before`` [T,B] u8 -- the sample had stopped before step t; T)."""
    T = int(res.get("steps", res["ended"].shape[0]))
    corners = res["corners"][:T]                                   # [T,B,4,2] gps
    B = corners.shape[1]
    ended_before = torch.zeros((T, B), dtype=torch.uint8, device=agent.device)
    ended_before[1:] = res["ended"][:T - 1]
    tgt_xy, tgt_alt, prog = agent.teacher_action(corners.reshape(T * B, 4, 2),
                                                 [gt_path_corners[k % B] for k in range(T * B)],
                                                 ended_before.reshape(-1), feedback="student")
    geo = batch["geo"].contiguous()
    px = torch.empty((T * B, 4, 2), dtype=torch.int32, device=agent.device)
    _lib.call("avdn_gps_to_pixels", _lib.ptr(corners.reshape(T * B, 4, 2).contiguous()),
              _lib.ptr(geo.repeat(T, 1).contiguous()), T * B, _lib.ptr(px))
    tb = lambda a: a.view(T, B, *a.shape[1:]).transpose(0, 1).contiguous()
    ti = batch.get("tile_idx")
    out = dict(corners_px=tb(px), tile_idx=None if ti is None else ti.view(B, 1).expand(B, T).contiguous(),
               gt_xy=tb(tgt_xy.float()), gt_alt=tb(tgt_alt.float()), gt_prog=tb(prog.float()))
    return out, ended_before, T
