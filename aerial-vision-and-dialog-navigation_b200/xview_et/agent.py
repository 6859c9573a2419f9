"""``NavCMTAgent`` -- the training / inference agent of the HAA-Transformer
(mirror of src/xview_et/agent.py, hot-path subset).

What is here
------------
* ``train_step``: ONE fused, device-resident training iteration of BASELINE
  configs[1]: render the B*T views of the batch (stage 1) -> Darknet trunk in
  train mode (stage 2) -> ET forward, loss, backward (stage 3) -> Darknet
  backward -> (data-parallel gradient all-reduce) -> clip + AdamW.  No autograd
  graph, no host round trip besides the final loss read.
* ``forward_loss``: the same forward + loss without backward (validation).
* ``NSS`` (agent.py:256-270), ``postprocess_waypoints`` (agent.py:637-653,745-752),
  ``move_view_corners`` / ``get_direction`` (agent.py:83-101,285-384: host float64,
  restated because the reference evaluates them on the host per sample),
  ``save`` / ``load`` (agent.py:899-940; ``lang_model`` is written when one is attached, optimiser
  moments in the flat-arena format).

* ``rollout_greedy``: the student-feedback (inference / validation) loop of ``rollout``
  (agent.py:580-760) with the growing episode history: every step renders the B current views,
  runs the trunk in eval mode, appends the features and the heading to the history, runs the ET
  over the t+1 steps seen so far, discretises the waypoint and moves the view -- all on the device;
  the host reads the B stop flags once per step (the reference's ``lenths`` bookkeeping).

* ``rollout(train_ml, not_in_train, nss_w)`` / ``train(loader, n_epochs, feedback, nss_w_weighting)`` /
  ``test(loader, ...)``: the reference's agent loop with its signatures over ``self.env`` (an ``ANDHNavBatch``):
  tokenizer -> ``CustomBERTModel`` -> poses of the rollout (teacher: ground-truth actions, ``avdn_teacher_action`` +
  ``avdn_waypoint_step`` on the device; student: a no-grad greedy rollout) -> ``train_rollout_step`` (views, trunk,
  T encoder passes with loss and backward) -> trajectory dicts, ``self.loss``, ``self.logs['IL_loss']``.

* ``student_rollout_step`` (``rollout`` with ``args.on_policy_student``): the reference's on-policy student-feedback
  training rollout in one pass -- every step renders the current views, runs its own train-mode trunk pass and the
  ET in train mode over the history, takes the step's loss and backward, and moves the simulator by that same
  train-mode prediction.

Both training rollouts run each step of their ET pass as ``_history_step_forward`` and ``_history_step_backward``;
``train_step`` and both rollouts end in ``_finish_backward`` (BERT backward, all-reduce, trunk backward, optimiser).
``history_lengths`` gives the ``lenths`` of a rollout whose poses are known in advance.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import _lib
from ..env import ViewRenderer
from ..models.ET_haa import ET
from ..models import dark_net as DN
from ..models.dark_net import Darknet
from ..optim import FusedAdamW
from .. import parallel
from ..agent_common import (RolloutTrainer, pack_gt_paths, render_rollout_views, rollout_pose_batch,
                            rollout_step_bufs, rollout_trunk_backward, rollout_trunk_forward, student_targets)

PI_REF = 3.14159


def get_direction(start, end):
    """src/xview_et/agent.py:83-101 (host float64)."""
    vec = np.array(end) - np.array(start)
    if vec[1] > 0:
        ang = np.arctan(vec[0] / vec[1]) / 1.57 * 90
    elif vec[1] < 0:
        ang = np.arctan(vec[0] / vec[1]) / 1.57 * 90 + 180
    else:
        ang = 90 if np.sign(vec[0]) == 1 else 270
    return (360 - ang + 90) % 360


def history_lengths(ended):
    """The ``lenths`` of a rollout (agent.py:603-620): the history length each sample's ET sees at step t -- it grows
    by one every step until the sample has ended, then stays.  ``ended`` host bool [T,B]: the sticky stop flags after
    each step.  Returns int64 [B,T]."""
    alive = np.ones(ended.shape, dtype=bool)
    alive[1:] = ~ended[:-1]
    return np.cumsum(alive, axis=0).T


class NavCMTAgent(RolloutTrainer):
    def __init__(self, args, rank=0, world_size=1, device=None, process_group=None):
        if not torch.cuda.is_available():
            raise RuntimeError("NavCMTAgent needs a CUDA device (sm_100); there is no CPU fallback")
        _lib.lib()
        self.args = args
        self.rank, self.world = rank, world_size
        self.pg = process_group
        self.device = torch.device(device if device is not None else "cuda")
        self.results = {}
        self.losses = []
        self.logs = {"IL_loss": []}
        self.env = []
        self.vision_model = Darknet(args.darknet_model_file, 224).to(self.device)
        wf = getattr(args, "darknet_weight_file", None)
        if wf and os.path.exists(wf):                           # agent.py:136-141
            new_state = torch.load(wf, map_location=self.device)
            state = self.vision_model.state_dict()
            state.update({k: v for k, v in new_state["model"].items() if k in state})
            self.vision_model.load_state_dict(state)
        self.vln_model = ET(args).to(self.device)
        self.vln_model.drop_rank = rank              # data-parallel replicas draw different dropout masks
        self.tokenizer = getattr(args, "tokenizer", None)     # agent.py:124 (BertTokenizerFast; no vocabulary offline)
        self.feedback = "student"
        self.env_name = ""
        self.loss = 0
        self.exposed_events = None                   # bench: [(event, event)] around the wait for the last gradient bucket
        lr = getattr(args, "lr", 1e-5)
        if getattr(args, "optim", "adamW") not in ("adamW", "adam"):
            raise ValueError("optim must be 'adam' or 'adamW' (agent.py:151)")
        if getattr(args, "optim", "adamW") == "adam":
            raise NotImplementedError("optim='adam' (no decoupled weight decay) is not implemented: use 'adamW'")
        # agent.py:153-156: one AdamW per model, default weight decay; only ET is clipped (agent.py:247)
        self.et_optimizer = FusedAdamW(self.vln_model.used_parameters(), lr=lr, max_norm=40.0)
        self.vision_model_optimizer = FusedAdamW(dict(self.vision_model.named_parameters()), lr=lr)
        self.vln_model._grad_arena = self.et_optimizer.grads
        self.vision_model._grad_arena = self.vision_model_optimizer.grads
        self.optimizers = (self.et_optimizer, self.vision_model_optimizer)
        # language encoder (agent.py:125-126,155: trained with its own AdamW): built on demand, see attach_lang_model
        self.lang_model, self.lang_optimizer = None, None
        self.renderer = ViewRenderer(self.device)
        self.use_graphs = os.environ.get("AVDN_CUDA_GRAPHS", "1") != "0"     # rollouts replay the frozen trunk pass
        self.loss_total = torch.zeros(1, dtype=torch.float64, device=self.device)
        self._bufs = {}
        self.launches = 0
        self._comm_stream = torch.cuda.Stream(self.device) if world_size > 1 else None
        self._ar_bf16 = str(getattr(args, "allreduce_dtype", os.environ.get("AVDN_ALLREDUCE_DTYPE", "fp32"))) == "bf16"
        self._ar_bufs = {}
        self._buckets = None
        if world_size > 1:
            self.broadcast_parameters()

    # ------------------------------------------------------------ distributed
    def attach_lang_model(self, lang_model=None, lr=None):
        """Put ``CustomBERTModel`` into the training loop (src/xview_et/agent.py:125-126,155,249): ``train_step``
        then takes ``input_ids`` / ``attention_mask`` (and optionally ``cls_input_ids`` / ``cls_attention_mask``: the
        reference's second pass over pre_dialogs + instructions that produces ``linear_cls``, agent.py:530-538)
        instead of ``lang`` / ``lang_cls``, and the gradients of both
        flow back into BERT and its head (one encoder pass per step = the reference's ``train_val_on_full`` mode,
        agent.py:530-538)."""
        lm = super().attach_lang_model(lang_model, lr)
        if self.world > 1:
            # every rank built (and randomly initialised) its own encoder: replicas start from rank 0's, like the
            # other two models in __init__
            parallel.broadcast_([self.lang_optimizer.p], 0, self.pg)
        return lm

    def broadcast_parameters(self):
        """Replicas start identical (DDP semantics): rank 0's arenas and BN buffers."""
        parallel.broadcast_([opt.p for opt in self.optimizers], 0, self.pg)
        parallel.broadcast_(list(self.vision_model.buffers()), 0, self.pg)

    def _trunk_buckets(self, eng):
        """Slices of the trunk's gradient arena in backward-completion order.  The deep
        7x7 / 14x14 blocks hold most parameters and finish first; the shallow blocks
        hold most of the time: 3 buckets let NCCL run under the rest of the backward."""
        if self._buckets is None:
            offs = self.vision_model_optimizer.offsets
            first = [offs[f"module_list.{L.idx}.conv_{L.idx}.weight"][0] for L in eng.layers]
            self._buckets = parallel.bucket_edges(first, self.vision_model_optimizer.n)
        return self._buckets

    def _allreduce_async(self, flat, lo, hi):
        """Sum ``flat[lo:hi]`` (a slice of a gradient arena) over the ranks on the communication stream, behind
        everything enqueued so far.  ``args.allreduce_dtype == 'bf16'`` (or AVDN_ALLREDUCE_DTYPE=bf16) ships the
        bucket as bf16 -- half the NVLink bytes; every rank receives the same rounded sum, so the replicas stay
        bit-identical -- the default is fp32."""
        cs = self._comm_stream
        cs.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cs):
            if self._ar_bf16:
                buf = self._ar_bufs.get(flat.data_ptr())
                if buf is None:
                    buf = torch.empty(flat.numel(), dtype=torch.bfloat16, device=flat.device)
                    self._ar_bufs[flat.data_ptr()] = buf
                buf[lo:hi].copy_(flat[lo:hi])
                parallel.allreduce_sum_(buf, lo, hi, self.pg)
                flat[lo:hi].copy_(buf[lo:hi])
            else:
                parallel.allreduce_sum_(flat, lo, hi, self.pg)

    # ----------------------------------------------------------------- buffers
    def _get_bufs(self, B, T):
        key = (B, T)
        b = self._bufs.get(key)
        if b is None:
            dev = self.device
            b = dict(
                x=torch.empty((B * T, 224, 224, 4), dtype=torch.bfloat16, device=dev),
                att=torch.empty((B, 224, 224), dtype=torch.uint8, device=dev),
                frames=torch.empty((B * T, 512, 7, 7), dtype=torch.float32, device=dev),
                d_frames=torch.empty((B * T, 512, 49), dtype=torch.float32, device=dev),
                d_output=torch.empty((B, 4), dtype=torch.float32, device=dev),
                d_h_sali=torch.empty((B, 64), dtype=torch.float32, device=dev),
                loss_i=torch.empty(B, dtype=torch.float64, device=dev),
            )
            self._bufs[key] = b
        return b

    # ------------------------------------------------------------------- steps
    def _forward(self, batch, train):
        """Stages 1-3 forward + loss.  ``batch`` (device tensors unless noted):
        ``corners_px`` i32 [B,T,4,2] pose corners (FL,FR,BR,BL; pixel x,y) or ``images``
        bf16 [B*T,224,224,4] (pre-rendered, normalised NHWC); ``tile_idx`` i32 [B,T] or None;
        ``lang`` f32 [B,L,768]; ``lang_cls`` f32 [B,49]; ``directions`` f32 [B,T,2];
        ``lenths`` host list[int]; ``gt_xy`` [B,2], ``gt_alt`` [B], ``gt_prog`` [B] f32;
        optional ``att`` u8 [B,224,224], ``jitter`` f32 [B]; or, with an attached language model, ``input_ids`` /
        ``attention_mask`` (and optionally ``cls_input_ids`` / ``cls_attention_mask``) instead of ``lang`` /
        ``lang_cls``.  Sets ``self._ctx = (trunk engine, ET engine, buffers)``; returns ``(output, h_sali, BERT
        engines of the training pass or None, trunk launch count before the pass, ET launch count before the pass)``."""
        ptr = _lib.ptr
        lengs = None
        if "input_ids" in batch:
            if train:
                seq, lin, *lengs = self._lang_train_forward(batch)
            else:
                seq, lin = self._lang_eval_forward(batch)
            batch = dict(batch, lang=seq, lang_cls=lin)
        lang, lang_cls, dirs = batch["lang"], batch["lang_cls"], batch["directions"]
        B, T = dirs.shape[0], dirs.shape[1]
        L = lang.shape[1]
        bufs = self._get_bufs(B, T)
        n = 0
        att = batch.get("att")
        if "images" in batch:
            x = batch["images"]
        else:
            r = self.renderer
            c = batch["corners_px"].view(B * T, 4, 2)
            ti = batch.get("tile_idx")
            minv = r.homography(c)
            r.render(None, None if ti is None else ti.view(-1), views=False, norm_nhwc=True, minv=minv,
                     out={"norm_nhwc": bufs["x"]})
            n += 2
            x = bufs["x"]
            if att is None and self.nss_w != 0:
                # human-attention target of the current (last) step of every episode (env.py:292-293)
                last = minv.view(B, T, 3, 3)[:, -1].contiguous()
                r.render(None, None if ti is None else ti.view(B, T)[:, -1].contiguous(), views=False, att=True,
                         minv=last, out={"att": bufs["att"]})
                att = bufs["att"]
                n += 2
        vm = self.vision_model
        teng = vm.engine(B * T, 224, 224, self.device)
        l0 = teng.launches
        DN._trunk_forward(vm, teng, x, train, out=bufs["frames"])
        et = self.vln_model
        eng = et.engine(B, L, T, self.device)
        e0 = eng.launches
        et.train(bool(train) and not getattr(self.args, "no_dropout", False))
        eng.set_dropout(*et.dropout_config())
        output, h_sali = eng.forward(bufs["frames"].view(B * T, 512, 49), lang, lang_cls, dirs, batch["lenths"],
                                     et.encoder_vl.enc_pos.pe[0])
        self.loss_total.zero_()
        scale = float(self.train_ml) / B                               # agent.py:883-885
        _lib.call("avdn_loss", ptr(output), ptr(h_sali), ptr(batch["gt_xy"]), ptr(batch["gt_alt"]),
                  ptr(batch["gt_prog"]), ptr(att), ptr(batch.get("jitter")), B, float(self.nss_w),
                  int(getattr(self.args, "nss_r", 0)), scale, ptr(self.loss_total), ptr(bufs["loss_i"]),
                  ptr(bufs["d_output"]), ptr(bufs["d_h_sali"]))
        n += 2
        self._ctx = (teng, eng, bufs)
        self.launches += n
        return output, h_sali, lengs, l0, e0

    def forward_loss(self, batch):
        """Validation: forward + loss (trunk in eval mode).  Returns (loss, output, h_sali)."""
        self.vision_model.eval()
        output, h_sali, _, _, _ = self._forward(batch, False)
        return self.loss_total.clone(), output, h_sali

    def train_step(self, batch, sync_loss=False):
        """One training iteration (see the module docstring).  Returns the device
        tensor holding the step loss (float64 [1]); ``sync_loss=True`` returns a host float."""
        self.vision_model.train()
        for opt in self.optimizers:
            opt.zero_grad()
        self.launches += 2
        _, _, lengs, l0, e0 = self._forward(batch, True)
        teng, eng, bufs = self._ctx
        lang = None
        if lengs is None:
            eng.backward(bufs["d_output"], bufs["d_h_sali"], d_frames=bufs["d_frames"])
        else:
            d_cls = torch.zeros((eng.B, 49), dtype=torch.float32, device=self.device)
            _, d_lang = eng.backward(bufs["d_output"], bufs["d_h_sali"], d_frames=bufs["d_frames"], need_lang_grad=True,
                                     d_lang_cls=d_cls)
            lang = (*lengs, d_lang, d_cls)
        n = self._finish_backward(lang, teng, None, l0, bufs["d_frames"], eng.B, eng.T)
        self.launches += n + (eng.launches - e0)
        self._log_loss()
        if sync_loss:
            return float(self.loss_total.item())
        return self.loss_total

    def _finish_backward(self, lang, teng, tengs, l0, d_frames, B, T, steps=None, step=True):
        """What follows the ET backward of ``train_step`` and both training rollouts: BERT's backward of ``lang`` =
        (engine, cls engine, d_lang, d_cls) from ``_lang_train_forward``, or None; with ``step`` on more than one GPU
        the all-reduce of the language and ET arenas and of the trunk's gradient buckets as the trunk backward
        completes them (gradients are reduced once, after the iteration's last rollout); ``rollout_trunk_backward``
        (arguments as there); then, with ``step``, every optimiser with ``grad_scale = 1/world``.  Returns the
        launches of the trunk, forward included, and of the optimisers."""
        if lang is not None:
            self._lang_train_backward(*lang)
        dp = self.world > 1 and step
        hook = flush = None
        if dp:
            if self.lang_optimizer is not None:
                self._allreduce_async(self.lang_optimizer.g, 0, self.lang_optimizer.n)
            self._allreduce_async(self.et_optimizer.g, 0, self.et_optimizer.n)
            buckets = {c: (lo, hi) for c, lo, hi in self._trunk_buckets(teng)}
            hook = lambda li: (self._allreduce_async(self.vision_model_optimizer.g, *buckets[li])
                               if li in buckets else None)
            flush = set(buckets)
        n = rollout_trunk_backward(self, teng, tengs, l0, d_frames, B, T, after_layer=hook, flush_layers=flush,
                                   steps=steps)
        if dp:
            self._wait_comm()
        if step:
            gs = 1.0 / self.world
            for opt in self.optimizers:
                n += opt.step(grad_scale=gs)
        return n

    def _wait_comm(self):
        """The optimiser waits for the last gradient bucket; with ``exposed_events`` set (bench) the wait is bracketed
        by CUDA events: the all-reduce time the backward pass did not hide."""
        cur = torch.cuda.current_stream()
        if self.exposed_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(cur)
            cur.wait_stream(self._comm_stream)
            e1.record(cur)
            self.exposed_events.append((e0, e1))
        else:
            cur.wait_stream(self._comm_stream)

    def _train_rollout_step(self, batch, sync_loss=False, zero=True, step=True, collect=None, bn_per_step=None):
        """One teacher-forced training ROLLOUT (agent.py:580-760, 883-885, 245-251) as one batched pass: the loss is
        taken at EVERY step t of every episode on the history ``[:t+1]``, summed over steps and samples and scaled
        by ``ml_weight / B``, as the reference accumulates ``ml_loss`` over its step loop.

        The poses of all steps are known before the pass (teacher feedback: the ground-truth path; student
        feedback: a no-grad ``rollout_greedy`` -- see ``student_batch``), so the B*T views are rendered and pushed
        through the trunk ONCE (forward and backward); the transformer then makes the reference's T encoder calls
        over the growing history, each followed at once by its loss and its backward pass; the gradient of a
        frame is the sum over the steps whose history contains it.  (The reference's train-mode trunk normalises
        each step's B views with their own batch statistics; here the statistics are over all B*T views,
        DESIGN.md §8.)

        ``batch``: ``corners_px`` i32 [B,T,4,2] (or ``images``), ``tile_idx`` i32 [B,T] | None, ``lang`` [B,L,768],
        ``lang_cls`` [B,49] (or, with an attached language model, ``input_ids`` / ``attention_mask`` and optionally
        ``cls_input_ids`` / ``cls_attention_mask``: the encoder runs once per rollout and receives the gradients of
        every step), ``directions`` f32 [B,T,2], ``gt_xy`` [B,T,2], ``gt_alt`` / ``gt_prog`` [B,T], optional
        ``lenths`` host int [B][T] (history length seen at step t: stops growing once a sample has ended,
        agent.py:603-620; default t+1), ``att`` u8 [B,T,224,224] (default: rendered from the poses), ``jitter``
        f32 [B,T].  ``zero=False`` keeps the gradients already in the arenas, ``step=False`` leaves them there
        without an optimiser step (``train_iteration`` chains the two rollouts of an iteration that way).
        ``nss_w`` / ``train_ml`` (``train_rollout_step``): this rollout's loss weights (default: ``args.nss_w``,
        ``args.ml_weight``); with ``nss_w == 0`` no human-attention maps are rendered.  ``collect``: a list that
        receives the per-step ``output`` [B,4] tensors (the trajectory log of ``rollout``).
        ``bn_per_step`` (default ``args.bn_per_step``, false): the reference's BatchNorm semantics -- one train-mode
        trunk pass per time step over that step's B views (its own batch statistics, one running-statistics update
        per step, agent.py:593), each pass kept for its own backward -- instead of one pass over all B*T views."""
        self.vision_model.train()
        n = 0
        if zero:
            for opt in self.optimizers:
                opt.zero_grad()
            n += 2
        lengs = None
        if "input_ids" in batch:
            # the language encoder runs once per rollout (agent.py:519-538) and collects the gradients of all steps
            seq, lin, *lengs = self._lang_train_forward(batch)
            batch = dict(batch, lang=seq, lang_cls=lin)
        dirs = batch["directions"].contiguous().float()
        B, T = dirs.shape[0], dirs.shape[1]
        BT = B * T
        lang, lang_cls = batch["lang"].contiguous().float(), batch["lang_cls"].contiguous().float()
        dev = self.device
        bufs = self._get_bufs(B, T)
        key = ("rollout_train", B, T)
        xb = self._bufs.get(key)
        if xb is None:
            xb = dict(att=torch.empty((BT, 224, 224), dtype=torch.uint8, device=dev),
                      d_frames=torch.empty((BT, 512, 49), dtype=torch.float32, device=dev))
            self._bufs[key] = xb
        x, att, k = render_rollout_views(self, batch, BT, bufs["x"], xb["att"])
        n += k
        teng, tengs, l0, k = rollout_trunk_forward(self, x, B, T, bufs["frames"], bn_per_step)
        n += k
        # ---- step t: the encoder over the history [:t+1], its loss, and straight back (the loss is a sum over steps,
        #      so only one step's activations are alive at a time; every step adds into the one gradient arena) ----
        frames = bufs["frames"].view(B, T, 512, 49)
        d_frames = bufs["d_frames"].view(B, T, 512, 49)
        d_frames.zero_()
        lens = batch.get("lenths")
        gt_xy = batch["gt_xy"].float().transpose(0, 1).contiguous()     # [T,B,2]
        gt_alt = batch["gt_alt"].float().transpose(0, 1).contiguous()
        gt_prog = batch["gt_prog"].float().transpose(0, 1).contiguous()
        jit = batch.get("jitter")
        jit = None if jit is None else jit.float().transpose(0, 1).contiguous()
        att_t = None if att is None else att.view(B, T, 224, 224).transpose(0, 1).contiguous()
        n += 6
        self.vln_model.train(not getattr(self.args, "no_dropout", False))
        self.loss_total.zero_()
        d_lang = None                              # the sums of every step's lang / lang_cls gradients
        if lengs is not None:
            d_lang = (torch.zeros((B, lang.shape[1], 768), dtype=torch.float32, device=dev),
                      torch.zeros((B, 49), dtype=torch.float32, device=dev))
        et_launches = 0
        for t in range(T):
            lens_t = [int(lens[i][t]) for i in range(B)] if lens is not None else [t + 1] * B
            eng, e0, output = self._history_step_forward(t, frames, dirs, lang, lang_cls, lens_t,
                                                         (gt_xy[t], gt_alt[t], gt_prog[t]),
                                                         None if att_t is None else att_t[t],
                                                         None if jit is None else jit[t], bufs)
            if collect is not None:
                collect.append(output.detach().clone())
            et_launches += self._history_step_backward(eng, e0, bufs, xb["d_frames"], d_frames, d_lang)
            n += 4
        self._ctx = (teng, eng, bufs)
        n += self._finish_backward(None if lengs is None else (*lengs, *d_lang), teng, tengs, l0, bufs["d_frames"],
                                   B, T, step=step)
        self.launches += n + et_launches
        self._log_loss()
        return float(self.loss_total.item()) if sync_loss else self.loss_total

    def _history_step_forward(self, t, frames, dirs, lang, lang_cls, lens, targets, att, jitter, gb):
        """Step t of a training rollout's ET pass: the ET over the history ``[:t+1]`` of ``frames`` [B,T,512,49] /
        ``dirs`` [B,T,2] (fresh dropout masks) with the history lengths ``lens``, then the step's ``avdn_loss`` against
        ``targets`` = (xy [B,2], alt [B], prog [B]) into ``loss_total`` and ``gb``'s output gradients.  Returns
        (engine, its launch count before the step, output [B,4])."""
        ptr = _lib.ptr
        et = self.vln_model
        B, L, Tc = lang.shape[0], lang.shape[1], t + 1
        eng = et.engine(B, L, Tc, self.device)
        e0 = eng.launches
        eng.set_dropout(*et.dropout_config())
        output, h_sali = eng.forward(frames[:, :Tc].contiguous().view(B * Tc, 512, 49), lang, lang_cls,
                                     dirs[:, :Tc].contiguous(), lens, et.encoder_vl.enc_pos.pe[0])
        xy, alt, prog = targets
        _lib.call("avdn_loss", ptr(output), ptr(h_sali), ptr(xy), ptr(alt), ptr(prog), ptr(att), ptr(jitter), B,
                  float(self.nss_w), int(getattr(self.args, "nss_r", 0)), float(self.train_ml) / B,   # agent.py:883-885
                  ptr(self.loss_total), ptr(gb["loss_i"]), ptr(gb["d_output"]), ptr(gb["d_h_sali"]))
        return eng, e0, output

    def _history_step_backward(self, eng, e0, gb, d_frames_t, d_frames, d_lang):
        """The backward of ``_history_step_forward``'s step: the frame gradients (into the scratch ``d_frames_t``) are
        added into the history's ``d_frames`` [B,T,512,49], and with ``d_lang`` = (sum [B,L,768], sum [B,49]) the
        language gradients into it.  Returns the step's launches since ``e0``."""
        B, L, Tc = eng.B, eng.L, eng.T
        if d_lang is None:
            df, _ = eng.backward(gb["d_output"], gb["d_h_sali"], d_frames=d_frames_t[:B * Tc])
        else:
            df, dl = eng.backward(gb["d_output"], gb["d_h_sali"], d_frames=d_frames_t[:B * Tc], need_lang_grad=True,
                                  d_lang_cls=d_lang[1])
            d_lang[0].add_(dl.view(B, L, 768))
        d_frames[:, :Tc] += df.view(B, Tc, 512, 49)
        return eng.launches - e0 + 1 + (d_lang is not None)

    @torch.no_grad()
    def student_batch(self, batch, gt_path_corners, max_action_len=None):
        """The student-feedback half of a training iteration (agent.py:245-251 runs ``rollout`` twice): a no-grad
        greedy rollout fixes the poses, ``teacher_action`` supplies the target of every step (one launch), and the
        result is a ``train_rollout_step`` batch.  ``batch`` as for ``rollout_greedy``; returns the training batch
        (device tensors; ``lenths`` from the steps each sample was alive)."""
        res = self.rollout_greedy(batch, max_action_len=max_action_len)
        T = int(res["steps"])
        corners, ended = res["corners"][:T], res["ended"][:T]
        out = rollout_pose_batch(corners, batch["geo"], batch.get("tile_idx"),
                                 student_targets(self, corners, ended, gt_path_corners))
        rad = res["directions"][:T].float() / 180 * PI_REF
        out.update(lang=batch["lang"], lang_cls=batch["lang_cls"],
                   directions=torch.stack([torch.sin(rad), torch.cos(rad)], -1).transpose(0, 1).contiguous(),
                   lenths=history_lengths(ended.cpu().numpy().astype(bool)).tolist())
        return out

    _LANG_KEYS = ("lang", "lang_cls", "input_ids", "attention_mask", "cls_input_ids", "cls_attention_mask")

    def student_rollout_step(self, batch, gt_path_corners, max_action_len=None, nss_w=None, train_ml=None, zero=True,
                             step=True, sync_loss=False, collect=None, bn_per_step=None):
        """One on-policy student-feedback training rollout, as the reference runs it (src/xview_et/agent.py:580-760):
        every step runs the trunk and the ET in train mode, takes the step's loss, and the simulator moves by that
        same train-mode prediction (stop threshold 0.5), so the model is trained on the states its own train-mode
        policy visits.  Step t: render the B current views into trunk slot ``1 + t`` and run a train-mode pass on
        the step's own batch statistics (kept for the backward) -> the features and the heading join the history,
        ``lenths`` grows for the samples that have not ended (agent.py:603-620) -> the ``teacher_action`` target at
        the pose -> the ET over the history ``[:t+1]`` with fresh dropout masks and ``avdn_loss``
        (``_history_step_forward``) -> ``avdn_waypoint_step`` -> the ET backward of the step, its frame gradients
        added into the history's (``_history_step_backward``).  One host read of the B stop flags per step gives the
        next step's ``lenths``; the loop stops after the step at which every sample has ended (agent.py:773-774).
        Then ``_finish_backward``, as in ``train_rollout_step``: the BERT backward, the trunk backward of the executed
        passes and (``step``) the data-parallel reduction and the optimiser step.

        ``batch`` as for ``rollout_greedy``; with an attached language model it may carry ``input_ids`` /
        ``attention_mask`` (and ``cls_*``) instead of ``lang`` / ``lang_cls``: BERT then runs once in train mode,
        its outputs steer the rollout and one backward receives the gradients of every step.  ``gt_path_corners``:
        per sample the ``[n_i,4,2]`` ground-truth view corners.  The per-step trunk passes are required
        (``bn_per_step`` false raises ``ValueError``): the views of step t+1 depend on the features of step t.  What
        the rollout visited, and the ``train_rollout_step`` batch of those poses, is kept in ``self._last_rollout``."""
        if bn_per_step is None:
            bn_per_step = bool(getattr(self.args, "bn_per_step", True))
        if not bn_per_step:
            raise ValueError("an on-policy student rollout needs one trunk pass per step (bn_per_step): the views of "
                             "step t+1 depend on the features of step t")
        with self._weights(nss_w, train_ml):
            return self._student_rollout_step(batch, gt_path_corners, max_action_len, zero, step, sync_loss, collect)

    def _on_policy_bufs(self, B, T):
        """Pose, history and gradient buffers of an on-policy training rollout of B episodes and T steps."""
        key = ("on_policy", B, T)
        b = self._bufs.get(key)
        if b is None:
            dev = self.device
            f64, i32, f32 = torch.float64, torch.int32, torch.float32
            b = dict(corners=torch.empty((B, 4, 2), dtype=f64, device=dev),
                     cur_dir=torch.empty(B, dtype=f64, device=dev),
                     ended=torch.empty(B, dtype=torch.uint8, device=dev),
                     minv=torch.empty((B, 3, 3), dtype=f64, device=dev),
                     att=torch.empty((B, 224, 224), dtype=torch.uint8, device=dev),
                     corners_hist=torch.empty((T + 1, B, 4, 2), dtype=f64, device=dev),
                     dir_hist=torch.empty((T + 1, B), dtype=f64, device=dev),
                     px_hist=torch.empty((T, B, 4, 2), dtype=i32, device=dev),
                     ended_before=torch.zeros((T, B), dtype=torch.uint8, device=dev),
                     ended_hist=torch.empty((T, B), dtype=torch.uint8, device=dev),
                     output_hist=torch.empty((T, B, 4), dtype=f32, device=dev),
                     tgt_xy=torch.empty((T, B, 2), dtype=f32, device=dev),
                     tgt_alt=torch.empty((T, B), dtype=f32, device=dev),
                     tgt_prog=torch.empty((T, B), dtype=f32, device=dev),
                     frames=torch.empty((B, T, 512, 49), dtype=f32, device=dev),
                     dirs=torch.empty((B, T, 2), dtype=f32, device=dev),
                     d_frames=torch.empty((B, T, 512, 49), dtype=f32, device=dev),
                     d_frames_t=torch.empty((B * T, 512, 49), dtype=f32, device=dev),
                     d_output=torch.empty((B, 4), dtype=f32, device=dev),
                     d_h_sali=torch.empty((B, 64), dtype=f32, device=dev),
                     loss_i=torch.empty(B, dtype=f64, device=dev),
                     angle=torch.empty((T, B), dtype=i32, device=dev),
                     altitude=torch.empty((T, B), dtype=i32, device=dev),
                     dist=torch.empty((T, B), dtype=f64, device=dev),
                     ended_h=torch.empty(B, dtype=torch.uint8, pin_memory=True))
            self._bufs[key] = b
        return b

    def _student_rollout_step(self, batch, gt_path_corners, max_action_len, zero, step, sync_loss, collect):
        ptr, call = _lib.ptr, _lib.call
        T = int(max_action_len if max_action_len is not None else getattr(self.args, "max_action_len", 20))
        dev = self.device
        n = 0
        if zero:
            for opt in self.optimizers:
                opt.zero_grad()
            n += 2
        lang_in = {k: batch[k] for k in self._LANG_KEYS if k in batch}
        lengs = None
        if "input_ids" in batch:
            # the language encoder runs once per rollout (agent.py:519-538): its train-mode outputs steer the rollout
            seq, lin, *lengs = self._lang_train_forward(batch)
            batch = dict(batch, lang=seq, lang_cls=lin)
        lang, lang_cls = batch["lang"].contiguous().float(), batch["lang_cls"].contiguous().float()
        B, L = lang.shape[0], lang.shape[1]
        vm, et, r = self.vision_model, self.vln_model, self.renderer
        vm.train()
        et.train(not getattr(self.args, "no_dropout", False))
        bf = self._on_policy_bufs(B, T)
        sb = rollout_step_bufs(self, B, T)
        geo = batch["geo"].contiguous()
        bounds = geo[:, :4].contiguous()
        ti = batch.get("tile_idx")
        gt_pack = pack_gt_paths(gt_path_corners, dev)              # once: the loop does no host packing
        bf["corners"].copy_(batch["corners_gps"])
        bf["cur_dir"].copy_(batch["directions"])
        bf["ended"].zero_()
        bf["d_frames"].zero_()
        no_dir = bool(getattr(self.args, "no_direction", False))
        if no_dir:
            bf["dirs"].zero_()
        self.loss_total.zero_()
        thr = float(self.STOP_THRESHOLD)
        d_lang = None                              # the sums of every step's lang / lang_cls gradients
        if lengs is not None:
            d_lang = (torch.zeros((B, L, 768), dtype=torch.float32, device=dev),
                      torch.zeros((B, 49), dtype=torch.float32, device=dev))
        lens = [0] * B
        lens_hist = []                                                 # [steps][B]: history length seen at step t
        ended_host = np.zeros(B, dtype=bool)
        tengs, l0, et_launches = [], 0, 0
        steps = T
        for t in range(T):
            # ---- 1. the pose and its observation (agent.py:742): the views into this step's trunk slot ----
            bf["corners_hist"][t].copy_(bf["corners"])
            bf["dir_hist"][t].copy_(bf["cur_dir"])
            if t > 0:
                bf["ended_before"][t].copy_(bf["ended"])
            px = bf["px_hist"][t]
            call("avdn_gps_to_pixels", ptr(bf["corners"]), ptr(geo), B, ptr(px))
            call("avdn_homography_from_corners", ptr(px), B, ptr(bf["minv"]))
            r.render(None, ti, views=False, norm_nhwc=True, minv=bf["minv"], out={"norm_nhwc": sb["x"][t]})
            att = None
            if self.nss_w != 0:
                r.render(None, ti, views=False, att=True, minv=bf["minv"], out={"att": bf["att"]})
                att = bf["att"]
                n += 1
            # ---- 2. train-mode trunk pass on the step's own batch statistics (agent.py:593), kept for the backward ----
            teng = vm.engine(B, 224, 224, dev, slot=1 + t)
            l0 += teng.launches
            tengs.append(teng)
            DN._trunk_forward(vm, teng, sb["x"][t], True, out=sb["f"])
            bf["frames"][:, t].copy_(sb["f"].view(B, 512, 49))
            # ---- 3. heading of the step (agent.py:605-606) and the history lengths (agent.py:603-620) ----
            if not no_dir:
                rad = bf["cur_dir"].float() / 180 * PI_REF
                bf["dirs"][:, t, 0] = torch.sin(rad)
                bf["dirs"][:, t, 1] = torch.cos(rad)
            for i in range(B):
                if not ended_host[i]:
                    lens[i] += 1
            lens_hist.append(list(lens))
            # ---- 4. the teacher's target at the pose (agent.py:655-661), 5. the ET over the history [:t+1] (train
            #      mode, fresh dropout masks) and 6. the step's loss ----
            xy, alt, prog = self.teacher_action(bf["corners"], gt_pack, bf["ended_before"][t], feedback="student")
            eng, e0, output = self._history_step_forward(t, bf["frames"], bf["dirs"], lang, lang_cls, lens,
                                                         (xy, alt, prog), att, None, bf)
            bf["tgt_xy"][t].copy_(xy)
            bf["tgt_alt"][t].copy_(alt)
            bf["tgt_prog"][t].copy_(prog)
            # ---- 7. the simulator moves by the train-mode prediction (agent.py:637-653,736-760) ----
            bf["output_hist"][t].copy_(output)
            if collect is not None:
                collect.append(output.detach().clone())
            call("avdn_waypoint_step", ptr(output), ptr(bf["corners"]), ptr(bounds), ptr(bf["cur_dir"]),
                 ptr(bf["ended"]), B, thr, int(t == T - 1), ptr(bf["angle"][t]), ptr(bf["dist"][t]),
                 ptr(bf["altitude"][t]))
            bf["ended_hist"][t].copy_(bf["ended"])
            # ---- 8. the step's backward straight away: one encoder's activations are alive at a time ----
            et_launches += self._history_step_backward(eng, e0, bf, bf["d_frames_t"], bf["d_frames"], d_lang)
            n += 19                                 # the step's other kernels outside the trunk and ET engines
            # ---- 9. the step's only host read: the stop flags (next lenths; agent.py:773-774 early exit) ----
            if t < T - 1:
                bf["ended_h"].copy_(bf["ended"])
                ended_host = bf["ended_h"].numpy().astype(bool)
                if ended_host.all():
                    steps = t + 1
                    break
        bf["corners_hist"][steps].copy_(bf["corners"])
        bf["dir_hist"][steps].copy_(bf["cur_dir"])
        self._ctx = (tengs[0], eng, bf)
        n += self._finish_backward(None if lengs is None else (*lengs, *d_lang), tengs[0], tengs, l0, bf["d_frames"],
                                   B, T, steps, step)
        self.launches += n + et_launches
        self._log_loss()
        # what the rollout visited (inspection / tests): poses before every step and after the last, stop flags,
        # train-mode outputs, targets, and the teacher-forced batch of the same poses
        # [steps,B,...] -> [B,steps,...], always a copy: the buffers are rewritten by the next rollout
        tb = lambda a: a[:steps].transpose(0, 1).clone(memory_format=torch.contiguous_format)
        lenths = np.array(lens_hist, dtype=np.int64).T                 # [B, steps]
        rb = dict(lang_in, corners_px=tb(bf["px_hist"]),
                  directions=bf["dirs"][:, :steps].clone(memory_format=torch.contiguous_format),
                  tile_idx=None if ti is None else ti.view(B, 1).expand(B, steps).contiguous(),
                  gt_xy=tb(bf["tgt_xy"]), gt_alt=tb(bf["tgt_alt"]), gt_prog=tb(bf["tgt_prog"]), lenths=lenths.tolist())
        self._last_rollout = dict(
            corners=bf["corners_hist"][:steps + 1].clone(), directions=bf["dir_hist"][:steps + 1].clone(),
            ended=bf["ended_hist"][:steps].clone(), output=bf["output_hist"][:steps].clone(), steps=steps,
            lenths=lenths, tgt_xy=bf["tgt_xy"][:steps].clone(), tgt_alt=bf["tgt_alt"][:steps].clone(),
            tgt_prog=bf["tgt_prog"][:steps].clone(), batch=rb)
        return float(self.loss_total.item()) if sync_loss else self.loss_total

    # ----------------------------------------------------------------- inference
    STOP_THRESHOLD = 0.5               # agent.py:738-745 (the LSTM agent uses 0.25)

    @torch.no_grad()
    def rollout_greedy(self, batch, max_action_len=None, stop_threshold=None, incremental=True):
        """Greedy (student-feedback) rollout of ``B`` episodes, the inference path of the HAA-Transformer
        (agent.py:580-760 with ``feedback == 'student'``, no teacher / loss).

        ``batch`` (device tensors): ``corners_gps`` f64 [B,4,2] (lat,lng; FL,FR,BR,BL = gt_path_corners[0]),
        ``directions`` [B] (starting_angle, degrees), ``geo`` f64 [B,5] = (bl_lat, bl_lng, tr_lat, tr_lng,
        lat_ratio), ``tile_idx`` i32 [B] or None, ``lang`` f32 [B,L,768], ``lang_cls`` f32 [B,49].

        Step t: observation at the current corners (env._get_obs, agent.py:769) -> Darknet, eval mode ->
        ``frames`` / ``directions`` grow by one step for EVERY sample, ``lenths`` only for the samples that
        have not ended (agent.py:603-620) -> ``ET`` over the t+1 steps -> post-processing, stop test
        (progress > 0.5 or last step) and ``move_view_corners`` (agent.py:637-653,736-760).  The loop ends
        early once every sample has ended (agent.py:773-774).

        ``incremental=True`` (default): step 0 runs the full encoder once, later steps compute only their
        two new rows per sample against cached keys / values (``ETDecodeState``: earlier rows cannot change
        under the causal mask); ``False`` re-runs the encoder over the whole history every step, exactly as
        the reference does.  The two agree to bf16 rounding for every sample that has not ended.

        Returns device tensors: ``corners`` [T+1,B,4,2], ``directions`` [T+1,B], ``ended`` [T,B],
        ``output`` [T,B,4], ``angle`` / ``altitude`` [T,B], ``dist`` [T,B], and ``steps`` (the number of
        steps actually run).  Rows after ``steps`` repeat the final state."""
        ptr, call = _lib.ptr, _lib.call
        T = int(max_action_len if max_action_len is not None else getattr(self.args, "max_action_len", 20))
        thr = float(self.STOP_THRESHOLD if stop_threshold is None else stop_threshold)
        lang, lang_cls = batch["lang"].contiguous().float(), batch["lang_cls"].contiguous().float()
        B, L = lang.shape[0], lang.shape[1]
        dev = self.device
        key = ("rollout", B, T)
        bf = self._bufs.get(key)
        if bf is None:
            f64, i32 = torch.float64, torch.int32
            bf = dict(x=torch.empty((B, 224, 224, 4), dtype=torch.bfloat16, device=dev),
                      frames=torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev),
                      frames_hist=torch.zeros((T, B, 512, 49), dtype=torch.float32, device=dev),
                      dirs_hist=torch.zeros((T, B, 2), dtype=torch.float32, device=dev),
                      corners=torch.empty((B, 4, 2), dtype=f64, device=dev),
                      cur_dir=torch.empty(B, dtype=f64, device=dev),
                      ended=torch.empty(B, dtype=torch.uint8, device=dev),
                      px=torch.empty((B, 4, 2), dtype=i32, device=dev),
                      minv=torch.empty((B, 3, 3), dtype=f64, device=dev),
                      corners_hist=torch.empty((T + 1, B, 4, 2), dtype=f64, device=dev),
                      dir_hist=torch.empty((T + 1, B), dtype=f64, device=dev),
                      ended_hist=torch.empty((T, B), dtype=torch.uint8, device=dev),
                      output_hist=torch.zeros((T, B, 4), dtype=torch.float32, device=dev),
                      angle=torch.zeros((T, B), dtype=i32, device=dev),
                      altitude=torch.zeros((T, B), dtype=i32, device=dev),
                      dist=torch.zeros((T, B), dtype=f64, device=dev))
            self._bufs[key] = bf
        geo = batch["geo"].contiguous()
        bounds = geo[:, :4].contiguous()
        ti = batch.get("tile_idx")
        bf["corners"].copy_(batch["corners_gps"])
        bf["cur_dir"].copy_(batch["directions"])
        bf["ended"].zero_()
        vm, et, r = self.vision_model, self.vln_model, self.renderer
        vm.eval()
        et.eval()
        teng = vm.engine(B, 224, 224, dev)
        l0 = teng.launches
        lens = [0] * B
        ended_host = [False] * B
        n, steps = 0, 0
        for t in range(T):
            steps = t + 1
            bf["corners_hist"][t].copy_(bf["corners"])
            bf["dir_hist"][t].copy_(bf["cur_dir"])
            # ---- observation -> trunk features of the step ----
            call("avdn_gps_to_pixels", ptr(bf["corners"]), ptr(geo), B, ptr(bf["px"]))
            call("avdn_homography_from_corners", ptr(bf["px"]), B, ptr(bf["minv"]))
            r.render(None, ti, views=False, norm_nhwc=True, minv=bf["minv"], out={"norm_nhwc": bf["x"]})
            if t == 0 or not self.use_graphs:
                DN._trunk_forward(vm, teng, bf["x"], False, out=bf["frames"], frozen=(t > 0))
            else:
                DN._trunk_forward_graphed(vm, teng, bf["x"], bf["frames"])
            bf["frames_hist"][t].copy_(bf["frames"].view(B, 512, 49))
            rad = bf["cur_dir"].float() / 180 * PI_REF                  # agent.py:605-606 (float32, pi = 3.14159)
            bf["dirs_hist"][t, :, 0] = torch.sin(rad)
            bf["dirs_hist"][t, :, 1] = torch.cos(rad)
            for i in range(B):
                if not ended_host[i]:
                    lens[i] += 1
            # ---- ET over the history [B, t+1, ...] ----
            Tc = t + 1
            pe = et.encoder_vl.enc_pos.pe[0]
            if incremental and t > 0:
                dec = et.decoder(B, L, T, dev)
                e0 = dec.launches
                output, _ = dec.step(t, bf["frames_hist"][t], bf["dirs_hist"][t], lang_cls, pe)
                n += dec.launches - e0
            else:
                frames = bf["frames_hist"][:Tc].permute(1, 0, 2, 3).contiguous().view(B * Tc, 512, 49)
                dirs = bf["dirs_hist"][:Tc].permute(1, 0, 2).contiguous()
                eng = et.engine(B, L, Tc, dev)
                e0 = eng.launches
                eng.set_dropout(0.0, 0.0, 0)
                output, _ = eng.forward(frames, lang, lang_cls, dirs, lens if not incremental else [1] * B, pe)
                n += eng.launches - e0
                if incremental:
                    et.decoder(B, L, T, dev).start()
            bf["output_hist"][t].copy_(output)
            # ---- simulator: post-processing, stop test, move_view_corners ----
            call("avdn_waypoint_step", ptr(output), ptr(bf["corners"]), ptr(bounds), ptr(bf["cur_dir"]),
                 ptr(bf["ended"]), B, thr, int(t == T - 1), ptr(bf["angle"][t]), ptr(bf["dist"][t]),
                 ptr(bf["altitude"][t]))
            bf["ended_hist"][t].copy_(bf["ended"])
            n += 12
            ended_host = [bool(v) for v in bf["ended"].cpu().tolist()]  # the step's only host read
            if all(ended_host):
                break
        for t2 in range(steps, T + 1):
            bf["corners_hist"][t2].copy_(bf["corners"])
            bf["dir_hist"][t2].copy_(bf["cur_dir"])
        for t2 in range(steps, T):
            bf["ended_hist"][t2].copy_(bf["ended"])
        self.launches += n + (teng.launches - l0)
        return dict(corners=bf["corners_hist"], directions=bf["dir_hist"], ended=bf["ended_hist"],
                    output=bf["output_hist"], angle=bf["angle"], altitude=bf["altitude"], dist=bf["dist"],
                    steps=steps)

    @staticmethod
    def trajectories(res):
        """Host view of a rollout result: per sample the list of (corners [4,2], direction) the reference
        appends to ``traj['path_corners']`` (agent.py:563,762-767)."""
        corners = res["corners"].cpu().numpy()
        dirs = res["directions"].cpu().numpy()
        ended = res["ended"].cpu().numpy().astype(bool)
        T, B = ended.shape
        out = []
        for i in range(B):
            path = [(corners[0, i], dirs[0, i])]
            for t in range(min(T, int(res.get("steps", T)))):
                if not ended[t, i]:
                    path.append((corners[t + 1, i], dirs[t + 1, i]))
            out.append(path)
        return out

    # ------------------------------------------------------------ API helpers
    def NSS(self, sal, fix):
        """src/xview_et/agent.py:256-270 on device tensors (torch elementwise; off the hot
        path -- the training step uses the fused ``avdn_loss`` kernel instead)."""
        nss_r = int(getattr(self.args, "nss_r", 0))
        m = torch.mean(sal.view(-1, 224 * 224), 1).view(-1, 1, 1)
        std = torch.std(sal.view(-1, 224 * 224), 1).view(-1, 1, 1)
        n_sal = (sal - m) / std
        if nss_r == 1:
            n_sal = n_sal / 2 + 1
        elif nss_r == -1:
            n_sal = n_sal / 2 - 1
        s_fix = torch.sum(fix.view(-1, 224 * 224), 1) + 0.001
        s_ns = torch.sum((n_sal * fix).view(-1, 224 * 224), 1)
        return -torch.mean(s_ns / s_fix)

    def postprocess_waypoints(self, output, edge_len, stop_threshold=0.5):
        """agent.py:637-653,738,745-752 for the whole batch in one kernel.
        ``output`` [B,4] f32, ``edge_len`` [B] f64 -> dict of device tensors."""
        B = output.shape[0]
        dev = output.device
        res = dict(angle=torch.empty(B, dtype=torch.int32, device=dev),
                   dist=torch.empty(B, dtype=torch.float64, device=dev),
                   altitude=torch.empty(B, dtype=torch.int32, device=dev),
                   stop=torch.empty(B, dtype=torch.uint8, device=dev),
                   xy=torch.empty((B, 2), dtype=torch.float32, device=dev))
        el = torch.as_tensor(edge_len, dtype=torch.float64, device=dev).contiguous()
        out_c = output.contiguous()                  # named: a temporary inside ptr() would dangle
        _lib.call("avdn_postprocess_waypoints", _lib.ptr(out_c), _lib.ptr(el), B, float(stop_threshold),
                  _lib.ptr(res["angle"]), _lib.ptr(res["dist"]), _lib.ptr(res["altitude"]), _lib.ptr(res["stop"]),
                  _lib.ptr(res["xy"]))
        return res

    def gps_to_img_coords(self, gps, ob):
        """agent.py:508-509 (twin of env.py:189-196)."""
        return (int(round((gps[1] - ob["gps_botm_left"][1]) / ob["lat_ratio"])),
                int(round((ob["gps_top_right"][0] - gps[0]) / ob["lat_ratio"])))

    def move_view_corners(self, corners, angle, distance, altitude, gps_botm_left, gps_top_right,
                          input_current_direction=None):
        """agent.py:285-384: zoom to ``altitude``, rotate by ``-angle`` about the centre, move
        forward by ``distance``; each stage is rejected if a corner leaves the map.  Host
        float64, evaluated in the reference's operation order."""
        corners = np.asarray(corners, dtype=np.float64)
        norm = np.linalg.norm

        def inside(p):
            return gps_botm_left[0] < p[0] < gps_top_right[0] and gps_botm_left[1] < p[1] < gps_top_right[1]

        def rot(theta, p):
            t = theta / 180 * PI_REF
            M = np.array([[np.cos(t), np.sin(t)], [-np.sin(t), np.cos(t)]])
            return np.matmul(M, np.array([p[0], p[1]]))

        def zoom(cs, ch):
            o = np.zeros((4, 2))
            o[0] = cs[0] + (cs[0] - cs[1]) / norm(cs[1] - cs[0]) * ch
            o[0] += (cs[0] - cs[3]) / norm(cs[3] - cs[0]) * ch
            o[1] = cs[1] + (cs[1] - cs[0]) / norm(cs[1] - cs[0]) * ch
            o[1] += (cs[1] - cs[2]) / norm(cs[2] - cs[1]) * ch
            o[2] = cs[2] + (cs[2] - cs[3]) / norm(cs[2] - cs[3]) * ch
            o[2] += (cs[2] - cs[1]) / norm(cs[2] - cs[1]) * ch
            o[3] = cs[3] + (cs[3] - cs[2]) / norm(cs[2] - cs[3]) * ch
            o[3] += (cs[3] - cs[0]) / norm(cs[3] - cs[0]) * ch
            return o

        def forward(cs, ch):
            o = np.zeros((4, 2))
            o[0] = cs[0] + (cs[0] - cs[3]) / norm(cs[3] - cs[0]) * ch
            o[1] = cs[1] + (cs[1] - cs[2]) / norm(cs[2] - cs[1]) * ch
            o[2] = cs[2] + (cs[1] - cs[2]) / norm(cs[2] - cs[1]) * ch
            o[3] = cs[3] + (cs[0] - cs[3]) / norm(cs[3] - cs[0]) * ch
            return o

        cur = round(get_direction(np.mean(corners, axis=0), (corners[0] + corners[1]) / 2)) % 360
        if input_current_direction is not None and abs(input_current_direction - cur) > 2:
            angle += input_current_direction
        edge = norm(corners[1] - corners[0]) * 11.13 * 1e4
        zoomed = zoom(corners, 0.5 * (altitude - edge) / 11.13 / 1e4)
        if not all(inside(p) for p in zoomed):
            return np.array(corners), cur
        corners = zoomed
        centre = np.mean(corners, axis=0)
        rotated = [centre + rot(-angle, corners[i] - centre) for i in range(4)]
        if not all(inside(p) for p in rotated):
            return np.array(corners), cur
        moved = forward(np.array(rotated), distance)
        if not all(inside(p) for p in moved):
            return np.array(rotated), (cur + angle) % 360
        return np.array(moved), (cur + angle) % 360

    # ------------------------------------------------- the reference's agent loop (drop-in signatures)
    def rollout(self, train_ml=None, not_in_train=False, nss_w=0, **kwargs):
        """Drop-in for ``NavCMTAgent.rollout`` (src/xview_et/agent.py:512-894) over ``self.env`` (an
        ``ANDHNavBatch`` whose ``batch`` / maps the data loader has filled): one rollout of the current batch under
        ``self.feedback``; returns the list of trajectory dicts the reference returns.

        * training (``not_in_train`` false): the rollout's loss ``ml_loss * train_ml / B`` is added to ``self.loss`` and
          its gradients to the optimiser arenas -- the reference builds an autograd graph here and calls
          ``self.loss.backward()`` in ``train``; this implementation has no graph, so the backward of a rollout runs
          inside it and ``train`` only clips and steps.  Teacher feedback: the poses come from the ground-truth
          actions; student feedback: from a no-grad greedy rollout (``student_batch``).  Language: tokenizer +
          ``CustomBERTModel``, trained in the loop.
        * ``args.on_policy_student`` (default false): a student-feedback training rollout is instead one
          ``student_rollout_step``, the reference's single pass -- the poses follow the train-mode predictions that
          are trained (trunk on per-step batch statistics, dropout on), as in agent.py:580-760.
        * ``not_in_train``: no gradients; student feedback is ``rollout_greedy``; teacher feedback additionally logs
          ``human_att_performance`` / ``nss`` per step (agent.py:683-693)."""
        env = self.env
        dev = self.device
        T = int(getattr(self.args, "max_action_len", 15))
        _, lb, gps0, geo, tidx, dirs0, gt_paths, traj = self._rollout_setup()
        has_gt = "test" not in self.env_name
        prev_r, self.renderer = self.renderer, env.renderer
        try:
            if not_in_train and self.feedback == "student":
                seq, lin = self._lang_eval_forward(lb)
                res = self.rollout_greedy(dict(corners_gps=torch.from_numpy(gps0).to(dev), directions=dirs0, geo=geo,
                                               tile_idx=tidx, lang=seq.float(), lang_cls=lin.float()), max_action_len=T)
                steps = int(res["steps"])
                tgt = None
                if has_gt:
                    tgt = tuple(a.cpu().numpy() for a in student_targets(self, res["corners"][:steps],
                                                                         res["ended"][:steps], gt_paths))
                self._log_traj(traj, res["output"][:steps].cpu().numpy(), tgt,
                               res["ended"][:steps].cpu().numpy().astype(bool), res["corners"].cpu().numpy(),
                               res["directions"].cpu().numpy(), steps)
                return traj
            if self.feedback == "student" and not not_in_train and getattr(self.args, "on_policy_student", False):
                self._on_policy_rollout(lb, gps0, dirs0, geo, tidx, gt_paths, traj, T, train_ml, nss_w, has_gt)
                return traj
            # ---- poses of the rollout ----
            if self.feedback == "teacher":
                Hh, steps = self._teacher_rollout_poses(torch.from_numpy(gps0), dirs0, geo, gt_paths, T)
                corners, ended, heads = Hh["corners"][:steps], Hh["ended"][:steps], Hh["dirs"][:steps]
                tgt = (Hh["xy"][:steps], Hh["alt"][:steps], Hh["prog"][:steps])
                c_all, d_all = Hh["corners"], Hh["dirs"]
            elif self.feedback == "student":
                # the student's own (no-grad, eval-mode) greedy rollout fixes the poses; the teacher supplies the
                # target of every visited pose (agent.py:655-661)
                with torch.no_grad():
                    seq, lin = self._lang_eval_forward(lb)
                    res = self.rollout_greedy(dict(corners_gps=torch.from_numpy(gps0).to(dev), directions=dirs0, geo=geo,
                                                   tile_idx=tidx, lang=seq.float().clone(), lang_cls=lin.float().clone()),
                                              max_action_len=T)
                steps = int(res["steps"])
                corners, ended, heads = res["corners"][:steps], res["ended"][:steps], res["directions"][:steps]
                c_all, d_all = res["corners"], res["directions"]
                tgt = student_targets(self, corners, ended, gt_paths)
            else:
                raise SystemExit("Invalid feedback option")
            ended_h = ended.cpu().numpy().astype(bool)
            lens = history_lengths(ended_h)
            rad = heads.float() / 180 * PI_REF                            # agent.py:605-606
            batch = dict(lb, **rollout_pose_batch(corners, geo, tidx, tgt),
                         directions=torch.stack([torch.sin(rad), torch.cos(rad)], -1).transpose(0, 1).contiguous(),
                         lenths=lens.tolist())
            if getattr(self.args, "no_direction", False):
                batch["directions"] = torch.zeros_like(batch["directions"])
            outs = []
            if not_in_train:
                loss = self._eval_rollout(batch, traj, outs)
            else:
                loss = self.train_rollout_step(batch, zero=False, step=False, nss_w=float(nss_w),
                                               train_ml=train_ml if train_ml is not None else 0.0, collect=outs,
                                               bn_per_step=bool(getattr(self.args, "bn_per_step", True)))
            # what the rollout was made of (inspection / tests): poses, stop flags, targets, the training batch
            self._last_rollout = dict(corners=corners, ended=ended, steps=steps, tgt_xy=tgt[0], tgt_alt=tgt[1],
                                      tgt_prog=tgt[2], batch=batch, lenths=lens)
            tgt_h = tuple(a.cpu().numpy() for a in tgt) if has_gt else None
            self._log_traj(traj, torch.stack(outs).cpu().numpy(), tgt_h, ended_h, c_all.cpu().numpy(), d_all.cpu().numpy(),
                           steps)
            self._add_rollout_loss(loss, train_ml)
        finally:
            self.renderer = prev_r
        return traj

    def _on_policy_rollout(self, lb, gps0, dirs0, geo, tidx, gt_paths, traj, T, train_ml, nss_w, has_gt):
        """The student-feedback training rollout of ``rollout`` with ``args.on_policy_student``: one
        ``student_rollout_step`` (BERT, trunk and ET in train mode; the poses follow the train-mode predictions).
        The trajectory dicts log the outputs and poses the rollout used."""
        outs = []
        batch = dict(lb, corners_gps=torch.from_numpy(gps0).to(self.device), directions=dirs0, geo=geo, tile_idx=tidx)
        loss = self.student_rollout_step(batch, gt_paths, max_action_len=T, nss_w=float(nss_w),
                                         train_ml=train_ml if train_ml is not None else 0.0, zero=False, step=False,
                                         collect=outs)
        lr = self._last_rollout
        tgt = (lr["tgt_xy"].cpu().numpy(), lr["tgt_alt"].cpu().numpy(), lr["tgt_prog"].cpu().numpy()) if has_gt else None
        self._log_traj(traj, torch.stack(outs).cpu().numpy(), tgt, lr["ended"].cpu().numpy().astype(bool),
                       lr["corners"].cpu().numpy(), lr["directions"].cpu().numpy(), lr["steps"])
        self._add_rollout_loss(loss, train_ml)

    @torch.no_grad()
    def _eval_rollout(self, batch, traj, outs):
        """``not_in_train`` with teacher feedback (validation of the human-attention head, agent.py:673-693): the ET in
        eval mode over the growing history of the given poses; per step the loss terms and, for samples with a
        fixation map, precision / recall of the clipped saliency map and the NSS value.  Returns the loss."""
        ptr = _lib.ptr
        dev = self.device
        self.vision_model.eval()
        et = self.vln_model
        et.eval()
        seq, lin = self._lang_eval_forward(batch)
        lang, lang_cls = seq.float().contiguous(), lin.float().contiguous()
        dirs = batch["directions"].contiguous().float()
        B, T = dirs.shape[:2]
        L = lang.shape[1]
        r = self.renderer
        ti = batch["tile_idx"].reshape(-1)
        minv = r.homography(batch["corners_px"].view(B * T, 4, 2))
        x = torch.empty((B * T, 224, 224, 4), dtype=torch.bfloat16, device=dev)
        att = torch.empty((B * T, 224, 224), dtype=torch.uint8, device=dev)
        r.render(None, ti, views=False, norm_nhwc=True, minv=minv, out={"norm_nhwc": x})
        r.render(None, ti, views=False, att=True, minv=minv, out={"att": att})
        att = att.view(B, T, 224, 224)
        xs = x.view(B, T, 224, 224, 4)
        fr = torch.empty((B, T, 512, 49), dtype=torch.float32, device=dev)
        for t in range(T):                                   # the reference's eval-mode trunk sees B views per call
            teng = self.vision_model.engine(B, 224, 224, dev)
            o = torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev)
            DN._trunk_forward(self.vision_model, teng, xs[:, t].contiguous(), False, out=o)
            fr[:, t] = o.view(B, 512, 49)
        lens = batch["lenths"]
        pe = et.encoder_vl.enc_pos.pe[0]
        total = torch.zeros(1, dtype=torch.float64, device=dev)
        loss_i = torch.empty(B, dtype=torch.float64, device=dev)
        d_o = torch.empty((B, 4), device=dev); d_h = torch.empty((B, 64), device=dev)
        scale = float(self.train_ml) / B
        for t in range(T):
            Tc = t + 1
            eng = et.engine(B, L, Tc, dev)
            eng.set_dropout(0.0, 0.0, 0)
            output, h_sali = eng.forward(fr[:, :Tc].contiguous().view(B * Tc, 512, 49), lang, lang_cls,
                                         dirs[:, :Tc].contiguous(), [int(lens[i][t]) for i in range(B)], pe)
            outs.append(output.detach().clone())
            att_t = att[:, t].contiguous()
            _lib.call("avdn_loss", ptr(output), ptr(h_sali), ptr(batch["gt_xy"][:, t].contiguous()),
                      ptr(batch["gt_alt"][:, t].contiguous()), ptr(batch["gt_prog"][:, t].contiguous()), ptr(att_t), None, B,
                      float(self.nss_w), int(getattr(self.args, "nss_r", 0)), scale, ptr(total), ptr(loss_i), ptr(d_o), ptr(d_h))
            if self.feedback == "teacher":
                sal = torch.empty((B, 224, 224), dtype=torch.float32, device=dev)
                _lib.call("avdn_upsample_saliency", ptr(h_sali.contiguous()), B, ptr(sal))
                gt = att_t.double() / 255
                for i in range(B):
                    if float(gt[i].sum()) > 0:
                        nss = self.NSS(sal[i].double(), gt[i])
                        p = sal[i].clip(0, 1).double()
                        tp = float((p * gt[i]).sum())
                        sp = float(p.sum())
                        traj[i].setdefault("human_att_performance", []).append([tp / sp if sp != 0 else 0.0,
                                                                                tp / float(gt[i].sum())])
                        traj[i].setdefault("nss", []).append(float(nss))
        return total

    def _reduce_and_step(self):
        if self.world > 1:
            for opt in self.optimizers:
                self._allreduce_async(opt.g, 0, opt.n)
            self._wait_comm()
        gs = 1.0 / self.world
        for opt in self.optimizers:
            self.launches += opt.step(grad_scale=gs)

    # ------------------------------------------------------------- checkpoints
    def _checkpoint_items(self):
        """agent.py:899-916: vision_model, vln_model and (when attached) lang_model; optimiser moments in the
        flat-arena format (``RolloutTrainer.save`` / ``load``)."""
        items = [("vision_model", self.vision_model, self.vision_model_optimizer, None),
                 ("vln_model", self.vln_model, self.et_optimizer, None)]
        if self.lang_model is not None:
            items.insert(0, ("lang_model", self.lang_model, self.lang_optimizer, None))
        return items
