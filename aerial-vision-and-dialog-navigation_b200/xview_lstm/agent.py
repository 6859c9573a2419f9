"""``NavCMTAgent`` of the LSTM baseline (mirror of src/xview_lstm/agent.py, hot-path subset): greedy
waypoint-rollout inference (BASELINE config 5), teacher-forced training (``train_rollout_step``,
``student_batch``, ``train_iteration``: the ET agent's batch-level training API, ``agent_common.RolloutTrainer``),
and the reference's agent loop with its signatures: ``attach_lang_model``, ``rollout(train_ml, not_in_train, nss_w)``,
``train(loader, n_epochs, feedback, nss_w_weighting)``, ``test(loader, ...)``, ``save`` / ``load``.

``rollout_greedy`` is the student-feedback loop of ``rollout`` (src/xview_lstm/agent.py:518-750)
with every per-step stage on the device and no host round trip inside the loop:

    corners (GPS) -> pixel corners (env.py:189-196) -> homography + rendered views (env.py:287-293,
    agent.py:575-582) -> Darknet trunk, eval mode (vln_model.py:216) -> ViT_LSTM step
    (vln_model.py:219-248) -> post-processing + stop test + move_view_corners
    (agent.py:607-626,700-730; xview_et/agent.py:285-384)

The language side (BERT -> ``lang_feature`` [B,L,768], ``cls_hidden`` = linear_cls [B,49],
agent.py:527-543) is an input of the path (SURVEY.md §8f N1).

Student-feedback training runs in one of two ways.  By default (``rollout``, ``student_batch``) a no-grad
``rollout_greedy`` in eval mode fixes the poses and ``train_rollout_step`` then trains on them.  With
``args.on_policy_student`` ``rollout`` calls ``student_rollout_step`` instead, the reference's single pass
(agent.py:518-774): every step renders the current views, runs its own train-mode trunk pass (per-step batch
statistics) and ``_TrainEngine.step`` with dropout on, and the simulator moves by that train-mode output; the targets,
loss and backward through time follow once the loop has ended.  Both training rollouts end in ``_finish_backward``
(backward through time, BERT backward, trunk backward, optimiser).

Training: one ``FusedAdamW`` over ``vln_model.used_parameters()`` (gradients clipped to a global norm of 40) and one
over the trunk (unclipped), built here before any rollout captures a CUDA graph of the trunk (the arenas re-home
the parameter storage).  AdamW is elementwise, so two optimisers update as one would; the clipping mirrors the ET
agent, which the in-tree record of the reference supports for ET only (DESIGN.md §8).  With ``attach_lang_model``
``CustomBERTModel`` is trained in the loop by a third, unclipped ``FusedAdamW``.

Checkpoints (``save`` / ``load``, ``agent_common.RolloutTrainer``): a ``torch.save`` dict with the entries
``vision_model`` (the trunk), ``vln_model`` (the ``ViT_LSTM`` state without the ``vision_model.*`` keys: the trunk is
written once) and, when attached, ``lang_model``; each ``{'epoch', 'state_dict', 'optimizer': {'m', 'v', 'step'}}``
with the flat AdamW arena of that model.  ``load`` also takes a ``vln_model`` entry holding a full
``ViT_LSTM.state_dict()`` (the reference's layout: the trunk is a sub-module, agent.py:140-142); its
``vision_model.*`` keys then load into the trunk.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import _lib
from ..agent_common import (RolloutTrainer, render_rollout_views, rollout_pose_batch, rollout_step_bufs,
                            rollout_trunk_backward, rollout_trunk_forward, steps_until_all_ended, student_targets)
from ..env import ViewRenderer
from ..models import dark_net as DN
from ..models.dark_net import Darknet
from ..models.vln_model import ViT_LSTM, NCH, NSP
from ..optim import FusedAdamW

STOP_THRESHOLD_STUDENT = 0.25          # src/xview_lstm/agent.py:705 (the ET agent uses 0.5)


class NavCMTAgent(RolloutTrainer):
    # stop threshold of the simulator on the progress output (agent.py:701,705): the student path's value, also used
    # for the teacher path's ground-truth progress, whose value in the reference is unverified (DESIGN.md §8)
    STOP_THRESHOLD = STOP_THRESHOLD_STUDENT

    def __init__(self, args, rank=0, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("NavCMTAgent needs a CUDA device (sm_100); there is no CPU fallback")
        _lib.lib()
        self.args, self.rank = args, rank
        self.device = torch.device(device if device is not None else "cuda")
        self.results, self.losses, self.env = {}, [], []
        self.vision_model = Darknet(args.darknet_model_file, 224)
        wf = getattr(args, "darknet_weight_file", None)
        if wf and os.path.exists(wf):                           # agent.py:130-135
            new_state = torch.load(wf, map_location="cpu")
            state = self.vision_model.state_dict()
            state.update({k: v for k, v in new_state["model"].items() if k in state})
            self.vision_model.load_state_dict(state)
        self.vln_model = ViT_LSTM(args, self.vision_model).to(self.device)      # trunk is a sub-module (agent.py:140-142)
        self.vln_model.drop_rank = rank
        lr = getattr(args, "lr", 1e-5)
        if getattr(args, "optim", "adamW") != "adamW":
            raise NotImplementedError("only optim='adamW' is implemented")
        self.policy_optimizer = FusedAdamW(self.vln_model.used_parameters(), lr=lr, max_norm=40.0)
        self.vision_model_optimizer = FusedAdamW(dict(self.vision_model.named_parameters()), lr=lr)
        self.vln_model._grad_arena = self.policy_optimizer.grads
        self.vision_model._grad_arena = self.vision_model_optimizer.grads
        self.optimizers = (self.policy_optimizer, self.vision_model_optimizer)
        self.lang_model, self.lang_optimizer = None, None     # attach_lang_model
        self.tokenizer = getattr(args, "tokenizer", None)     # BertTokenizerFast in the reference (agent.py:124)
        self.feedback = "student"
        self.env_name = ""
        self.loss = 0
        self.logs = {"IL_loss": []}
        self.loss_total = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.renderer = ViewRenderer(self.device)
        self.use_graphs = os.environ.get("AVDN_CUDA_GRAPHS", "1") != "0"     # rollouts replay the frozen trunk pass
        self.launches = 0
        self._bufs = {}

    def _get_bufs(self, B, T, kind=None):
        """Pose and simulator buffers of a rollout of B episodes and T steps; ``kind`` keeps the greedy rollout's
        (None) and the on-policy training rollout's ('on_policy') apart."""
        key = (B, T) if kind is None else (kind, B, T)
        b = self._bufs.get(key)
        if b is None:
            dev = self.device
            b = dict(x=torch.empty((B, 224, 224, 4), dtype=torch.bfloat16, device=dev),
                     frames=torch.empty((B, NCH, 7, 7), dtype=torch.float32, device=dev),
                     corners=torch.empty((B, 4, 2), dtype=torch.float64, device=dev),
                     cur_dir=torch.empty(B, dtype=torch.float64, device=dev),
                     ended=torch.empty(B, dtype=torch.uint8, device=dev),
                     px=torch.empty((B, 4, 2), dtype=torch.int32, device=dev),
                     minv=torch.empty((B, 3, 3), dtype=torch.float64, device=dev),
                     corners_hist=torch.empty((T + 1, B, 4, 2), dtype=torch.float64, device=dev),
                     dir_hist=torch.empty((T + 1, B), dtype=torch.float64, device=dev),
                     ended_hist=torch.empty((T, B), dtype=torch.uint8, device=dev),
                     output_hist=torch.empty((T, B, 4), dtype=torch.float32, device=dev),
                     angle=torch.empty((T, B), dtype=torch.int32, device=dev),
                     altitude=torch.empty((T, B), dtype=torch.int32, device=dev),
                     dist=torch.empty((T, B), dtype=torch.float64, device=dev))
            self._bufs[key] = b
        return b

    @torch.no_grad()
    def rollout_greedy(self, batch, max_action_len=None, stop_threshold=STOP_THRESHOLD_STUDENT):
        """Greedy (student) rollout of ``B`` episodes for ``max_action_len`` steps.

        ``batch`` (device tensors): ``corners_gps`` f64 [B,4,2] (lat,lng; FL,FR,BR,BL = gt_path_corners[0]),
        ``directions`` [B] (starting_angle, degrees), ``geo`` f64 [B,5] = (bl_lat, bl_lng, tr_lat, tr_lng,
        lat_ratio), ``tile_idx`` i32 [B] or None, ``lang_feature`` f32 [B,L,768], ``cls_hidden`` f32 [B,49].

        Returns device tensors: ``corners`` [T+1,B,4,2] (pose before every step and after the last),
        ``directions`` [T+1,B], ``ended`` [T,B] (sticky stop flags after each step), ``output`` [T,B,4]
        (raw network outputs), ``angle`` / ``altitude`` [T,B] (discretised action), ``dist`` [T,B].
        A trajectory is the poses of the steps at which the sample had not ended yet
        (``traj['path_corners']``, agent.py:735-739)."""
        self.vln_model.eval()
        T = int(max_action_len if max_action_len is not None else getattr(self.args, "max_action_len", 20))
        lang, cls = batch["lang_feature"].contiguous(), batch["cls_hidden"].contiguous()
        B, L = lang.shape[0], lang.shape[1]
        ptr, call = _lib.ptr, _lib.call
        bf = self._get_bufs(B, T)
        geo = batch["geo"].contiguous()
        bounds = geo[:, :4].contiguous()
        ti = batch.get("tile_idx")
        bf["corners"].copy_(batch["corners_gps"])
        bf["cur_dir"].copy_(batch["directions"])
        bf["ended"].zero_()
        vm, r = self.vision_model, self.renderer
        eng = vm.engine(B, 224, 224, self.device)
        l0, v0 = eng.launches, self.vln_model.launches
        self.vln_model.reset_state(B, L, self.device)
        n = 0
        for t in range(T):
            bf["corners_hist"][t].copy_(bf["corners"])
            bf["dir_hist"][t].copy_(bf["cur_dir"])
            # ---- observation: env._get_obs(corners=current_view_corners) (agent.py:742) ----
            call("avdn_gps_to_pixels", ptr(bf["corners"]), ptr(geo), B, ptr(bf["px"]))
            call("avdn_homography_from_corners", ptr(bf["px"]), B, ptr(bf["minv"]))
            r.render(None, ti, views=False, norm_nhwc=True, minv=bf["minv"], out={"norm_nhwc": bf["x"]})
            # ---- policy (agent.py:592-602) ----
            if t == 0 or not self.use_graphs:
                DN._trunk_forward(vm, eng, bf["x"], False, out=bf["frames"], frozen=(t > 0))
            else:
                DN._trunk_forward_graphed(vm, eng, bf["x"], bf["frames"])
            output, _ = self.vln_model.step(bf["frames"].view(B, NCH, NSP), bf["cur_dir"], cls, lang,
                                            want_saliency=False)
            bf["output_hist"][t].copy_(output)
            # ---- simulator (agent.py:607-626,700-730) ----
            call("avdn_waypoint_step", ptr(output), ptr(bf["corners"]), ptr(bounds), ptr(bf["cur_dir"]),
                 ptr(bf["ended"]), B, float(stop_threshold), int(t == T - 1), ptr(bf["angle"][t]),
                 ptr(bf["dist"][t]), ptr(bf["altitude"][t]))
            bf["ended_hist"][t].copy_(bf["ended"])
            n += 4
        bf["corners_hist"][T].copy_(bf["corners"])
        bf["dir_hist"][T].copy_(bf["cur_dir"])
        self.launches += n + (eng.launches - l0) + (self.vln_model.launches - v0)
        return dict(corners=bf["corners_hist"], directions=bf["dir_hist"], ended=bf["ended_hist"],
                    output=bf["output_hist"], angle=bf["angle"], altitude=bf["altitude"], dist=bf["dist"])

    # ------------------------------------------------------------------ training
    def _rollout_bufs(self, B, T):
        """Views, attention maps and trunk features of the B*T poses of a rollout."""
        key = ("rollout_train", B, T)
        tb = self._bufs.get(key)
        if tb is None:
            dev, BT = self.device, B * T
            tb = dict(x=torch.empty((BT, 224, 224, 4), dtype=torch.bfloat16, device=dev),
                      att=torch.empty((BT, 224, 224), dtype=torch.uint8, device=dev),
                      frames=torch.empty((BT, NCH, 7, 7), dtype=torch.float32, device=dev))
            self._bufs[key] = tb
        return tb

    def _train_rollout_step(self, batch, sync_loss=False, zero=True, step=True, collect=None, bn_per_step=None):
        """One teacher-forced training rollout (src/xview_lstm/agent.py:546-550,592-602,636; ``train_rollout_step``):
        the B*T views of the given poses are rendered and pushed through the train-mode trunk (one pass over all of
        them, or one per step with ``bn_per_step`` / ``args.bn_per_step``, ``agent_common.rollout_trunk_forward``),
        then ``ViT_LSTM``'s T recurrent steps run with the loss of every step (``avdn_loss``, jitter 0, scale
        ``train_ml / B``), the backward through time, the trunk backward and (``step``) the optimiser step.
        There are no ``lenths``: a sample that has stopped keeps stepping on its final pose and contributes loss,
        as in the reference loop.

        ``batch``: ``corners_px`` i32 [B,T,4,2] (or ``images`` bf16 [B*T,224,224,4]), ``tile_idx`` i32 [B,T] | None,
        ``lang_feature`` [B,L,768], ``cls_hidden`` [B,49], ``directions`` [B,T] (headings in DEGREES),
        ``gt_xy`` [B,T,2], ``gt_alt`` / ``gt_prog`` [B,T], optional ``att`` u8 [B,T,224,224] (default: rendered
        from the poses when ``nss_w != 0``).  ``zero`` / ``step`` / ``collect`` as in the ET agent.
        With an attached language model the batch may carry ``input_ids`` / ``attention_mask`` (and optionally
        ``cls_input_ids`` / ``cls_attention_mask``) instead of ``lang_feature`` / ``cls_hidden``: BERT runs once per
        rollout in train mode, its sequence output is ``lang_feature`` and its ``linear_cls`` is ``cls_hidden``
        (agent.py:527-543), and the gradients of both, summed over the T steps, go through one BERT backward (two
        with the cls pass) into the language arena."""
        deg = batch["directions"].contiguous().float()
        B, T = deg.shape
        BT = B * T
        dev = self.device
        n = 0
        if zero:
            for opt in self.optimizers:
                opt.zero_grad()
            n += 2
        lengs = None
        if "input_ids" in batch:
            seq, lin, *lengs = self._lang_train_forward(batch)
            batch = dict(batch, lang_feature=seq, cls_hidden=lin)
        lang, cls = batch["lang_feature"].contiguous().float(), batch["cls_hidden"].contiguous().float()
        L = lang.shape[1]
        tb = self._rollout_bufs(B, T)
        x, att, k = render_rollout_views(self, batch, BT, tb["x"], tb["att"])
        n += k
        vln, vm = self.vln_model, self.vision_model
        vln.train(not getattr(self.args, "no_dropout", False))
        vm.train()
        teng, tengs, l0, k = rollout_trunk_forward(self, x, B, T, tb["frames"], bn_per_step)
        n += k
        eng = vln.train_engine(B, L, T, dev)
        e0 = eng.launches
        eng.forward(tb["frames"].view(BT, NCH, NSP), deg, cls, lang, *vln.dropout_config())
        tr = lambda a: a.float().transpose(0, 1).contiguous()          # [B,T,...] -> step-major [T,B,...]
        att_t = None if att is None else att.view(B, T, 224, 224).transpose(0, 1).contiguous()
        self.loss_total.zero_()
        eng.loss(tr(batch["gt_xy"]), tr(batch["gt_alt"]), tr(batch["gt_prog"]), att_t, self.nss_w,
                 int(getattr(self.args, "nss_r", 0)), float(self.train_ml) / B, self.loss_total)
        n += 5
        if collect is not None:
            collect.extend(eng.output[t].clone() for t in range(T))
        n += self._finish_backward(eng, lengs, teng, tengs, l0, T, step)
        self._ctx = (teng, tengs, eng, tb)
        self.launches += n + (eng.launches - e0)
        self._log_loss()
        return float(self.loss_total.item()) if sync_loss else self.loss_total

    def _finish_backward(self, eng, lengs, teng, tengs, l0, steps, step):
        """What follows the loss of both training rollouts: the backward through time over the first ``steps`` steps
        (with ``lengs``, ``_lang_train_forward``'s engines, it also sums the ``lang_feature`` / ``cls_hidden``
        gradients for BERT's backward), ``rollout_trunk_backward`` and, with ``step``, the optimiser step.  Returns
        the launches outside the policy engine."""
        B, L, T = eng.B, eng.L, eng.T
        if lengs is None:
            eng.backward(n_steps=steps)
        else:
            d_lang = torch.zeros((B, L, 768), dtype=torch.float32, device=self.device)
            d_cls = torch.zeros((B, 49), dtype=torch.float32, device=self.device)
            eng.backward(d_lang, d_cls, n_steps=steps)
            self._lang_train_backward(*lengs, d_lang, d_cls)
        n = rollout_trunk_backward(self, teng, tengs, l0, eng.d_frames, B, T, steps=steps)
        if step:
            for opt in self.optimizers:
                n += opt.step()
        return n

    @torch.no_grad()
    def student_batch(self, batch, gt_path_corners, max_action_len=None):
        """The student-feedback half of a training iteration: a no-grad greedy rollout (stop threshold 0.25) fixes
        the poses, ``teacher_action`` supplies the target of every step (one launch), and the result is a
        ``train_rollout_step`` batch.  ``batch`` as for ``rollout_greedy``; ``gt_path_corners``: per sample the
        ``[n_i,4,2]`` ground-truth view corners."""
        res = self.rollout_greedy(batch, max_action_len=max_action_len)
        T = res["ended"].shape[0]
        corners = res["corners"][:T]
        out = rollout_pose_batch(corners, batch["geo"], batch.get("tile_idx"),
                                 student_targets(self, corners, res["ended"], gt_path_corners))
        out.update(lang_feature=batch["lang_feature"], cls_hidden=batch["cls_hidden"],
                   directions=res["directions"][:T].float().t().contiguous())
        return out

    def student_rollout_step(self, batch, gt_path_corners, max_action_len=None, nss_w=None, train_ml=None, zero=True,
                             step=True, sync_loss=False, collect=None, bn_per_step=None):
        """One on-policy student-feedback training rollout, as the reference runs it (src/xview_lstm/agent.py:518-774):
        every step runs the policy in train mode -- the trunk on the step's own batch statistics, the four Dropout(0.2)
        sites active -- and the simulator moves by that same train-mode prediction (stop threshold 0.25).  The loop
        stops after the step at which every sample has ended (one host read of the B stop flags per step).  Then one
        ``teacher_action`` launch gives the target of every visited pose, and the loss and ``_finish_backward`` (the
        backward through time, the BERT backward, the trunk backward of the executed per-step passes and (``step``)
        the optimiser step) run as in ``train_rollout_step``.

        ``batch`` as for ``rollout_greedy``; with an attached language model it may carry ``input_ids`` /
        ``attention_mask`` (and ``cls_*``) instead of ``lang_feature`` / ``cls_hidden``: BERT then runs once in train
        mode, and its outputs both steer the rollout and receive the gradients.  ``gt_path_corners``: per sample the
        ``[n_i,4,2]`` ground-truth view corners.  The per-step trunk passes are required (``bn_per_step`` false
        raises ``ValueError``): the views of step t+1 depend on step t's features.  What the rollout visited is kept
        in ``self._last_rollout``."""
        if bn_per_step is None:
            bn_per_step = bool(getattr(self.args, "bn_per_step", True))
        if not bn_per_step:
            raise ValueError("an on-policy student rollout needs one trunk pass per step (bn_per_step): the views of "
                             "step t+1 depend on the features of step t")
        with self._weights(nss_w, train_ml):
            return self._student_rollout_step(batch, gt_path_corners, max_action_len, zero, step, sync_loss, collect)

    def _student_rollout_step(self, batch, gt_path_corners, max_action_len, zero, step, sync_loss, collect):
        T = int(max_action_len if max_action_len is not None else getattr(self.args, "max_action_len", 20))
        ptr, call = _lib.ptr, _lib.call
        dev = self.device
        n = 0
        if zero:
            for opt in self.optimizers:
                opt.zero_grad()
            n += 2
        lengs = None
        if "input_ids" in batch:
            seq, lin, *lengs = self._lang_train_forward(batch)
            batch = dict(batch, lang_feature=seq, cls_hidden=lin)
        lang, cls = batch["lang_feature"].contiguous().float(), batch["cls_hidden"].contiguous().float()
        B, L = lang.shape[0], lang.shape[1]
        vln, vm, r = self.vln_model, self.vision_model, self.renderer
        vln.train(not getattr(self.args, "no_dropout", False))
        vm.train()
        eng = vln.train_engine(B, L, T, dev)
        e0 = eng.launches
        eng.begin(cls, lang, *vln.dropout_config())
        bf = self._get_bufs(B, T, "on_policy")
        sb = rollout_step_bufs(self, B, T)
        geo = batch["geo"].contiguous()
        bounds = geo[:, :4].contiguous()
        ti = batch.get("tile_idx")
        bf["corners"].copy_(batch["corners_gps"])
        bf["cur_dir"].copy_(batch["directions"])
        bf["ended"].zero_()
        ended_h = torch.empty(B, dtype=torch.uint8, pin_memory=True)
        tengs, l0 = [], 0
        steps = T
        for t in range(T):
            bf["corners_hist"][t].copy_(bf["corners"])
            bf["dir_hist"][t].copy_(bf["cur_dir"])
            # ---- observation of the current pose (agent.py:742) ----
            call("avdn_gps_to_pixels", ptr(bf["corners"]), ptr(geo), B, ptr(bf["px"]))
            call("avdn_homography_from_corners", ptr(bf["px"]), B, ptr(bf["minv"]))
            r.render(None, ti, views=False, norm_nhwc=True, minv=bf["minv"], out={"norm_nhwc": sb["x"][t]})
            # ---- train-mode policy step (agent.py:592-602): its own trunk pass, kept for the backward ----
            teng = vm.engine(B, 224, 224, dev, slot=1 + t)
            l0 += teng.launches
            tengs.append(teng)
            DN._trunk_forward(vm, teng, sb["x"][t], True, out=sb["f"])
            output = eng.step(t, sb["f"].view(B, NCH, NSP), bf["cur_dir"])
            # ---- the simulator moves by the train-mode prediction (agent.py:607-626,700-730) ----
            call("avdn_waypoint_step", ptr(output), ptr(bf["corners"]), ptr(bounds), ptr(bf["cur_dir"]),
                 ptr(bf["ended"]), B, float(STOP_THRESHOLD_STUDENT), int(t == T - 1), ptr(bf["angle"][t]),
                 ptr(bf["dist"][t]), ptr(bf["altitude"][t]))
            bf["ended_hist"][t].copy_(bf["ended"])
            n += 9
            if t < T - 1:                                # agent.py:773-774: stop once every sample has ended
                ended_h.copy_(bf["ended"])
                if bool(ended_h.numpy().all()):
                    steps = t + 1
                    break
        bf["corners_hist"][steps].copy_(bf["corners"])
        bf["dir_hist"][steps].copy_(bf["cur_dir"])
        eng.finish()
        # ---- the teacher's target at every visited pose, one launch (agent.py:655-661) ----
        corners = bf["corners_hist"][:steps]
        tgt = student_targets(self, corners, bf["ended_hist"][:steps], gt_path_corners)
        poses = rollout_pose_batch(corners, geo, ti, tgt)
        att = None
        if self.nss_w != 0:
            key = ("on_policy_att", B, T)
            if key not in self._bufs:
                self._bufs[key] = torch.empty((T * B, 224, 224), dtype=torch.uint8, device=dev)
            att = self._bufs[key][:steps * B]
            minv = r.homography(poses["corners_px"].transpose(0, 1).reshape(steps * B, 4, 2))
            r.render(None, None if ti is None else ti.repeat(steps), views=False, att=True, minv=minv,
                     out={"att": att})
            att = att.view(steps, B, 224, 224)
            n += 2
        self.loss_total.zero_()
        eng.loss(*tgt, att, self.nss_w, int(getattr(self.args, "nss_r", 0)), float(self.train_ml) / B, self.loss_total,
                 n_steps=steps)
        n += 6
        if collect is not None:
            collect.extend(eng.output[t].clone() for t in range(steps))
        n += self._finish_backward(eng, lengs, tengs[0], tengs, l0, steps, step)
        self._ctx = (tengs[0], tengs, eng, sb)
        # what the rollout visited (inspection / tests): poses before every step and after the last, stop flags,
        # train-mode outputs, targets, and the teacher-forced batch of the same poses
        self._last_rollout = dict(
            corners=bf["corners_hist"][:steps + 1].clone(), directions=bf["dir_hist"][:steps + 1].clone(),
            ended=bf["ended_hist"][:steps].clone(), output=eng.output[:steps].clone(), steps=steps,
            tgt_xy=tgt[0], tgt_alt=tgt[1], tgt_prog=tgt[2],
            batch=dict(batch, directions=bf["dir_hist"][:steps].float().t().contiguous(), **poses))
        self.launches += n + (eng.launches - e0)
        self._log_loss()
        return float(self.loss_total.item()) if sync_loss else self.loss_total

    @staticmethod
    def trajectories(res):
        """Host view of a rollout result: per sample the list of (corners [4,2], direction) the
        reference appends to ``traj['path_corners']`` (agent.py:556-558,735-739)."""
        corners = res["corners"].cpu().numpy()
        dirs = res["directions"].cpu().numpy()
        ended = res["ended"].cpu().numpy().astype(bool)
        T, B = ended.shape
        out = []
        for i in range(B):
            path = [(corners[0, i], dirs[0, i])]
            for t in range(T):
                if not ended[t, i]:
                    path.append((corners[t + 1, i], dirs[t + 1, i]))
            out.append(path)
        return out

    # ------------------------------------------------- the reference's agent loop (drop-in signatures)
    def rollout(self, train_ml=None, not_in_train=False, nss_w=0, **kwargs):
        """Drop-in for ``NavCMTAgent.rollout`` (src/xview_lstm/agent.py:518-894) over ``self.env`` (an
        ``ANDHNavBatch`` whose ``batch`` / maps the data loader has filled): one rollout of the current batch under
        ``self.feedback``; returns the list of trajectory dicts the reference returns.

        * Poses: teacher feedback from the ground-truth actions (``_teacher_rollout_poses``), student feedback from a
          no-grad greedy rollout on BERT's eval-mode features, with the ``teacher_action`` target of every pose.  The
          loop stops after the step at which every sample has ended (agent.py:773-774).
        * ``args.on_policy_student`` (default false): a student-feedback training rollout is instead one
          ``student_rollout_step``, the reference's single pass -- the poses follow the train-mode predictions that
          are trained (trunk on per-step batch statistics, dropout on), as in agent.py:518-774.
        * Training (``not_in_train`` false): ``train_rollout_step`` over the poses with BERT in train mode -- the loss
          ``ml_loss * train_ml / B`` is added to ``self.loss`` and the gradients to the arenas (the reference's
          ``self.loss.backward()`` in ``train``; ``train`` then only clips and steps).  The LSTM has no ``lenths``: a
          sample that has stopped keeps stepping on its final pose, as in the reference.
        * ``not_in_train``: no gradients; student feedback logs the greedy rollout; teacher feedback also logs
          ``human_att_performance`` / ``nss`` per step (``_eval_rollout``)."""
        env = self.env
        dev = self.device
        T = int(getattr(self.args, "max_action_len", 20))
        _, lb, gps0, geo, tidx, dirs0, gt_paths, traj = self._rollout_setup()
        has_gt = "test" not in self.env_name
        prev_r, self.renderer = self.renderer, env.renderer
        try:
            if self.feedback == "student" and not not_in_train and getattr(self.args, "on_policy_student", False):
                self._on_policy_rollout(lb, gps0, dirs0, geo, tidx, gt_paths, traj, T, train_ml, nss_w, has_gt)
                return traj
            if self.feedback == "teacher":
                H, steps = self._teacher_rollout_poses(torch.from_numpy(gps0), dirs0, geo, gt_paths, T)
                corners, ended, heads = H["corners"][:steps], H["ended"][:steps], H["dirs"][:steps]
                tgt = (H["xy"][:steps], H["alt"][:steps], H["prog"][:steps])
                c_all, d_all = H["corners"], H["dirs"]
            elif self.feedback == "student":
                seq, lin = self._lang_eval_forward(lb)
                res = self.rollout_greedy(dict(corners_gps=torch.from_numpy(gps0).to(dev), directions=dirs0, geo=geo,
                                               tile_idx=tidx, lang_feature=seq.float().clone(),
                                               cls_hidden=lin.float().clone()), max_action_len=T)
                steps = steps_until_all_ended(res["ended"])
                corners, ended, heads = res["corners"][:steps], res["ended"][:steps], res["directions"][:steps]
                c_all, d_all = res["corners"], res["directions"]
                tgt = None
                if has_gt or not not_in_train:
                    tgt = student_targets(self, corners, ended, gt_paths)
            else:
                raise SystemExit("Invalid feedback option")
            ended_h = ended.cpu().numpy().astype(bool)
            tgt_h = tuple(a.cpu().numpy() for a in tgt) if has_gt else None
            if not_in_train and self.feedback == "student":
                self._log_traj(traj, res["output"][:steps].cpu().numpy(), tgt_h, ended_h, c_all.cpu().numpy(),
                               d_all.cpu().numpy(), steps)
                return traj
            batch = dict(lb, **rollout_pose_batch(corners, geo, tidx, tgt), directions=heads.float().t().contiguous())
            outs = []
            if not_in_train:
                loss = self._eval_rollout(batch, traj, outs)
            else:
                loss = self.train_rollout_step(batch, zero=False, step=False, nss_w=float(nss_w),
                                               train_ml=train_ml if train_ml is not None else 0.0, collect=outs,
                                               bn_per_step=bool(getattr(self.args, "bn_per_step", True)))
            # what the rollout was made of (inspection / tests): poses, stop flags, targets, the training batch
            self._last_rollout = dict(corners=corners, ended=ended, steps=steps, tgt_xy=tgt[0], tgt_alt=tgt[1],
                                      tgt_prog=tgt[2], batch=batch)
            self._log_traj(traj, torch.stack(outs).cpu().numpy(), tgt_h, ended_h, c_all.cpu().numpy(),
                           d_all.cpu().numpy(), steps)
            self._add_rollout_loss(loss, train_ml)
        finally:
            self.renderer = prev_r
        return traj

    def _on_policy_rollout(self, lb, gps0, dirs0, geo, tidx, gt_paths, traj, T, train_ml, nss_w, has_gt):
        """The student-feedback training rollout of ``rollout`` with ``args.on_policy_student``: one
        ``student_rollout_step`` (BERT, trunk and policy in train mode; the poses follow the train-mode predictions).
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
        """``not_in_train`` with teacher feedback (validation of the human-attention head, agent.py:673-693): trunk
        and policy in eval mode over the given poses (the T policy steps in one ``train_engine`` forward with p = 0),
        the loss of every step, and for every step and every sample with a non-empty fixation map precision / recall
        of the clipped saliency map and its NSS -- all T*B rows scored by one ``avdn_saliency_metrics`` launch and
        read back in one copy.  Appends the per-step outputs to ``outs``; returns the loss."""
        ptr = _lib.ptr
        dev = self.device
        vm, vln = self.vision_model, self.vln_model
        vm.eval()
        vln.eval()
        seq, lin = self._lang_eval_forward(batch)
        lang, cls = seq.float().contiguous(), lin.float().contiguous()
        deg = batch["directions"].contiguous().float()
        B, T = deg.shape
        BT, L = B * T, lang.shape[1]
        tb = self._rollout_bufs(B, T)
        r = self.renderer
        ti = batch["tile_idx"].reshape(-1)
        minv = r.homography(batch["corners_px"].view(BT, 4, 2))
        r.render(None, ti, views=False, norm_nhwc=True, minv=minv, out={"norm_nhwc": tb["x"]})
        r.render(None, ti, views=False, att=True, minv=minv, out={"att": tb["att"]})
        teng = vm.engine(BT, 224, 224, dev)
        DN._trunk_forward(vm, teng, tb["x"], False, out=tb["frames"])
        eng = vln.train_engine(B, L, T, dev)
        eng.forward(tb["frames"].view(BT, NCH, NSP), deg, cls, lang, 0.0, 0)
        tr = lambda a: a.float().transpose(0, 1).contiguous()          # [B,T,...] -> step-major [T,B,...]
        att_t = tb["att"].view(B, T, 224, 224).transpose(0, 1).contiguous()
        nss_r = int(getattr(self.args, "nss_r", 0))
        total = torch.zeros(1, dtype=torch.float64, device=dev)
        eng.loss(tr(batch["gt_xy"]), tr(batch["gt_alt"]), tr(batch["gt_prog"]), att_t, self.nss_w, nss_r,
                 float(self.train_ml) / B, total)
        outs.extend(eng.output[t].clone() for t in range(T))
        metrics = torch.empty((T, B, 4), dtype=torch.float64, device=dev)
        _lib.call("avdn_saliency_metrics", ptr(eng.h_sali), ptr(att_t), BT, nss_r, ptr(metrics))
        self.launches += 5
        mh = metrics.cpu().numpy()
        for t in range(T):
            for i in range(B):
                if mh[t, i, 3] > 0:                          # the sample's fixation map is not empty
                    traj[i].setdefault("human_att_performance", []).append([float(mh[t, i, 0]), float(mh[t, i, 1])])
                    traj[i].setdefault("nss", []).append(float(mh[t, i, 2]))
        self._ctx_eval = (eng, att_t)
        return total

    # ------------------------------------------------------------- checkpoints
    def _checkpoint_items(self):
        """The trunk, the policy (its ``vision_model.*`` keys are the trunk's: written once, under ``vision_model``)
        and, when attached, the language model -- see the module docstring."""
        items = [("vision_model", self.vision_model, self.vision_model_optimizer, None),
                 ("vln_model", self.vln_model, self.policy_optimizer, ("vision_model.",))]
        if self.lang_model is not None:
            items.insert(0, ("lang_model", self.lang_model, self.lang_optimizer, None))
        return items
