"""``NavCMTAgent`` of the LSTM baseline (mirror of src/xview_lstm/agent.py, hot-path subset): greedy
waypoint-rollout inference (BASELINE config 5) and teacher-forced training (``train_rollout_step``,
``student_batch``, ``train_iteration``: the ET agent's batch-level training API, ``agent_common.RolloutTrainer``).

``rollout_greedy`` is the student-feedback loop of ``rollout`` (src/xview_lstm/agent.py:518-750)
with every per-step stage on the device and no host round trip inside the loop:

    corners (GPS) -> pixel corners (env.py:189-196) -> homography + rendered views (env.py:287-293,
    agent.py:575-582) -> Darknet trunk, eval mode (vln_model.py:216) -> ViT_LSTM step
    (vln_model.py:219-248) -> post-processing + stop test + move_view_corners
    (agent.py:607-626,700-730; xview_et/agent.py:285-384)

The language side (BERT -> ``lang_feature`` [B,L,768], ``cls_hidden`` = linear_cls [B,49],
agent.py:527-543) is an input of the path (SURVEY.md §8f N1).

Training: one ``FusedAdamW`` over ``vln_model.used_parameters()`` (gradients clipped to a global norm of 40) and one
over the trunk (unclipped), built here before any rollout captures a CUDA graph of the trunk (the arenas re-home
the parameter storage).  AdamW is elementwise, so two optimisers update as one would; the clipping mirrors the ET
agent, which the in-tree record of the reference supports for ET only (DESIGN.md §8).
"""
from __future__ import annotations

import os

import torch

from .. import _lib
from ..agent_common import (RolloutTrainer, render_rollout_views, rollout_trunk_backward, rollout_trunk_forward,
                            student_rollout_targets)
from ..env import ViewRenderer
from ..models import dark_net as DN
from ..models.dark_net import Darknet
from ..models.vln_model import ViT_LSTM, NCH, NSP
from ..optim import FusedAdamW

STOP_THRESHOLD_STUDENT = 0.25          # src/xview_lstm/agent.py:705 (the ET agent uses 0.5)


class NavCMTAgent(RolloutTrainer):
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
        self.feedback = "student"
        self.logs = {"IL_loss": []}
        self.loss_total = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.renderer = ViewRenderer(self.device)
        self.use_graphs = os.environ.get("AVDN_CUDA_GRAPHS", "1") != "0"     # rollouts replay the frozen trunk pass
        self.launches = 0
        self._bufs = {}

    def _get_bufs(self, B, T):
        b = self._bufs.get((B, T))
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
            self._bufs[(B, T)] = b
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
        from the poses when ``nss_w != 0``).  ``zero`` / ``step`` / ``collect`` as in the ET agent."""
        deg = batch["directions"].contiguous().float()
        B, T = deg.shape
        BT = B * T
        lang, cls = batch["lang_feature"].contiguous().float(), batch["cls_hidden"].contiguous().float()
        L = lang.shape[1]
        dev = self.device
        n = 0
        if zero:
            for opt in self.optimizers:
                opt.zero_grad()
            n += 2
        key = ("rollout_train", B, T)
        tb = self._bufs.get(key)
        if tb is None:
            tb = dict(x=torch.empty((BT, 224, 224, 4), dtype=torch.bfloat16, device=dev),
                      att=torch.empty((BT, 224, 224), dtype=torch.uint8, device=dev),
                      frames=torch.empty((BT, NCH, 7, 7), dtype=torch.float32, device=dev))
            self._bufs[key] = tb
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
        eng.backward()
        trunk_launches = rollout_trunk_backward(self, teng, tengs, l0, eng.d_frames, B, T)
        self._ctx = (teng, tengs, eng, tb)
        if step:
            for opt in self.optimizers:
                n += opt.step()
        self.launches += n + trunk_launches + (eng.launches - e0)
        self._log_loss()
        return float(self.loss_total.item()) if sync_loss else self.loss_total

    @torch.no_grad()
    def student_batch(self, batch, gt_path_corners, max_action_len=None):
        """The student-feedback half of a training iteration: a no-grad greedy rollout (stop threshold 0.25) fixes
        the poses, ``teacher_action`` supplies the target of every step (one launch), and the result is a
        ``train_rollout_step`` batch.  ``batch`` as for ``rollout_greedy``; ``gt_path_corners``: per sample the
        ``[n_i,4,2]`` ground-truth view corners."""
        res = self.rollout_greedy(batch, max_action_len=max_action_len)
        out, _, T = student_rollout_targets(self, batch, res, gt_path_corners)
        out.update(lang_feature=batch["lang_feature"], cls_hidden=batch["cls_hidden"],
                   directions=res["directions"][:T].float().t().contiguous())
        return out

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
