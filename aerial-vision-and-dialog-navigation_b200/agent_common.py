"""What the two agents (``xview_et.agent`` and ``xview_lstm.agent``, twins in the reference) share for training:
the batch-level training API (``RolloutTrainer``: loss weights, ``train_rollout_step``, ``train_iteration``, the
loss log, ``teacher_action``), the model-independent parts of the reference's agent loop (tokenizer, BERT passes,
teacher poses, trajectory dicts, ``train``, ``test``, ``save`` / ``load``), the views and trunk passes of a
teacher-forced training rollout, the targets of the poses a student-feedback rollout visited (``student_targets``)
and the pose batch of a rollout (``rollout_pose_batch``).  Each agent supplies ``_train_rollout_step`` (its policy's
forward, loss and backward), ``rollout`` and ``_checkpoint_items``."""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib
from .models import dark_net as DN
from .optim import FusedAdamW


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
            gt_path_corners = pack_gt_paths(gt_path_corners, dev)
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

    # ------------------------------------------------- the reference's agent loop (drop-in signatures)
    def attach_lang_model(self, lang_model=None, lr=None):
        """Put ``CustomBERTModel`` (default: BERT-base) into the training loop with a third ``FusedAdamW`` (lr
        ``args.lr`` unless given; not clipped, agent.py:155,247-249).  Returns the model."""
        from .models.bert import CustomBERTModel
        self.lang_model = (lang_model if lang_model is not None else CustomBERTModel()).to(self.device)
        self.lang_optimizer = FusedAdamW(self.lang_model.used_parameters(),
                                         lr=lr if lr is not None else getattr(self.args, "lr", 1e-5))
        self.lang_model._grad_arena = self.lang_optimizer.grads
        self.lang_model._engines.clear()
        self.lang_model.drop_rank = self.rank
        self.optimizers = self.optimizers[:2] + (self.lang_optimizer,)
        return self.lang_model

    def _language_batch(self, items):
        """agent.py:519-538: the dialog of every episode through the tokenizer -- ``instructions`` for the
        policy's language rows, ``pre_dialogs + instructions`` for ``linear_cls`` unless ``args.train_val_on_full``.
        Needs ``self.tokenizer`` (the reference's ``BertTokenizerFast``: any callable
        ``tok(list[str], padding=True, return_tensors='pt')`` -> ``input_ids`` / ``attention_mask``) and an attached
        language model."""
        if self.lang_model is None or self.tokenizer is None:
            raise RuntimeError("rollout() tokenises the dialogs and runs CustomBERTModel (agent.py:124-126,519-538): "
                               "set agent.tokenizer and call attach_lang_model() first")
        vis_only = bool(getattr(self.args, "vision_only", False))
        texts = ["" if vis_only else it["instructions"] for it in items]
        enc = self.tokenizer(texts, padding=True, return_tensors="pt")
        out = {"input_ids": enc["input_ids"].to(self.device), "attention_mask": enc["attention_mask"].to(self.device)}
        lang_inputs = texts
        if not bool(getattr(self.args, "train_val_on_full", False)):
            lang_inputs = [it["pre_dialogs"] + it["instructions"] for it in items]
            enc2 = self.tokenizer(lang_inputs, padding=True, return_tensors="pt")
            out["cls_input_ids"] = enc2["input_ids"].to(self.device)
            out["cls_attention_mask"] = enc2["attention_mask"].to(self.device)
        return out, lang_inputs

    @torch.no_grad()
    def _lang_eval_forward(self, lb):
        """BERT in eval mode over a ``_language_batch``: (sequence output, ``linear_cls``) -- the latter from the
        second pass over ``pre_dialogs + instructions`` when the batch has one (agent.py:519-538)."""
        lm, dev = self.lang_model, self.device
        if lm is None:
            raise RuntimeError("batch carries input_ids but no language model is attached (attach_lang_model)")
        lm.eval()
        leng = lm.engine(lb["input_ids"].shape[0], lb["input_ids"].shape[1], dev)
        leng.set_dropout(*lm.dropout_config())
        seq, lin, _ = leng.forward(lb["input_ids"].long(), lb["attention_mask"])
        if "cls_input_ids" in lb:
            leng2 = lm.engine(lb["cls_input_ids"].shape[0], lb["cls_input_ids"].shape[1], dev, slot=1)
            leng2.set_dropout(*lm.dropout_config())
            _, lin, _ = leng2.forward(lb["cls_input_ids"].long(), lb["cls_attention_mask"])
        return seq, lin

    def _lang_train_forward(self, batch):
        """BERT in train mode once per rollout over ``input_ids`` / ``attention_mask`` (and the ``cls_*`` pass when
        given).  Returns (sequence output, ``linear_cls``, engine, cls engine or None); ``_lang_train_backward``
        then takes the gradients collected over all steps."""
        if self.lang_model is None:
            raise RuntimeError("batch carries input_ids but no language model is attached (attach_lang_model)")
        lm = self.lang_model
        lm.train(not getattr(self.args, "no_dropout", False))
        ids, am = batch["input_ids"], batch["attention_mask"]
        leng = lm.engine(ids.shape[0], ids.shape[1], self.device)
        leng.set_dropout(*lm.dropout_config())
        l0 = leng.launches
        seq, lin, _ = leng.forward(ids.long(), am)
        self.launches += leng.launches - l0
        leng2 = None
        if "cls_input_ids" in batch:
            ids2, am2 = batch["cls_input_ids"], batch["cls_attention_mask"]
            leng2 = lm.engine(ids2.shape[0], ids2.shape[1], self.device, slot=1)
            leng2.set_dropout(*lm.dropout_config())
            l0 = leng2.launches
            _, lin, _ = leng2.forward(ids2.long(), am2)
            self.launches += leng2.launches - l0
        return seq, lin, leng, leng2

    def _lang_train_backward(self, leng, leng2, d_lang, d_cls):
        """The BERT backward of ``_lang_train_forward``: both passes accumulate into the one gradient arena."""
        l0 = leng.launches
        if leng2 is None:
            leng.backward(d_lang, d_cls, None)
        else:
            leng.backward(d_lang, None, None)
            l1 = leng2.launches
            leng2.backward(None, d_cls, None)
            self.launches += leng2.launches - l1
        self.launches += leng.launches - l0

    @torch.no_grad()
    def _teacher_rollout_poses(self, corners0, dirs0, geo, gt_paths, T):
        """The pose sequence of a teacher-feedback rollout (agent.py:580-770 with ``feedback == 'teacher'``): the
        action of every step is the ground-truth action, so the sequence does not depend on the model.  Per step:
        ``teacher_action`` (target waypoint / altitude / progress at the current view) and the simulator update with
        that target -- stop once the ground-truth progress exceeds ``self.STOP_THRESHOLD`` or at the last step.  All on
        the device; the host reads the stop flags once at the end.  Returns a dict of ``[T, B, ...]`` tensors and the
        step count."""
        ptr, call = _lib.ptr, _lib.call
        dev = self.device
        B = corners0.shape[0]
        f64, i32 = torch.float64, torch.int32
        corners = corners0.to(dev, f64).contiguous().clone()
        cur = dirs0.to(dev, f64).contiguous().clone()
        ended = torch.zeros(B, dtype=torch.uint8, device=dev)
        bounds = geo[:, :4].contiguous()
        H = dict(corners=torch.empty((T + 1, B, 4, 2), dtype=f64, device=dev), dirs=torch.empty((T + 1, B), dtype=f64, device=dev),
                 ended=torch.empty((T, B), dtype=torch.uint8, device=dev), xy=torch.empty((T, B, 2), device=dev),
                 alt=torch.empty((T, B), device=dev), prog=torch.empty((T, B), device=dev))
        ang = torch.empty(B, dtype=i32, device=dev); dist = torch.empty(B, dtype=f64, device=dev); alt_i = torch.empty(B, dtype=i32, device=dev)
        gt_pack = pack_gt_paths([gt_paths[i] for i in range(B)], dev)
        for t in range(T):
            H["corners"][t].copy_(corners); H["dirs"][t].copy_(cur)
            xy, alt, prog = self.teacher_action(corners, gt_pack, ended, feedback="teacher")
            H["xy"][t].copy_(xy); H["alt"][t].copy_(alt); H["prog"][t].copy_(prog)
            out = torch.cat((xy, alt[:, None], prog[:, None]), 1).contiguous()
            call("avdn_waypoint_step", ptr(out), ptr(corners), ptr(bounds), ptr(cur), ptr(ended), B,
                 float(self.STOP_THRESHOLD), int(t == T - 1), ptr(ang), ptr(dist), ptr(alt_i))
            H["ended"][t].copy_(ended)
            self.launches += 8
        H["corners"][T].copy_(corners); H["dirs"][T].copy_(cur)
        return H, steps_until_all_ended(H["ended"])

    def _rollout_setup(self):
        """The host side of the start of ``rollout`` over ``self.env`` (agent.py:512-570): the batch's items, its
        language batch, start poses, map geometry and the trajectory dicts the rollout fills."""
        env = self.env
        items = list(env.batch)
        dev = self.device
        env._sync_maps()
        lb, lang_inputs = self._language_batch(items)
        gps0 = np.stack([np.asarray(it["gt_path_corners"][0], dtype=np.float64) for it in items])
        _, geo_h, tidx_h = env._gather_poses(None, 0)
        geo = torch.from_numpy(geo_h).to(dev)
        tidx = torch.from_numpy(tidx_h).to(dev)
        dirs0 = torch.tensor([float(it["angle"]) for it in items], dtype=torch.float64, device=dev)
        gt_paths = [np.asarray(it["gt_path_corners"], dtype=np.float64) for it in items]
        traj = []
        for i, it in enumerate(items):
            rounds = lang_inputs[i].split("[QUE]")
            remove = sum(1 for r in rounds if "Yes" in r[0:5])
            traj.append({"instr_id": it["map_name"] + "__" + it["route_index"], "num_dia": len(rounds) - remove,
                         "path_corners": [(np.array(it["gt_path_corners"][0]), it["angle"])],
                         "gt_path_corners": it["gt_path_corners"], "actions": [], "gt_actions": [], "gt_progress": [],
                         "progress": []})
        return items, lb, gps0, geo, tidx, dirs0, gt_paths, traj

    @staticmethod
    def _log_traj(traj, outs, tgt, ended, corners, dirs, steps):
        """agent.py:637-653,725-770: per alive step the clipped prediction, the ground-truth action / progress and the
        pose the simulator moved to."""
        B = len(traj)
        for i in range(B):
            alive = True
            for t in range(steps):
                if alive:
                    o = outs[t, i]
                    m = max(abs(float(o[0])), abs(float(o[1])), 1.0)
                    traj[i]["actions"].append([np.array([o[0] / m, o[1] / m], dtype=np.float32),
                                               np.float32(min(1.0, max(0.0, float(o[2]))))])
                    traj[i]["progress"].append(float(o[3]))
                    if tgt is not None:
                        traj[i]["gt_actions"].append([tgt[0][t, i].copy(), float(tgt[1][t, i])])
                        traj[i]["gt_progress"].append(float(tgt[2][t, i]))
                alive = not ended[t, i]
                if alive:
                    traj[i]["path_corners"].append((corners[t + 1, i].copy(), float(dirs[t + 1, i])))

    def test(self, batches, env_name="no_name_provided", feedback="student", not_in_train=False, **kwargs):
        """``agent.test`` (agent.py:191-206): greedy rollouts in eval mode, one trajectory dict per
        episode in ``self.results[instr_id]`` -- the structure ``ANDHNavBatch.eval_metrics`` scores.

        With ``self.env`` set to an ``ANDHNavBatch`` this is the reference's loop: ``batches`` is the data loader (it
        fills ``self.env`` as it is iterated) and every item triggers ``self.rollout(not_in_train=True)``.  Otherwise:

        Every batch is the ``rollout_greedy`` input dict plus host metadata: ``instr_id`` list[str],
        ``gt_path_corners`` list of ``[n_i,4,2]`` arrays (optional: without it ``gt_progress`` is omitted, as for
        the unseen test split, agent.py:655) and ``num_dia`` list[int] (optional).  ``gt_progress`` is the
        reference's per-step IoU of the current view with the goal (``teacher_action``'s progress, agent.py:660,
        721), evaluated for all steps of the batch in one ``avdn_teacher_action`` launch."""
        self.feedback, self.env_name = feedback, env_name
        self.results, self.losses = {}, []
        if hasattr(self.env, "_get_obs"):
            self.vln_model.eval(); self.vision_model.eval()
            if self.lang_model is not None:
                self.lang_model.eval()
            self.loss = 0
            for _ in batches:
                for traj in self.rollout(not_in_train=True, **kwargs):
                    self.loss = 0
                    self.results[traj["instr_id"]] = traj
            return self.results
        for batch in batches:
            meta = {k: batch[k] for k in ("instr_id", "gt_path_corners", "num_dia") if k in batch}
            res = self.rollout_greedy({k: v for k, v in batch.items() if k not in meta}, **kwargs)
            steps = int(res["steps"]) if "steps" in res else steps_until_all_ended(res["ended"])
            corners = res["corners"]                                       # [T+1,B,4,2]
            B = corners.shape[1]
            ended = res["ended"].cpu().numpy().astype(bool)
            prog = None
            gts = meta.get("gt_path_corners")
            if gts is not None:
                flat = corners[:steps].reshape(steps * B, 4, 2)
                _, _, pr = self.teacher_action(flat, [gts[i % B] for i in range(steps * B)],
                                               np.zeros(steps * B, dtype=np.uint8), feedback="student")
                prog = pr.view(steps, B).cpu().numpy()
            c_host = corners.cpu().numpy()
            d_host = res["directions"].cpu().numpy()
            out_host = res["output"].cpu().numpy()
            for i in range(B):
                traj = {"instr_id": meta["instr_id"][i] if "instr_id" in meta else f"{env_name}_{len(self.results)}",
                        "path_corners": [(c_host[0, i], d_host[0, i])], "actions": [], "progress": []}
                if "num_dia" in meta:
                    traj["num_dia"] = int(meta["num_dia"][i])
                if gts is not None:
                    traj["gt_path_corners"] = gts[i]
                    traj["gt_progress"] = []
                alive = True
                for t in range(steps):
                    if alive:                                              # logged while the episode has not ended
                        traj["actions"].append(out_host[t, i, :3].copy())
                        traj["progress"].append(float(out_host[t, i, 3]))
                        if prog is not None:
                            traj["gt_progress"].append(float(prog[t, i]))
                    alive = not ended[t, i]
                    if alive:
                        traj["path_corners"].append((c_host[t + 1, i], d_host[t + 1, i]))
                self.results[traj["instr_id"]] = traj
        return self.results

    def train(self, loader, n_epochs, feedback="student", nss_w_weighting=1, **kwargs):
        """Drop-in for ``NavCMTAgent.train`` (src/xview_et/agent.py:208-254): for every batch the loader yields (the
        loader fills ``self.env`` as a side effect, as the reference's ``num_workers=0`` DataLoader does): zero the
        gradients, one teacher rollout (``feedback='teacher'``) or a teacher rollout without the NSS term followed by
        a student rollout (``'student'``), clip the policy's gradients to 40, one step of every optimiser."""
        self.vision_model.train(); self.vln_model.train()
        if self.lang_model is not None:
            self.lang_model.train()
        self.losses = []
        for epoch in range(1, n_epochs + 1):
            for _ in loader:
                for opt in self.optimizers:
                    opt.zero_grad()
                self.loss = 0
                if feedback == "teacher":
                    self.feedback = "teacher"
                    self.rollout(train_ml=float(getattr(self.args, "teacher_weight", 1.0)), train_rl=False,
                                 nss_w=float(getattr(self.args, "nss_w", 1.0)) * nss_w_weighting, **kwargs)
                elif feedback == "student":
                    self.feedback = "teacher"
                    self.rollout(train_ml=float(getattr(self.args, "ml_weight", 0.2)), train_rl=False, nss_w=0, **kwargs)
                    self.feedback = "student"
                    self.rollout(train_ml=float(getattr(self.args, "ml_weight", 0.2)), train_rl=False,
                                 nss_w=float(getattr(self.args, "nss_w", 1.0)) * nss_w_weighting, **kwargs)
                else:
                    assert False
                # (the reference calls self.loss.backward() here; the rollouts above already left their gradients in
                #  the arenas)  gradient all-reduce, clip (the policy only, agent.py:247), step
                self._reduce_and_step()

    def _reduce_and_step(self):
        """One step of every optimiser (a single process; the ET agent adds the data-parallel reduction)."""
        for opt in self.optimizers:
            self.launches += opt.step()

    def _add_rollout_loss(self, loss, train_ml):
        """``self.loss`` / ``self.losses`` bookkeeping of a rollout (agent.py:883-894)."""
        if train_ml is not None:
            l = loss.clone()
            self.loss = l if isinstance(self.loss, (int, float)) else self.loss + l
            self.losses.append(l)
        else:
            self.losses.append(0.0)

    # ------------------------------------------------------------- checkpoints
    def _checkpoint_items(self):
        """(entry name, module, optimiser, state-dict key prefixes not written) of every model (agent supplies)."""
        raise NotImplementedError

    def save(self, epoch, path):
        """agent.py:899-916: one entry per model -- ``{'epoch': epoch + 1, 'state_dict': module.state_dict(),
        'optimizer': {'m', 'v', 'step'}}`` (the flat AdamW arena: first and second moments over the optimiser's
        parameters in arena order, and the step count)."""
        d = os.path.dirname(path)
        if d:
            os.makedirs(d, exist_ok=True)
        states = {}
        for name, model, opt, skip in self._checkpoint_items():
            sd = model.state_dict()
            if skip:
                sd = {k: v for k, v in sd.items() if not k.startswith(skip)}
            states[name] = {"epoch": epoch + 1, "state_dict": sd,
                            "optimizer": {"m": opt.m.clone(), "v": opt.v.clone(), "step": opt.step_count}}
        torch.save(states, path)

    def load(self, path):
        """agent.py:918-940: parameters and buffers of every entry present (keys the module lacks are ignored), and
        with ``args.resume_optimizer`` the optimiser moments and step counts.  Returns the saved epoch."""
        states = torch.load(path, map_location=self.device)
        for name, model, opt, _ in self._checkpoint_items():
            if name not in states:
                continue
            state = model.state_dict()                       # tensors alias the arena: copy IN PLACE
            with torch.no_grad():
                for k, v in states[name]["state_dict"].items():
                    if k in state:
                        state[k].copy_(v)
            if getattr(self.args, "resume_optimizer", False):
                o = states[name].get("optimizer", {})
                if "m" not in o:
                    raise ValueError(f"checkpoint '{name}': optimiser state is not in the flat-arena format this agent "
                                     "writes ({'m', 'v', 'step'}); torch per-parameter optimiser states (the reference's "
                                     "format) cannot be resumed -- load with resume_optimizer=False")
                opt.m.copy_(o["m"]); opt.v.copy_(o["v"]); opt.step_count = int(o["step"])
        return states.get("vln_model", {}).get("epoch", 0) - 1


def pack_gt_paths(gt_path_corners, device):
    """Per sample ``[n_i,4,2]`` ground-truth view corners -> the ``(gt [B,max n_i,4,2] f64, lengths [B] i32)`` device
    pair ``teacher_action`` takes (zero-padded), so a loop of ``teacher_action`` launches packs them once."""
    lens = [len(g) for g in gt_path_corners]
    gt = np.zeros((len(lens), max(lens), 4, 2), dtype=np.float64)
    for i, g in enumerate(gt_path_corners):
        gt[i, :lens[i]] = np.asarray(g, dtype=np.float64)
    return torch.from_numpy(gt).to(device), torch.tensor(lens, dtype=torch.int32, device=device)


def steps_until_all_ended(ended):
    """The number of steps a rollout runs with the reference's early exit (agent.py:773-774): up to and including the
    first step after which every sample has ended.  ``ended`` [T,B] sticky stop flags (one host read)."""
    e = ended.cpu().numpy().astype(bool)
    for t in range(e.shape[0]):
        if e[t].all():
            return t + 1
    return e.shape[0]


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
    sb = rollout_step_bufs(agent, B, T)
    tengs = [vm.engine(B, 224, 224, dev, slot=1 + t) for t in range(T)]
    l0 = sum(e.launches for e in tengs)
    x5 = x.view(B, T, 224, 224, 4)
    f5 = frames_out.view(B, T, 512, 49)
    for t in range(T):
        sb["x"][t].copy_(x5[:, t])
        DN._trunk_forward(vm, tengs[t], sb["x"][t], True, out=sb["f"])
        f5[:, t].copy_(sb["f"].view(B, 512, 49))
    return tengs[0], tengs, l0, 2 * T


def rollout_step_bufs(agent, B, T):
    """Buffers of the per-step trunk passes of a rollout of B episodes and T steps: the views of every step, one
    step's features and their gradient."""
    key = ("rollout_steps", B, T)
    sb = agent._bufs.get(key)
    if sb is None:
        dev = agent.device
        sb = dict(x=[torch.empty((B, 224, 224, 4), dtype=torch.bfloat16, device=dev) for _ in range(T)],
                  f=torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev),
                  df=torch.empty((B, 512, 7, 7), dtype=torch.float32, device=dev))
        agent._bufs[key] = sb
    return sb


def rollout_trunk_backward(agent, teng, tengs, l0, d_frames, B, T, after_layer=None, flush_layers=None, steps=None):
    """Backward of ``rollout_trunk_forward`` from ``d_frames`` [B*T,512,49]; parameter gradients accumulate into
    the trunk's arena.  With per-step passes every pass runs back through its own activations and the last one
    (step 0) carries ``after_layer`` / ``flush_layers`` (the data-parallel buckets); ``steps`` (default T): only
    the passes of the first ``steps`` steps ran (a rollout that ended early).  Returns the launches."""
    vm = agent.vision_model
    if tengs is None:
        DN._trunk_backward(vm, teng, d_frames.view(-1, 512, 7, 7), after_layer=after_layer, flush_layers=flush_layers)
        return teng.launches - l0
    sb = agent._bufs[("rollout_steps", B, T)]
    d5 = d_frames.view(B, T, 512, 49)
    steps = T if steps is None else int(steps)
    for t in reversed(range(steps)):
        sb["df"].view(B, 512, 49).copy_(d5[:, t])
        last = (t == 0)
        DN._trunk_backward(vm, tengs[t], sb["df"], after_layer=after_layer if last else None,
                           flush_layers=flush_layers if last else None)
    return steps + sum(e.launches for e in tengs) - l0


def student_targets(agent, corners, ended, gt_path_corners):
    """The ``teacher_action`` target of every pose a student-feedback rollout visited (agent.py:655-661), in one
    launch.  ``corners`` [T,B,4,2] f64 (lat,lng) the pose before each step; ``ended`` [T,B] the sticky stop flags
    after each step -- the teacher sees at step t whether the sample had stopped before it; ``gt_path_corners``: per
    sample the ``[n_i,4,2]`` ground-truth view corners.  Returns ``(xy [T,B,2], alt [T,B], prog [T,B])`` f32."""
    T, B = corners.shape[0], corners.shape[1]
    ended_before = torch.zeros((T, B), dtype=torch.uint8, device=agent.device)
    ended_before[1:] = ended[:T - 1]
    xy, alt, prog = agent.teacher_action(corners.reshape(T * B, 4, 2), [gt_path_corners[k % B] for k in range(T * B)],
                                         ended_before.reshape(-1), feedback="student")
    return xy.view(T, B, 2), alt.view(T, B), prog.view(T, B)


def rollout_pose_batch(corners, geo, tile_idx, targets):
    """The poses of a ``train_rollout_step`` batch: a rollout that visited ``corners`` [T,B,4,2] (f64 lat,lng) on the
    maps ``geo`` [B,5] (``tile_idx`` i32 [B] or None), with ``targets`` = ``(xy [T,B,2], alt [T,B], prog [T,B])``.
    Returns a dict of [B,T,...] tensors ``corners_px`` (i32 pixel corners), ``tile_idx`` (or None), ``gt_xy``,
    ``gt_alt`` and ``gt_prog``."""
    T, B = corners.shape[0], corners.shape[1]
    px = torch.empty((T * B, 4, 2), dtype=torch.int32, device=corners.device)
    _lib.call("avdn_gps_to_pixels", _lib.ptr(corners.reshape(T * B, 4, 2).contiguous()),
              _lib.ptr(geo.repeat(T, 1).contiguous()), T * B, _lib.ptr(px))
    tb = lambda a: a.transpose(0, 1).contiguous()                  # step-major [T,B,...] -> [B,T,...]
    xy, alt, prog = targets
    return dict(corners_px=tb(px.view(T, B, 4, 2)),
                tile_idx=None if tile_idx is None else tile_idx.view(B, 1).expand(B, T).contiguous(),
                gt_xy=tb(xy.float()), gt_alt=tb(alt.float()), gt_prog=tb(prog.float()))
