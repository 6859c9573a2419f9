"""``ViT_LSTM`` -- the recurrent policy of AVDN's LSTM baseline, mirror of
src/models/vln_model.py:163-250 (BASELINE config 5: greedy waypoint rollout).

Same constructor (``ViT_LSTM(args, vit_model)``), same sub-module names and therefore
the same ``state_dict`` keys (including the ``pos_embedding`` and
``attention_layer_vision_lang`` parameters that the reference's forward never uses),
same ``forward(current_direct, im_input, pos_input, cls_hidden, lang_feature, h_0, c_0,
hh_0, cc_0) -> (h_1, c_1, hh_1, cc_1, output, pred_saliency)``.

``step`` / ``forward`` are the inference step (the rollout of ``agent.test``,
src/xview_lstm/agent.py:191-206, runs under ``.eval()``): dropout is the identity and the trunk uses its
running statistics; ``.train()`` + ``step`` raises.

Device work per step: trunk (tcgen05 convs, eval-mode BN folded into the apply pass),
``avdn_frame_attn_fwd`` (SoftDotAttention(49) over the 512 channels), ``avdn_linear_f32`` +
``avdn_lstm_cell`` for the two LSTM cells, ``avdn_lang_attn_fwd`` (SoftDotAttention(768) over
the dialog tokens) and fp32 linear layers for the two heads.

Training (``train_engine``): a whole teacher-forced rollout of T steps -- forward with train-mode dropout at the
four nn.Dropout sites as stateless hash masks, the loss of every step, backward through time
(``avdn_lstm_cell_bwd``, ``avdn_lang_attn_bwd``, ``avdn_frame_attn_bwd_cls`` without fc2,
``avdn_direction_embed_bwd``, ``avdn_linear_f32_bwd``) into the optimiser's gradient arena.  The trunk's forward
and backward around it belong to the agent (``xview_lstm.agent.NavCMTAgent.train_rollout_step``).
"""
from __future__ import annotations

import torch
from torch import nn

from .. import _lib

NCH, NSP, HID = 512, 49, 768


class SoftDotAttention(nn.Module):
    """Parameter container of src/models/vln_model.py:12-46."""

    def __init__(self, dim):
        super().__init__()
        self.linear_in = nn.Linear(dim, dim, bias=False)
        self.sm = nn.Softmax(dim=1)
        self.linear_out = nn.Linear(dim * 2, dim, bias=False)
        self.tanh = nn.Tanh()


class _StepBufs:
    """Per-(B, L) device buffers of one policy step.  The recurrent state lives here, double
    buffered by step parity: ``cat2[k]`` = [weighted (768) | h (192) | hh (576)] is at once the input of
    ``attention_layer_lang.linear_out`` and the home of the new hidden states."""

    def __init__(self, B, L, dev):
        f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        self.attn512, self.wc, self.e49 = f(B, NCH), f(B, NSP), f(B, NSP)
        self.gates_v, self.gates_d = f(B, 4 * 576), f(B, 4 * 192)
        self.deg, self.dir_emb = f(B), f(B, 32)
        self.cat2 = [f(B, 2 * HID), f(B, 2 * HID)]
        self.c_d, self.c_v = [f(B, 192), f(B, 192)], [f(B, 576), f(B, 576)]
        self.target, self.act_in = f(B, HID), f(B, HID)
        self.m0, self.m1, self.output = f(B, 256), f(B, 32), f(B, 4)
        self.s0, self.h_sali = f(B, 128), f(B, 64)
        self.k = 0                                   # parity of the NEXT step
        self.has_state = False

    def h(self, k):
        return self.cat2[k][:, HID:HID + 192]

    def hh(self, k):
        return self.cat2[k][:, HID + 192:]


# hash-dropout sites of the training rollout (disjoint from ET's 0 .. 4*layers-1 and 1000-1002 and BERT's 96, 97,
# 100 + 3*layer + k): self.drop on the input of vision_lstm and the Dropout(0.2) inside fc cover every step at once
# (element index t*B*K + b*K + k over a [T,B,K] tensor); the two Dropout(0.2) of decoder_2_action_full run once per
# step, site SITE_DEC + 2t (after the first hidden ReLU) and SITE_DEC + 2t + 1 (after the second).
SITE_INPUT, SITE_FC, SITE_DEC = 3000, 3001, 3002
DROP_P = 0.2                       # nn.Dropout(p=0.2) at all four sites (vln_model.py:163-250)


class _TrainEngine:
    """Teacher-forced training rollout of ``ViT_LSTM`` over T steps (src/xview_lstm/agent.py:546-550,592-602,636):
    the forward of every step keeps its activations in step-t slots, the backward runs t = T-1 ... 0.

    Frame-major tensors ([B*T, ...], the trunk's order): ``attn512``, ``wc``, ``e49`` (frame attention of every step
    in one launch: the frames of all steps are known before the first step), ``d_frames``.  Step-major tensors
    ([T, B, ...]): everything else; ``cat2[t]`` = [weighted | h | hh] is the input of attention_layer_lang.linear_out
    and the home of step t's hidden states, as in ``_StepBufs``.

    Only the data-gradient chain through the two LSTM cells and the language attention is sequential.  The heads of
    every step are differentiated before the loop, and every weight gradient is ONE ``avdn_linear_f32_bwd`` over all
    T*B rows after it, accumulated into ``G`` (the optimiser arena when one is attached)."""

    def __init__(self, model, B, L, T, device, grads):
        f = lambda *s: torch.zeros(s, dtype=torch.float32, device=device)
        self.m, self.B, self.L, self.T = model, B, L, T
        BT = B * T
        self.attn512, self.wc, self.e49 = f(BT, NCH), f(BT, NSP), f(BT, NSP)
        self.e49_t, self.e49d = f(T, B, NSP), f(T, B, NSP)
        self.deg, self.dir_emb = f(T, B), f(T, B, 32)
        self.gates_v, self.gates_d = f(T, B, 4 * 576), f(T, B, 4 * 192)
        self.c_v, self.c_d = f(T, B, 576), f(T, B, 192)
        self.cat2 = f(T, B, 2 * HID)
        self.target, self.attn, self.act_in = f(T, B, HID), f(T, B, L), f(T, B, HID)
        self.m0, self.m1, self.output = f(T, B, 256), f(T, B, 32), f(T, B, 4)
        self.s0, self.h_sali = f(T, B, 128), f(T, B, 64)
        self.loss_i = torch.zeros(BT, dtype=torch.float64, device=device)
        self.d_output, self.d_h_sali = f(T, B, 4), f(T, B, 64)
        self.d_m1, self.d_m0, self.d_act_in = f(T, B, 32), f(T, B, 256), f(T, B, HID)
        self.d_cat2, self.d_target = f(T, B, 2 * HID), f(T, B, HID)
        self.dg_v, self.dg_d = f(T, B, 4 * 576), f(T, B, 4 * 192)
        self.dc_v, self.dc_d = f(B, 576), f(B, 192)          # cell-state gradient carried from step t+1 to t
        self.d_s0, self.d_e49, self.d_dir = f(T, B, 128), f(T, B, NSP), f(T, B, 32)
        self.d_e49_bt, self.d_frames = f(BT, NSP), f(BT, NCH, NSP)
        self.G = grads if grads is not None else {n: torch.zeros_like(p) for n, p in model.used_parameters().items()}
        self.p, self.seed = 0.0, 0
        self.launches = 0

    def _lin_bwd(self, x, w, y, dy, act, dx, name, bias=True, dx_accumulate=0):
        """avdn_linear_f32_bwd over 2-D views: dx (may be None) and the gradients of parameter ``name`` (+=)."""
        M, K = x.shape
        G = self.G
        _lib.call("avdn_linear_f32_bwd", _lib.ptr(x), x.stride(0), _lib.ptr(w), _lib.ptr(y), _lib.ptr(dy), M,
                  dy.shape[1], K, act, _lib.ptr(dx), dx.stride(0) if dx is not None else 0, dx_accumulate,
                  _lib.ptr(G[name + ".weight"] if bias else G[name]), _lib.ptr(G[name + ".bias"]) if bias else None)

    def forward(self, frames, deg, cls_hidden, lang_feature, p=0.0, seed=0):
        """The T policy steps on trunk features ``frames`` [B*T,512,49] f32 (episode-major, as the trunk emits them)
        with headings ``deg`` [B,T] (degrees), ``cls_hidden`` [B,49], ``lang_feature`` [B,L,768]; dropout ``p`` with
        hash seed ``seed`` (``ViT_LSTM.dropout_config``).  Returns ``output`` [T,B,4] and ``h_sali`` [T,B,64]."""
        m, B, L, T = self.m, self.B, self.L, self.T
        call, ptr = _lib.call, _lib.ptr
        BT = B * T
        l0 = m.launches
        self.p, self.seed = float(p), int(seed)
        self._in = (frames.contiguous(), cls_hidden.contiguous(), lang_feature.contiguous())
        frames, cls, lang = self._in
        av = m.attention_layer_vision
        # input_lstm_0 of every step (vln_model.py:219)
        call("avdn_frame_attn_fwd", ptr(frames), ptr(cls), ptr(av.linear_in.weight), ptr(av.linear_out.weight), None,
             None, B, T, ptr(self.attn512), ptr(self.wc), ptr(self.e49), None)
        self.e49_t.copy_(self.e49.view(B, T, NSP).transpose(0, 1))
        call("avdn_add_dropout_f32", ptr(self.e49_t), None, ptr(self.e49d), BT * NSP, self.p, self.seed, SITE_INPUT)
        # direction_embedding of every step (vln_model.py:228-229)
        self.deg.copy_(deg.t())
        call("avdn_direction_embed", ptr(self.deg), ptr(m.direction_embedding.weight), ptr(m.direction_embedding.bias),
             ptr(self.dir_emb), BT, 32)
        for t in range(T):
            self._step_body(t, lang)
        self._saliency(T)
        self.launches += 6 + 3 * T + (m.launches - l0)
        return self.output, self.h_sali

    def begin(self, cls_hidden, lang_feature, p=0.0, seed=0):
        """Start a step-wise forward (``step`` per time step, then ``finish``): the same activations as ``forward``,
        for a rollout whose frames and headings of step t+1 depend on the output of step t.  Arguments as for
        ``forward``."""
        self.p, self.seed = float(p), int(seed)
        if getattr(self, "_frames", None) is None:
            f = lambda *s: torch.zeros(s, dtype=torch.float32, device=self.deg.device)
            self._frames = f(self.B * self.T, NCH, NSP)                 # frame-major input, read by backward
            self._st = (f(self.B, NCH), f(self.B, NSP), f(self.B, NSP))  # attn512 / wc / e49 of one step
        self._in = (self._frames, cls_hidden.contiguous(), lang_feature.contiguous())
        self.n_run = 0

    def step(self, t, frames_t, deg_t):
        """Policy step ``t`` (0, 1, ... in order) of a ``begin``-started forward on the B frames ``frames_t``
        [B,512,49] f32 and headings ``deg_t`` [B] (degrees).  Returns ``output[t]`` [B,4] (a view, valid until the
        engine's next forward)."""
        m, B, T = self.m, self.B, self.T
        call, ptr = _lib.call, _lib.ptr
        if t != self.n_run or t >= T:
            raise ValueError(f"step {t}: expected step {self.n_run} of {T}")
        l0 = m.launches
        _, cls, lang = self._in
        av = m.attention_layer_vision
        imf = frames_t.contiguous()
        attn512, wc, e49 = self._st
        call("avdn_frame_attn_fwd", ptr(imf), ptr(cls), ptr(av.linear_in.weight), ptr(av.linear_out.weight), None,
             None, B, 1, ptr(attn512), ptr(wc), ptr(e49), None)
        # the frame-major rows b*T + t of step t
        self.attn512.view(B, T, NCH)[:, t].copy_(attn512)
        self.wc.view(B, T, NSP)[:, t].copy_(wc)
        self.e49.view(B, T, NSP)[:, t].copy_(e49)
        self._frames.view(B, T, NCH, NSP)[:, t].copy_(imf.view(B, NCH, NSP))
        self.e49_t[t].copy_(e49)
        # step t's slice of the [T,B,49] input dropout: the mask forward draws over the whole rollout
        call("avdn_add_dropout_f32_at", ptr(self.e49_t[t]), None, ptr(self.e49d[t]), B * NSP, t * B * NSP, self.p,
             self.seed, SITE_INPUT)
        self.deg[t].copy_(deg_t.reshape(B))
        call("avdn_direction_embed", ptr(self.deg[t]), ptr(m.direction_embedding.weight),
             ptr(m.direction_embedding.bias), ptr(self.dir_emb[t]), B, 32)
        self._step_body(t, lang)
        self.n_run = t + 1
        self.launches += 12 + (m.launches - l0)
        return self.output[t]

    def finish(self):
        """End a step-wise forward: the saliency branch of the steps that ran.  Returns ``output`` [T,B,4] and
        ``h_sali`` [T,B,64] (rows of the first ``n_run`` steps)."""
        l0 = self.m.launches
        self._saliency(self.n_run)
        self.launches += 1 + (self.m.launches - l0)
        return self.output, self.h_sali

    def _saliency(self, n):
        """pred_saliency's fc over the first n steps; it reads the undropped input_lstm_0 (vln_model.py:244)."""
        m, call, ptr = self.m, _lib.call, _lib.ptr
        fc, nB = m.fc, n * self.B
        m._linear(self.e49_t[:n].view(nB, NSP), fc[0].weight, fc[0].bias, self.s0[:n].view(nB, 128), act=1)
        call("avdn_dropout_f32", ptr(self.s0), None, nB * 128, self.p, self.seed, SITE_FC)
        m._linear(self.s0[:n].view(nB, 128), fc[3].weight, fc[3].bias, self.h_sali[:n].view(nB, 64), act=1)

    def _step_body(self, t, lang):
        """The recurrent part of step t on ``e49d[t]`` and ``dir_emb[t]``: the two LSTM cells, the language attention
        and the action head (3 launches of its own besides the linear layers)."""
        m, B, L = self.m, self.B, self.L
        call, ptr = _lib.call, _lib.ptr
        al, dec = m.attention_layer_lang, m.decoder_2_action_full
        cat = self.cat2[t]
        prev = self.cat2[t - 1] if t > 0 else None
        # hh_1, cc_1 = vision_lstm(drop(input_lstm_0), (hh_0, cc_0))                vln_model.py:220-226
        m._lstm(m.vision_lstm, self.e49d[t], prev[:, HID + 192:] if t else None, self.c_v[t - 1] if t else None,
                self.gates_v[t], cat[:, HID + 192:], self.c_v[t])
        m._lstm(m.direct_lstm, self.dir_emb[t], prev[:, HID:HID + 192] if t else None,
                self.c_d[t - 1] if t else None, self.gates_d[t], cat[:, HID:HID + 192], self.c_d[t])
        # action_module_input = SoftDotAttention(768)(cat(h_1, hh_1), lang_feature)  vln_model.py:238-239
        m._linear(cat[:, HID:], al.linear_in.weight, None, self.target[t])
        call("avdn_lang_attn_fwd", ptr(lang), ptr(self.target[t]), B, L, HID, ptr(self.attn[t]), ptr(cat),
             cat.stride(0))
        m._linear(cat, al.linear_out.weight, None, self.act_in[t], act=2)
        # output = decoder_2_action_full(action_module_input)                       vln_model.py:248
        m._linear(self.act_in[t], dec[0].weight, dec[0].bias, self.m0[t], act=1)
        call("avdn_dropout_f32", ptr(self.m0[t]), None, B * 256, self.p, self.seed, SITE_DEC + 2 * t)
        m._linear(self.m0[t], dec[3].weight, dec[3].bias, self.m1[t], act=1)
        call("avdn_dropout_f32", ptr(self.m1[t]), None, B * 32, self.p, self.seed, SITE_DEC + 2 * t + 1)
        m._linear(self.m1[t], dec[6].weight, dec[6].bias, self.output[t])

    def loss(self, gt_xy, gt_alt, gt_prog, att, nss_w, nss_r, scale, loss_total, n_steps=None):
        """``avdn_loss`` of every step in one launch (T*B independent rows; jitter 0, src/xview_lstm/agent.py:636):
        ``loss_total`` += scale * sum of the step losses; ``d_output`` / ``d_h_sali`` receive their gradients.
        ``gt_xy`` [T,B,2], ``gt_alt`` / ``gt_prog`` [T,B] f32, ``att`` u8 [T,B,224,224] or None.  ``n_steps`` (default
        T): only the first n_steps steps count (a rollout that ended early); the targets then hold n_steps rows."""
        ptr = _lib.ptr
        n = self.T if n_steps is None else int(n_steps)
        _lib.call("avdn_loss", ptr(self.output), ptr(self.h_sali), ptr(gt_xy), ptr(gt_alt), ptr(gt_prog), ptr(att),
                  None, self.B * n, float(nss_w), int(nss_r), float(scale), ptr(loss_total), ptr(self.loss_i),
                  ptr(self.d_output), ptr(self.d_h_sali))
        self.launches += 1

    def backward(self, d_lang=None, d_cls=None, n_steps=None):
        """Backward through time from ``d_output`` / ``d_h_sali`` (written by ``loss``).  Overwrites ``d_frames``
        [B*T,512,49] (returned); accumulates every parameter gradient into ``G`` and, when given, the gradients of
        ``lang_feature`` into ``d_lang`` [B,L,768] and of ``cls_hidden`` into ``d_cls`` [B,49] (+=).  ``n_steps``
        (default T, as given to ``loss``): the steps the rollout ran; the rows of later steps get zero ``d_frames``
        and contribute nothing."""
        m, B, L = self.m, self.B, self.L
        T = self.T if n_steps is None else int(n_steps)
        call, ptr = _lib.call, _lib.ptr
        BT = B * T
        l0 = m.launches
        p, seed = self.p, self.seed
        frames, cls, lang = self._in
        av, al, dec, fc = m.attention_layer_vision, m.attention_layer_lang, m.decoder_2_action_full, m.fc
        vl, dl = m.vision_lstm, m.direct_lstm
        r = lambda a: a[:T].view(BT, a.shape[-1])          # step-major: the first T steps are the first B*T rows
        n = 0
        # ---- the action head of every step (nothing recurrent), down to d cat2 = [d weighted | d h | d hh] ----
        self._lin_bwd(r(self.m1), dec[6].weight, r(self.d_output), r(self.d_output), 0, r(self.d_m1),
                      "decoder_2_action_full.6")
        for t in range(T):
            call("avdn_dropout_f32", ptr(self.d_m1[t]), None, B * 32, p, seed, SITE_DEC + 2 * t + 1)
        self._lin_bwd(r(self.m0), dec[3].weight, r(self.m1), r(self.d_m1), 1, r(self.d_m0), "decoder_2_action_full.3")
        for t in range(T):
            call("avdn_dropout_f32", ptr(self.d_m0[t]), None, B * 256, p, seed, SITE_DEC + 2 * t)
        self._lin_bwd(r(self.act_in), dec[0].weight, r(self.m0), r(self.d_m0), 1, r(self.d_act_in),
                      "decoder_2_action_full.0")
        self._lin_bwd(r(self.cat2), al.linear_out.weight, r(self.act_in), r(self.d_act_in), 2, r(self.d_cat2),
                      "attention_layer_lang.linear_out.weight", bias=False)
        n += 4 + 2 * T
        # ---- backward through time: the data gradients that cross steps ----
        w_in_t = al.linear_in.weight.t().contiguous()           # d hcat = d target W_in  (linear_f32: x w^T)
        w_hh_v_t, w_hh_d_t = vl.weight_hh.t().contiguous(), dl.weight_hh.t().contiguous()
        for t in reversed(range(T)):
            dcat = self.d_cat2[t]
            call("avdn_lang_attn_bwd", ptr(lang), ptr(self.target[t]), ptr(self.attn[t]), ptr(dcat), dcat.stride(0),
                 B, L, HID, ptr(self.d_target[t]), ptr(d_lang))
            m._linear(self.d_target[t], w_in_t, None, dcat[:, HID:], accumulate=1)
            first, last = t == 0, t == T - 1
            call("avdn_lstm_cell_bwd", ptr(self.gates_d[t]), None if first else ptr(self.c_d[t - 1]), ptr(self.c_d[t]),
                 ptr(dcat[:, HID:HID + 192]), dcat.stride(0), None if last else ptr(self.dc_d), ptr(self.dg_d[t]),
                 ptr(self.dc_d), B, 192)
            call("avdn_lstm_cell_bwd", ptr(self.gates_v[t]), None if first else ptr(self.c_v[t - 1]), ptr(self.c_v[t]),
                 ptr(dcat[:, HID + 192:]), dcat.stride(0), None if last else ptr(self.dc_v), ptr(self.dg_v[t]),
                 ptr(self.dc_v), B, 576)
            n += 3
            if not first:                  # h and hh of step t-1 fed this step's gates through W_hh
                prev = self.d_cat2[t - 1]
                m._linear(self.dg_d[t], w_hh_d_t, None, prev[:, HID:HID + 192], accumulate=1)
                m._linear(self.dg_v[t], w_hh_v_t, None, prev[:, HID + 192:], accumulate=1)
        # ---- weight gradients over all T*B rows ----
        cat = r(self.cat2)
        self._lin_bwd(cat[:, HID:], al.linear_in.weight, r(self.d_target), r(self.d_target), 0, None,
                      "attention_layer_lang.linear_in.weight", bias=False)
        for cell, name, dg, x, dx, lo in ((vl, "vision_lstm", self.dg_v, self.e49d, self.d_e49, HID + 192),
                                          (dl, "direct_lstm", self.dg_d, self.dir_emb, self.d_dir, HID)):
            G = self.G
            _lib.call("avdn_linear_f32_bwd", ptr(r(x)), x.shape[-1], ptr(cell.weight_ih), ptr(r(dg)), ptr(r(dg)), BT,
                      dg.shape[-1], x.shape[-1], 0, ptr(dx), dx.shape[-1], 0, ptr(G[name + ".weight_ih"]),
                      ptr(G[name + ".bias_ih"]))
            if T > 1:                      # step 0 ran from the zero state: W_hh saw h = 0 there
                H = cell.hidden_size
                h_prev = self.cat2[:T - 1].view((T - 1) * B, 2 * HID)[:, lo:lo + H]
                dg1 = dg[1:T].view((T - 1) * B, 4 * H)
                _lib.call("avdn_linear_f32_bwd", ptr(h_prev), h_prev.stride(0), ptr(cell.weight_hh), ptr(dg1),
                          ptr(dg1), (T - 1) * B, 4 * H, H, 0, None, 0, 0, ptr(G[name + ".weight_hh"]), None)
                n += 1
            call("avdn_colsum", ptr(dg), 1, BT, dg.shape[-1], dg.shape[-1], ptr(G[name + ".bias_hh"]))
            n += 2
        call("avdn_direction_embed_bwd", ptr(self.deg), ptr(self.d_dir), BT, 32, ptr(self.G["direction_embedding.weight"]),
             ptr(self.G["direction_embedding.bias"]))
        # ---- input_lstm_0: the dropped copy fed vision_lstm, the undropped one the saliency fc ----
        call("avdn_dropout_f32", ptr(self.d_e49), None, BT * NSP, p, seed, SITE_INPUT)
        self._lin_bwd(r(self.s0), fc[3].weight, r(self.h_sali), r(self.d_h_sali), 1, r(self.d_s0), "fc.3")
        call("avdn_dropout_f32", ptr(self.d_s0), None, BT * 128, p, seed, SITE_FC)
        self._lin_bwd(r(self.e49_t), fc[0].weight, r(self.s0), r(self.d_s0), 1, r(self.d_e49), "fc.0", dx_accumulate=1)
        if T < self.T:                     # steps that did not run: no gradient reaches their frames
            self.d_e49[T:].zero_()
        self.d_e49_bt.view(B, self.T, NSP).copy_(self.d_e49.transpose(0, 1))
        call("avdn_frame_attn_bwd_cls", ptr(frames), ptr(cls), ptr(av.linear_in.weight), ptr(av.linear_out.weight),
             None, B, self.T, ptr(self.attn512), ptr(self.wc), ptr(self.e49), ptr(self.d_e49_bt), ptr(self.d_frames),
             ptr(self.G["attention_layer_vision.linear_in.weight"]), ptr(self.G["attention_layer_vision.linear_out.weight"]),
             None, None, ptr(d_cls))
        n += 10
        self.launches += n + (m.launches - l0)
        return self.d_frames


class ViT_LSTM(nn.Module):
    def __init__(self, args, vit_model, hidden_size=768, dropout_ratio=0.5, im_channel_size=512, im_feature_size=49,
                 embedding_size=32):
        super().__init__()
        assert hidden_size == HID and im_channel_size == NCH and im_feature_size == NSP and embedding_size == 32, \
            "the reference hard-codes these sizes (vln_model.py:164-165,182,185)"
        self.args = args
        self.direction_embedding = nn.Linear(2, embedding_size)
        self.pos_embedding = nn.Linear(2, embedding_size)            # unused by forward (as in the reference)
        self.vision_model = vit_model
        self.attention_layer_lang = SoftDotAttention(hidden_size)
        self.attention_layer_vision_lang = SoftDotAttention(hidden_size)   # unused by forward
        self.attention_layer_vision = SoftDotAttention(im_feature_size)
        self.vision_lstm = nn.LSTMCell(im_feature_size, 576)
        self.drop = nn.Dropout(p=0.2)
        self.direct_lstm = nn.LSTMCell(embedding_size, 192)
        self.decoder_2_action_full = nn.Sequential(nn.Linear(hidden_size, 256), nn.ReLU(), nn.Dropout(0.2),
                                                   nn.Linear(256, 32), nn.ReLU(), nn.Dropout(0.2), nn.Linear(32, 4))
        self.fc = nn.Sequential(nn.Linear(im_feature_size, 128), nn.ReLU(), nn.Dropout(0.2), nn.Linear(128, 64),
                                nn.ReLU())
        self._bufs = {}
        self._train_engines = {}
        self._grad_arena = None          # name -> tensor, set by the optimiser arena (xview_lstm.agent)
        self.launches = 0

    # names of the parameters the training rollout updates: the trunk has its own optimiser arena, and the reference
    # forward never uses pos_embedding / attention_layer_vision_lang (their grad is None there)
    def used_parameters(self):
        skip = ("vision_model.", "pos_embedding.", "attention_layer_vision_lang.")
        return {n: p for n, p in self.named_parameters() if not n.startswith(skip)}

    def dropout_config(self):
        """(p, seed) of the next training rollout: nn.Dropout(0.2) at the four sites in train mode, (0, 0) in eval
        mode.  The seed advances every train-mode rollout and derives from torch's global seed and ``drop_rank``."""
        if not self.training:
            return 0.0, 0
        self._drop_step = getattr(self, "_drop_step", 0) + 1
        seed = (torch.initial_seed() * 1000003 + 7933 * self._drop_step
                + 0x9E3779B97F4A7C15 * int(getattr(self, "drop_rank", 0))) & 0xFFFFFFFFFFFFFFFF
        return DROP_P, seed

    def train_engine(self, B, L, T, device):
        """The training-rollout engine of (B episodes, L tokens, T steps) (``_TrainEngine``); parameter gradients go
        to the attached optimiser arena, or to engine-owned buffers ``engine.G`` when there is none."""
        key = (B, L, T, str(device))
        eng = self._train_engines.get(key)
        if eng is None:
            eng = self._train_engines[key] = _TrainEngine(self, B, L, T, device, self._grad_arena)
        return eng

    # ------------------------------------------------------------------ pieces
    def _linear(self, x, w, b, y, act=0, accumulate=0):
        M, K = x.shape
        N = w.shape[0]
        _lib.call("avdn_linear_f32", _lib.ptr(x), x.stride(0), _lib.ptr(w), w.stride(0), _lib.ptr(b), _lib.ptr(y),
                  y.stride(0), M, N, K, act, accumulate)
        self.launches += 1

    def _lstm(self, cell, x, h_prev, c_prev, gates, h_out, c_out):
        """nn.LSTMCell (vln_model.py:224-236): gates = W_ih x + b_ih + W_hh h + b_hh; zero state if None."""
        B, H = x.shape[0], cell.hidden_size
        if h_prev is None:                           # W_hh . 0 = 0: only the two bias vectors remain
            self._linear(x, cell.weight_ih, cell.bias_ih, gates)
            self._linear(torch.ones((B, 1), device=x.device), cell.bias_hh.view(-1, 1), None, gates, accumulate=1)
        else:
            self._linear(x, cell.weight_ih, cell.bias_ih, gates)
            self._linear(h_prev, cell.weight_hh, cell.bias_hh, gates, accumulate=1)
        _lib.call("avdn_lstm_cell", _lib.ptr(gates), _lib.ptr(c_prev), _lib.ptr(h_out), h_out.stride(0),
                  _lib.ptr(c_out), B, H)
        self.launches += 1

    def bufs(self, B, L, dev):
        # one key per physical device: reset_state(..., "cuda") and a step on tensors of "cuda:0" must share the state
        dev = torch.device(dev)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        key = (B, L, str(dev))
        bf = self._bufs.get(key)
        if bf is None:
            bf = self._bufs[key] = _StepBufs(B, L, dev)
        return bf

    def reset_state(self, B, L, dev):
        """Zero-init the recurrent state (src/xview_lstm/agent.py:546-550: h_0 = c_0 = hh_0 = cc_0 = None)."""
        bf = self.bufs(B, L, dev)
        bf.has_state, bf.k = False, 0
        return bf

    def step(self, im_feature, current_direct, cls_hidden, lang_feature, want_saliency=True):
        """One policy step on trunk features ``im_feature`` [B,512,49] f32 (device), advancing the
        recurrent state held in the (B, L) buffers.  Returns (output [B,4], h_sali [B,64] or None);
        both are views of step buffers, valid until the next call."""
        if self.training:
            raise NotImplementedError("ViT_LSTM is inference-only here (BASELINE config 5); call .eval()")
        _lib.require_cuda(im_feature, current_direct, cls_hidden, lang_feature)
        B, L = lang_feature.shape[0], lang_feature.shape[1]
        bf = self.bufs(B, L, im_feature.device)
        ptr, call = _lib.ptr, _lib.call
        k, p = bf.k, bf.k ^ 1
        prev = bf.has_state
        # named references: a temporary inside ptr(...) would be freed before the launch
        imf, cls, lf = im_feature.contiguous(), cls_hidden.contiguous(), lang_feature.contiguous()
        av, al = self.attention_layer_vision, self.attention_layer_lang
        # input_lstm_0 = SoftDotAttention(49)(cls_hidden, im_feature)              vln_model.py:219
        call("avdn_frame_attn_fwd", ptr(imf), ptr(cls), ptr(av.linear_in.weight),
             ptr(av.linear_out.weight), None, None, B, 1, ptr(bf.attn512), ptr(bf.wc), ptr(bf.e49), None)
        # hh_1, cc_1 = vision_lstm(drop(input_lstm_0), (hh_0, cc_0))                vln_model.py:220-226
        self._lstm(self.vision_lstm, bf.e49, bf.hh(p) if prev else None, bf.c_v[p] if prev else None, bf.gates_v,
                   bf.hh(k), bf.c_v[k])
        # direction_embedding([sin, cos](current_direct / 180 * 3.14159))           vln_model.py:228-229
        bf.deg.copy_(current_direct.reshape(B))      # int64 / float -> float32, as torch's true division does
        call("avdn_direction_embed", ptr(bf.deg), ptr(self.direction_embedding.weight),
             ptr(self.direction_embedding.bias), ptr(bf.dir_emb), B, 32)
        self._lstm(self.direct_lstm, bf.dir_emb, bf.h(p) if prev else None, bf.c_d[p] if prev else None, bf.gates_d,
                   bf.h(k), bf.c_d[k])
        # action_module_input = SoftDotAttention(768)(cat(h_1, hh_1), lang_feature)  vln_model.py:238-239
        hcat = bf.cat2[k][:, HID:]
        self._linear(hcat, al.linear_in.weight, None, bf.target)
        call("avdn_lang_attn_fwd", ptr(lf), ptr(bf.target), B, L, HID, None, ptr(bf.cat2[k]),
             bf.cat2[k].stride(0))
        self._linear(bf.cat2[k], al.linear_out.weight, None, bf.act_in, act=2)
        # output = decoder_2_action_full(action_module_input)                       vln_model.py:248
        dec = self.decoder_2_action_full
        self._linear(bf.act_in, dec[0].weight, dec[0].bias, bf.m0, act=1)
        self._linear(bf.m0, dec[3].weight, dec[3].bias, bf.m1, act=1)
        self._linear(bf.m1, dec[6].weight, dec[6].bias, bf.output)
        self.launches += 3
        h_sali = None
        if want_saliency:                                                          # vln_model.py:244
            self._linear(bf.e49, self.fc[0].weight, self.fc[0].bias, bf.s0, act=1)
            self._linear(bf.s0, self.fc[3].weight, self.fc[3].bias, bf.h_sali, act=1)
            h_sali = bf.h_sali
        bf.k, bf.has_state = p, True
        return bf.output, h_sali

    def state(self, B, L, dev):
        """(h, c, hh, cc) after the last step (copies)."""
        bf = self.bufs(B, L, dev)
        k = bf.k ^ 1
        return bf.h(k).clone(), bf.c_d[k].clone(), bf.hh(k).clone(), bf.c_v[k].clone()

    def forward(self, current_direct, im_input, pos_input, cls_hidden, lang_feature, h_0=None, c_0=None, hh_0=None,
                cc_0=None):
        """Reference signature (vln_model.py:213).  ``im_input`` [B,3,224,224] f32 normalised."""
        with torch.no_grad():
            feat = self.vision_model(im_input)                                      # [B,512,7,7]
            B, L = feat.shape[0], lang_feature.shape[1]
            given = [x is not None for x in (h_0, c_0, hh_0, cc_0)]
            if any(given) and not all(given):
                raise ValueError("pass all four recurrent states or none")
            bf = self.reset_state(B, L, feat.device)
            if all(given):                         # load the caller's state into the 'previous' buffers
                p = bf.k ^ 1
                bf.h(p).copy_(h_0); bf.c_d[p].copy_(c_0); bf.hh(p).copy_(hh_0); bf.c_v[p].copy_(cc_0)
                bf.has_state = True
            output, h_sali = self.step(feat.view(B, NCH, NSP), current_direct, cls_hidden, lang_feature)
            pred = torch.empty((B, 1, 224, 224), dtype=torch.float32, device=feat.device)
            _lib.call("avdn_upsample_saliency", _lib.ptr(h_sali), B, _lib.ptr(pred))
            h1, c1, hh1, cc1 = self.state(B, L, feat.device)
        return h1, c1, hh1, cc1, output.clone(), pred
