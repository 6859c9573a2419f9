"""``CustomBERTModel`` -- the language encoder that feeds the AVDN hot path (mirror of
src/models/vln_model.py:128-159; SURVEY.md §8f N1, the first row after the hot path itself).

Same module surface: ``self.bert`` is a HuggingFace ``BertModel`` ('bert-base-uncased' architecture) used as the
PARAMETER CONTAINER only (so that reference checkpoints / ``from_pretrained`` weights load under the same
``state_dict`` keys; its ``forward`` is never called), ``self.linears`` the reference's 2-layer head;
``forward(ids, mask) -> (sequence_output [B,S,768], linear_output [B,49], cls_hidden [B,768])``.

All arithmetic runs on libavdn: tcgen05 GEMMs (bf16 operands, fp32 accumulation) for the projections, QK^T, PV
and the FFN, with their backward; warp-level kernels for the embeddings + LayerNorm (eps 1e-12), the key-padding
softmax, erf-GELU and the small fp32 heads.  ``mask`` must be right-padded (what ``tokenizer(padding=True)``
produces, agent.py:527-529): sample b attends keys ``k < mask[b].sum()``.

Dropout (train mode): HF's sites -- after the embedding LayerNorm, on the attention probabilities, on the attention
output projection and on the FFN output (``hidden_dropout_prob`` / ``attention_probs_dropout_prob``) -- and the
head's Dropout(0.2), as stateless hash masks of (seed, site, element) re-evaluated by the backward kernels
(``BertEngine.set_dropout``; sites: 96 embeddings, 97 head, 100 + 3l + {0: probabilities, 1: attention output,
2: FFN output}).  Eval mode is deterministic.
"""
from __future__ import annotations

import math

import torch
from torch import nn

from .. import _lib
from .. import gemm as G
from ._lease import EnginePool, lease_slot

E = 768
LN_EPS = 1e-12


def _cdiv(a, b):
    return (a + b - 1) // b


class _LB:
    pass


class BertEngine:
    """Buffers and GEMM plans of one (B, S) shape; forward and backward of BertModel + the head."""

    def __init__(self, params: dict, n_layers: int, n_heads: int, d_ff: int, vocab: int, B: int, S: int, device,
                 grads: dict | None = None):
        assert E // n_heads == 64
        self.P, self.NL, self.H, self.FF, self.V = params, n_layers, n_heads, d_ff, vocab
        self.B, self.S = B, S
        self.Sp = _cdiv(S, 64) * 64
        self.M = B * S
        self.dev = device
        self.launches = 0
        f32, bf = torch.float32, torch.bfloat16
        M, H, Sp, FF = self.M, n_heads, self.Sp, d_ff
        buf = lambda shape, dt=f32: torch.empty(shape, dtype=dt, device=device)
        self.lens = torch.zeros(B, dtype=torch.int32, device=device)
        self.v0, self.x0, self.x0h = buf((M, E)), buf((M, E)), buf((M, E), bf)
        self.mean0, self.rstd0 = buf(M), buf(M)
        self.scores = buf((B, H, S, Sp))
        self.tmp = buf((M, E))
        self.layers = []
        for _ in range(n_layers):
            L = _LB()
            L.qkv, L.Pm, L.ctx = buf((M, 3 * E), bf), buf((B, H, S, Sp), bf), buf((M, E), bf)
            L.v1, L.x1, L.x1h, L.mean1, L.rstd1 = buf((M, E)), buf((M, E)), buf((M, E), bf), buf(M), buf(M)
            L.u, L.h = buf((M, FF), bf), buf((M, FF), bf)
            L.v2, L.x2, L.x2h, L.mean2, L.rstd2 = buf((M, E)), buf((M, E)), buf((M, E), bf), buf(M), buf(M)
            L.w_in, L.b_in = buf((3 * E, E), bf), buf(3 * E)
            L.w_o, L.w_1, L.w_2 = buf((E, E), bf), buf((FF, E), bf), buf((E, FF), bf)
            L.g_in, L.gb_in = torch.zeros((3 * E, E), dtype=f32, device=device), torch.zeros(3 * E, dtype=f32, device=device)
            self.layers.append(L)
        self.pooled, self.h1, self.lin = buf((B, E)), buf((B, 64)), buf((B, 49))
        # parameter gradients: the optimiser's flat arena when one is attached, engine-owned buffers otherwise
        self.G = {n: (grads[n] if grads is not None and n in grads else torch.zeros_like(p)) for n, p in params.items()}
        self._fwd_ready = self._bwd_ready = False
        self.p_hid, self.p_att, self.p_head, self.seed = 0.0, 0.0, 0.0, 0

    SITE_EMB, SITE_HEAD, SITE_LAYER0 = 96, 97, 100

    def set_dropout(self, p_hidden=0.0, p_attn=0.0, p_head=0.0, seed=0):
        """Dropout of the NEXT forward/backward pair (0 = off)."""
        self.p_hid, self.p_att, self.p_head = float(p_hidden), float(p_attn), float(p_head)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        if self.p_att > 0:
            for L in self.layers:
                if getattr(L, "Pu", None) is None:
                    L.Pu = torch.empty_like(L.Pm)

    @staticmethod
    def lp(l):
        return f"bert.encoder.layer.{l}."

    def _call(self, name, *a):
        _lib.call(name, *a)
        self.launches += 1

    def _run(self, plan):
        plan.run()
        self.launches += 1

    # ------------------------------------------------------------------ plans
    def _build_fwd(self):
        B, H, S, Sp, M, FF, P = self.B, self.H, self.S, self.Sp, self.M, self.FF, self.P
        for l, L in enumerate(self.layers):
            pre = self.lp(l)
            xin = self.x0h if l == 0 else self.layers[l - 1].x2h
            L.xin = xin
            L.p_qkv = G.plan_plain(M=M, N=3 * E, K=E, a_ptr=xin.data_ptr(), lda=E, a_mn=0, b_ptr=L.w_in.data_ptr(), ldb=E,
                                   b_mn=0, out=L.qkv, ldc=3 * E, bias=L.b_in, keep=(xin, L.w_in))
            q, k, v = L.qkv.data_ptr(), L.qkv.data_ptr() + E * 2, L.qkv.data_ptr() + 2 * E * 2
            hs, bs = 64, S * 3 * E
            L.p_scores = G.plan_plain(M=S, N=S, K=64, a_ptr=q, lda=3 * E, a_mn=0, b_ptr=k, ldb=3 * E, b_mn=0,
                                      out=self.scores, ldc=Sp, alpha=1.0 / 8.0, batch0=H, batch1=B, a_bs=(hs, bs),
                                      b_bs=(hs, bs), out_bs=(S * Sp, H * S * Sp), keep=(L.qkv,))
            L.p_pv = G.plan_plain(M=S, N=64, K=S, a_ptr=L.Pm.data_ptr(), lda=Sp, a_mn=0, b_ptr=v, ldb=3 * E, b_mn=1,
                                  out=L.ctx, ldc=E, batch0=H, batch1=B, a_bs=(S * Sp, H * S * Sp), b_bs=(hs, bs),
                                  out_bs=(64, S * E), keep=(L.Pm, L.qkv))
            L.p_o = G.plan_plain(M=M, N=E, K=E, a_ptr=L.ctx.data_ptr(), lda=E, a_mn=0, b_ptr=L.w_o.data_ptr(), ldb=E,
                                 b_mn=0, out=self.tmp, ldc=E, bias=P[pre + "attention.output.dense.bias"],
                                 keep=(L.ctx, L.w_o))
            L.p_ff1 = G.plan_plain(M=M, N=FF, K=E, a_ptr=L.x1h.data_ptr(), lda=E, a_mn=0, b_ptr=L.w_1.data_ptr(), ldb=E,
                                   b_mn=0, out=L.u, ldc=FF, bias=P[pre + "intermediate.dense.bias"], keep=(L.x1h, L.w_1))
            L.p_ff2 = G.plan_plain(M=M, N=E, K=FF, a_ptr=L.h.data_ptr(), lda=FF, a_mn=0, b_ptr=L.w_2.data_ptr(), ldb=FF,
                                   b_mn=0, out=self.tmp, ldc=E, bias=P[pre + "output.dense.bias"], keep=(L.h, L.w_2))
        self._fwd_ready = True

    def _build_bwd(self):
        B, H, S, Sp, M, FF = self.B, self.H, self.S, self.Sp, self.M, self.FF
        f32, bf, dev, Gd = torch.float32, torch.bfloat16, self.dev, self.G
        self.dx = torch.zeros((M, E), dtype=f32, device=dev)
        self.dva, self.dvb = torch.empty((M, E), dtype=f32, device=dev), torch.empty((M, E), dtype=f32, device=dev)
        self.dvh = torch.empty((M, E), dtype=bf, device=dev)
        self.dh, self.du = torch.empty((M, FF), dtype=bf, device=dev), torch.empty((M, FF), dtype=bf, device=dev)
        self.dbranch = torch.empty((M, E), dtype=f32, device=dev)
        self.dctx = torch.empty((M, E), dtype=bf, device=dev)
        self.dqkv = torch.empty((M, 3 * E), dtype=bf, device=dev)
        self.dS = torch.empty((B, H, S, Sp), dtype=bf, device=dev)
        self.dv0 = torch.empty((M, E), dtype=f32, device=dev)
        self.d_pooled, self.d_h1 = torch.empty((B, E), dtype=f32, device=dev), torch.empty((B, 64), dtype=f32, device=dev)
        sk = lambda gm, gn: max(1, min(_cdiv(M, 64), (2 * 148) // max(1, gm * gn)))
        for l, L in enumerate(self.layers):
            pre = self.lp(l)
            L.b_ff2_d = G.plan_plain(M=M, N=FF, K=E, a_ptr=self.dvh.data_ptr(), lda=E, a_mn=0, b_ptr=L.w_2.data_ptr(),
                                     ldb=FF, b_mn=1, out=self.dh, ldc=FF, keep=(self.dvh, L.w_2))
            L.b_ff2_w = G.plan_plain(M=E, N=FF, K=M, a_ptr=self.dvh.data_ptr(), lda=E, a_mn=1, b_ptr=L.h.data_ptr(),
                                     ldb=FF, b_mn=1, out=Gd[pre + "output.dense.weight"], ldc=FF, accumulate=2,
                                     split_k=sk(_cdiv(E, 128), _cdiv(FF, 256)), keep=(self.dvh, L.h))
            L.b_ff1_d = G.plan_plain(M=M, N=E, K=FF, a_ptr=self.du.data_ptr(), lda=FF, a_mn=0, b_ptr=L.w_1.data_ptr(),
                                     ldb=E, b_mn=1, out=self.dbranch, ldc=E, keep=(self.du, L.w_1))
            L.b_ff1_w = G.plan_plain(M=FF, N=E, K=M, a_ptr=self.du.data_ptr(), lda=FF, a_mn=1, b_ptr=L.x1h.data_ptr(),
                                     ldb=E, b_mn=1, out=Gd[pre + "intermediate.dense.weight"], ldc=E, accumulate=2,
                                     split_k=sk(_cdiv(FF, 128), _cdiv(E, 256)), keep=(self.du, L.x1h))
            L.b_o_d = G.plan_plain(M=M, N=E, K=E, a_ptr=self.dvh.data_ptr(), lda=E, a_mn=0, b_ptr=L.w_o.data_ptr(), ldb=E,
                                   b_mn=1, out=self.dctx, ldc=E, keep=(self.dvh, L.w_o))
            L.b_o_w = G.plan_plain(M=E, N=E, K=M, a_ptr=self.dvh.data_ptr(), lda=E, a_mn=1, b_ptr=L.ctx.data_ptr(), ldb=E,
                                   b_mn=1, out=Gd[pre + "attention.output.dense.weight"], ldc=E, accumulate=2,
                                   split_k=sk(_cdiv(E, 128), _cdiv(E, 256)), keep=(self.dvh, L.ctx))
            q, k, v = L.qkv.data_ptr(), L.qkv.data_ptr() + E * 2, L.qkv.data_ptr() + 2 * E * 2
            dq, dk, dv = self.dqkv.data_ptr(), self.dqkv.data_ptr() + E * 2, self.dqkv.data_ptr() + 2 * E * 2
            hs, bs, pbs = 64, S * 3 * E, (S * Sp, H * S * Sp)
            L.b_dp = G.plan_plain(M=S, N=S, K=64, a_ptr=self.dctx.data_ptr(), lda=E, a_mn=0, b_ptr=v, ldb=3 * E, b_mn=0,
                                  out=self.scores, ldc=Sp, batch0=H, batch1=B, a_bs=(64, S * E), b_bs=(hs, bs),
                                  out_bs=pbs, keep=(self.dctx, L.qkv))
            L.b_dv = G.plan_plain(M=S, N=64, K=S, a_ptr=L.Pm.data_ptr(), lda=Sp, a_mn=1, b_ptr=self.dctx.data_ptr(),
                                  ldb=E, b_mn=1, out=self.dqkv, out_ptr=dv, ldc=3 * E, batch0=H, batch1=B, a_bs=pbs,
                                  b_bs=(64, S * E), out_bs=(hs, bs), keep=(L.Pm, self.dctx))
            L.b_dq = G.plan_plain(M=S, N=64, K=S, a_ptr=self.dS.data_ptr(), lda=Sp, a_mn=0, b_ptr=k, ldb=3 * E, b_mn=1,
                                  out=self.dqkv, out_ptr=dq, ldc=3 * E, batch0=H, batch1=B, a_bs=pbs, b_bs=(hs, bs),
                                  out_bs=(hs, bs), keep=(self.dS, L.qkv))
            L.b_dk = G.plan_plain(M=S, N=64, K=S, a_ptr=self.dS.data_ptr(), lda=Sp, a_mn=1, b_ptr=q, ldb=3 * E, b_mn=1,
                                  out=self.dqkv, out_ptr=dk, ldc=3 * E, batch0=H, batch1=B, a_bs=pbs, b_bs=(hs, bs),
                                  out_bs=(hs, bs), keep=(self.dS, L.qkv))
            L.b_qkv_d = G.plan_plain(M=M, N=E, K=3 * E, a_ptr=self.dqkv.data_ptr(), lda=3 * E, a_mn=0,
                                     b_ptr=L.w_in.data_ptr(), ldb=E, b_mn=1, out=self.dbranch, ldc=E,
                                     keep=(self.dqkv, L.w_in))
            L.b_qkv_w = G.plan_plain(M=3 * E, N=E, K=M, a_ptr=self.dqkv.data_ptr(), lda=3 * E, a_mn=1,
                                     b_ptr=L.xin.data_ptr(), ldb=E, b_mn=1, out=L.g_in, ldc=E, accumulate=2,
                                     split_k=sk(_cdiv(3 * E, 128), _cdiv(E, 256)), keep=(self.dqkv, L.xin))
        self._bwd_ready = True

    # ---------------------------------------------------------------- forward
    def refresh_weights(self):
        ptr, P = _lib.ptr, self.P
        for l, L in enumerate(self.layers):
            pre = self.lp(l)
            for j, nm in enumerate(("query", "key", "value")):
                self._call("avdn_cast_f32_bf16", ptr(P[pre + f"attention.self.{nm}.weight"]),
                           L.w_in.data_ptr() + j * E * E * 2, E * E)
                L.b_in[j * E:(j + 1) * E].copy_(P[pre + f"attention.self.{nm}.bias"])
            for name, dst in ((pre + "attention.output.dense.weight", L.w_o), (pre + "intermediate.dense.weight", L.w_1),
                              (pre + "output.dense.weight", L.w_2)):
                self._call("avdn_cast_f32_bf16", ptr(P[name]), ptr(dst), dst.numel())

    def forward(self, ids, mask):
        """ids [B,S] int64, mask [B,S] (right-padded).  Returns (seq [B,S,768] fp32 view, lin [B,49], pooled [B,768])."""
        P, ptr = self.P, _lib.ptr
        B, S, M, H = self.B, self.S, self.M, self.H
        if not self._fwd_ready:
            self._build_fwd()
        self.ids = ids.contiguous()
        self.lens.copy_(mask.sum(dim=1).to(torch.int32))
        self.refresh_weights()
        e = "bert.embeddings."
        self._call("avdn_bert_embed_ln", ptr(self.ids), ptr(P[e + "word_embeddings.weight"]),
                   ptr(P[e + "position_embeddings.weight"]), ptr(P[e + "token_type_embeddings.weight"]),
                   ptr(P[e + "LayerNorm.weight"]), ptr(P[e + "LayerNorm.bias"]), B, S, self.V, LN_EPS, ptr(self.v0),
                   ptr(self.x0), ptr(self.x0h), ptr(self.mean0), ptr(self.rstd0))
        ph, pa, sd = self.p_hid, self.p_att, self.seed
        if ph > 0:
            self._call("avdn_dropout_f32", ptr(self.x0), ptr(self.x0h), self.x0.numel(), ph, sd, self.SITE_EMB)
        x = self.x0
        for l, L in enumerate(self.layers):
            pre = self.lp(l)
            st = self.SITE_LAYER0 + 3 * l
            self._run(L.p_qkv)
            self._run(L.p_scores)
            self._call("avdn_softmax_fwd_drop", ptr(self.scores), ptr(self.lens), B, H, S, 0, self.Sp, ptr(L.Pm),
                       ptr(L.Pu) if pa > 0 else None, pa, sd, st)
            self._run(L.p_pv)
            self._run(L.p_o)
            self._call("avdn_ln_fwd_drop", ptr(x), ptr(self.tmp), ptr(P[pre + "attention.output.LayerNorm.weight"]),
                       ptr(P[pre + "attention.output.LayerNorm.bias"]), M, E, LN_EPS, ptr(L.v1), ptr(L.x1), ptr(L.x1h),
                       ptr(L.mean1), ptr(L.rstd1), ph, sd, st + 1)
            self._run(L.p_ff1)
            self._call("avdn_gelu_fwd", ptr(L.u), ptr(L.h), L.u.numel())
            self._run(L.p_ff2)
            self._call("avdn_ln_fwd_drop", ptr(L.x1), ptr(self.tmp), ptr(P[pre + "output.LayerNorm.weight"]),
                       ptr(P[pre + "output.LayerNorm.bias"]), M, E, LN_EPS, ptr(L.v2), ptr(L.x2), ptr(L.x2h),
                       ptr(L.mean2), ptr(L.rstd2), ph, sd, st + 2)
            x = L.x2
        self.x_final = x
        lin = lambda xx, ldx, w, b, y, Mr, N, K, act: self._call("avdn_linear_f32", ptr(xx), ldx, ptr(w), K, ptr(b),
                                                                 ptr(y), N, Mr, N, K, act, 0)
        lin(x, S * E, P["bert.pooler.dense.weight"], P["bert.pooler.dense.bias"], self.pooled, B, E, E, 2)   # tanh(cls row)
        lin(self.pooled, E, P["linears.0.weight"], P["linears.0.bias"], self.h1, B, 64, E, 1)
        if self.p_head > 0:
            self._call("avdn_dropout_f32", ptr(self.h1), None, self.h1.numel(), self.p_head, sd, self.SITE_HEAD)
        lin(self.h1, 64, P["linears.3.weight"], P["linears.3.bias"], self.lin, B, 49, 64, 1)
        return x.view(B, S, E), self.lin, self.pooled

    # --------------------------------------------------------------- backward
    def zero_grads(self):
        for g in self.G.values():
            g.zero_()

    def backward(self, d_seq, d_lin, d_pooled):
        """Accumulates every parameter gradient into ``self.G``; inputs may be None (zero)."""
        P, Gd, ptr = self.P, self.G, _lib.ptr
        B, S, M, H, FF, Sp = self.B, self.S, self.M, self.H, self.FF, self.Sp
        if not self._bwd_ready:
            self._build_bwd()
        BF = 0
        if d_seq is None:
            self.dx.zero_()
        else:
            self.dx.copy_(d_seq.reshape(M, E))
        self.launches += 1
        # ---- heads: linears (agent-side linear_cls) and the pooler; d(cls row) is added into dx ----
        if d_pooled is None:
            self.d_pooled.zero_()
        else:
            self.d_pooled.copy_(d_pooled)
        if d_lin is not None:
            dl = d_lin.contiguous().float()
            self._call("avdn_linear_f32_bwd", ptr(self.h1), 64, ptr(P["linears.3.weight"]), ptr(self.lin), ptr(dl), B, 49,
                       64, 1, ptr(self.d_h1), 64, 0, ptr(Gd["linears.3.weight"]), ptr(Gd["linears.3.bias"]))
            if self.p_head > 0:          # through Dropout(0.2): the ReLU mask of the stored (dropped) h1 does the rest
                self._call("avdn_dropout_f32", ptr(self.d_h1), None, self.d_h1.numel(), self.p_head, self.seed,
                           self.SITE_HEAD)
            self._call("avdn_linear_f32_bwd", ptr(self.pooled), E, ptr(P["linears.0.weight"]), ptr(self.h1),
                       ptr(self.d_h1), B, 64, E, 1, ptr(self.d_pooled), E, 1, ptr(Gd["linears.0.weight"]),
                       ptr(Gd["linears.0.bias"]))
        self._call("avdn_linear_f32_bwd", ptr(self.x_final), S * E, ptr(P["bert.pooler.dense.weight"]), ptr(self.pooled),
                   ptr(self.d_pooled), B, E, E, 2, ptr(self.dx), S * E, 1, ptr(Gd["bert.pooler.dense.weight"]),
                   ptr(Gd["bert.pooler.dense.bias"]))
        ph, pa, sd = self.p_hid, self.p_att, self.seed
        dy1, dy2 = self.dx, None
        for l in reversed(range(self.NL)):
            L, pre = self.layers[l], self.lp(l)
            st = self.SITE_LAYER0 + 3 * l
            self._call("avdn_ln_bwd_drop", ptr(dy1), ptr(dy2), ptr(L.v2), ptr(L.mean2), ptr(L.rstd2),
                       ptr(P[pre + "output.LayerNorm.weight"]), M, E, ptr(self.dva), ptr(self.dvh),
                       ptr(Gd[pre + "output.LayerNorm.weight"]), ptr(Gd[pre + "output.LayerNorm.bias"]), ph, sd, st + 2)
            self._call("avdn_colsum", ptr(self.dvh), BF, M, E, E, ptr(Gd[pre + "output.dense.bias"]))
            self._run(L.b_ff2_w)
            self._run(L.b_ff2_d)
            self._call("avdn_gelu_bwd", ptr(L.u), ptr(self.dh), ptr(self.du), self.du.numel())
            self._call("avdn_colsum", ptr(self.du), BF, M, FF, FF, ptr(Gd[pre + "intermediate.dense.bias"]))
            self._run(L.b_ff1_w)
            self._run(L.b_ff1_d)
            self._call("avdn_ln_bwd_drop", ptr(self.dva), ptr(self.dbranch), ptr(L.v1), ptr(L.mean1), ptr(L.rstd1),
                       ptr(P[pre + "attention.output.LayerNorm.weight"]), M, E, ptr(self.dvb), ptr(self.dvh),
                       ptr(Gd[pre + "attention.output.LayerNorm.weight"]),
                       ptr(Gd[pre + "attention.output.LayerNorm.bias"]), ph, sd, st + 1)
            self._call("avdn_colsum", ptr(self.dvh), BF, M, E, E, ptr(Gd[pre + "attention.output.dense.bias"]))
            self._run(L.b_o_w)
            self._run(L.b_o_d)
            self._run(L.b_dp)
            self._run(L.b_dv)
            self._call("avdn_softmax_bwd_drop", ptr(L.Pu if pa > 0 else L.Pm), ptr(self.scores), B * H * S, S, Sp,
                       1.0 / 8.0, ptr(self.dS), pa, sd, st)
            self._run(L.b_dq)
            self._run(L.b_dk)
            L.g_in.zero_(); L.gb_in.zero_()
            self._call("avdn_colsum", ptr(self.dqkv), BF, M, 3 * E, 3 * E, ptr(L.gb_in))
            self._run(L.b_qkv_w)
            self._run(L.b_qkv_d)
            for j, nm in enumerate(("query", "key", "value")):
                Gd[pre + f"attention.self.{nm}.weight"].add_(L.g_in[j * E:(j + 1) * E])
                Gd[pre + f"attention.self.{nm}.bias"].add_(L.gb_in[j * E:(j + 1) * E])
            self.launches += 8
            dy1, dy2 = self.dvb, self.dbranch
        e = "bert.embeddings."
        if ph > 0:                       # through the embedding dropout: d(LN output) = dropout'(dy1 + dy2)
            self._call("avdn_add_dropout_f32", ptr(dy1), ptr(dy2), ptr(self.dva), self.dva.numel(), ph, sd, self.SITE_EMB)
            dy1, dy2 = self.dva, None
        self._call("avdn_ln_bwd", ptr(dy1), ptr(dy2), ptr(self.v0), ptr(self.mean0), ptr(self.rstd0),
                   ptr(P[e + "LayerNorm.weight"]), M, E, ptr(self.dv0), None, ptr(Gd[e + "LayerNorm.weight"]),
                   ptr(Gd[e + "LayerNorm.bias"]))
        self._call("avdn_bert_embed_bwd", ptr(self.ids), ptr(self.dv0), B, S, self.V, ptr(Gd[e + "word_embeddings.weight"]),
                   ptr(Gd[e + "position_embeddings.weight"]), ptr(Gd[e + "token_type_embeddings.weight"]))


class CustomBERTModel(nn.Module):
    def __init__(self, config=None, pretrained=None):
        """``pretrained``: a local directory for ``BertModel.from_pretrained`` (the reference downloads
        'bert-base-uncased', vln_model.py:131); default: random initialisation of the same architecture."""
        super().__init__()
        from transformers import BertConfig, BertModel
        if pretrained is not None:
            self.bert = BertModel.from_pretrained(pretrained)
        else:
            self.bert = BertModel(config if config is not None else BertConfig())
        cfg = self.bert.config
        if cfg.hidden_size != E or cfg.hidden_act != "gelu" or cfg.hidden_size // cfg.num_attention_heads != 64:
            raise NotImplementedError("only the bert-base geometry (768 wide, 64-wide heads, erf-GELU) is implemented")
        self.linears = nn.Sequential(nn.Linear(768, 64), nn.ReLU(), nn.Dropout(0.2), nn.Linear(64, 49), nn.ReLU())
        self._engines = {}
        self._pool = EnginePool(self._pool_engine)
        self._grad_arena = None          # name -> tensor, set by the optimiser arena (xview_et.agent.attach_lang_model)
        self._drop_step = 0

    def dropout_config(self):
        """(p_hidden, p_attention, p_head, seed) of the next forward: HF's and the head's dropout in train mode,
        zeros in eval mode; the seed advances every train-mode forward and derives from torch's global seed."""
        if not self.training:
            return 0.0, 0.0, 0.0, 0
        c = self.bert.config
        self._drop_step += 1
        seed = (torch.initial_seed() * 1000003 + 7919 * self._drop_step
                + 0x9E3779B97F4A7C15 * int(getattr(self, 'drop_rank', 0))) & 0xFFFFFFFFFFFFFFFF
        return float(c.hidden_dropout_prob), float(c.attention_probs_dropout_prob), float(self.linears[2].p), seed

    def used_parameters(self):
        return {n: p for n, p in self.named_parameters()}

    def engine(self, B, S, device, slot=0):
        """``slot`` separates engines of equal shape whose activations must coexist (the two passes of one rollout)."""
        key = (B, S, str(device), slot)
        e = self._engines.get(key)
        if e is None:
            c = self.bert.config
            e = BertEngine(self.used_parameters(), c.num_hidden_layers, c.num_attention_heads, c.intermediate_size,
                           c.vocab_size, B, S, device, grads=self._grad_arena)
            self._engines[key] = e
        return e

    def _pool_engine(self, key, slot):
        return self.engine(*key, slot=lease_slot(slot))

    def forward(self, ids, mask):
        _lib.require_cuda(ids, mask)
        B, S = ids.shape
        if S > self.bert.config.max_position_embeddings:
            raise ValueError("sequence longer than the position table")
        # with grad enabled the engine is held until this forward's backward (``_lease.EnginePool``)
        eng, lease = self._pool.acquire((B, S, ids.device), torch.is_grad_enabled())
        eng.set_dropout(*self.dropout_config())
        return _BertFn.apply(self, eng, lease, ids, mask, *self.used_parameters().values())


class _BertFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, eng, lease, ids, mask, *params):
        seq, lin, pooled = eng.forward(ids.long(), mask)
        ctx.mod, ctx.eng = mod, eng
        ctx.save_for_backward(lease)
        return seq.clone(), lin.clone(), pooled.clone()

    @staticmethod
    def backward(ctx, d_seq, d_lin, d_pooled):
        eng = ctx.eng
        eng.zero_grads()
        eng.backward(None if d_seq is None else d_seq.contiguous().float(), d_lin,
                     None if d_pooled is None else d_pooled.contiguous().float())
        return (None, None, None, None, None, *[eng.G[n].clone() for n in ctx.mod.used_parameters()])
