"""``EncoderVL`` -- mirror of src/models/enc_vl.py:8-83 (same constructor, same
sub-module names so ``state_dict`` keys match).  The sub-modules are parameter
containers; the arithmetic runs in ``_et_engine.ETEngine`` on libavdn kernels."""
import numpy as np
import torch
from torch import nn

from .. import _lib
from . import model_util
from ._et_engine import ETEngine, E
from ._lease import EnginePool, lease_slot
from .encodings import PosEncoding


class EncoderVL(nn.Module):
    def __init__(self, args):
        super().__init__()
        if args.demb != E:
            raise NotImplementedError("the AVDN transformer is 768-wide (ET_haa.py:98-119 hard-codes it)")
        encoder_layer = nn.TransformerEncoderLayer(args.demb, args.encoder_heads, args.demb,
                                                   args.dropout_transformer_encoder)
        self.enc_transformer = nn.TransformerEncoder(encoder_layer, args.encoder_layers, enable_nested_tensor=False)
        self.num_input_actions = args.num_input_actions
        self.enc_pos = PosEncoding(args.demb)
        self.enc_pos_learn = None
        self.enc_token = None
        self.enc_layernorm = nn.LayerNorm(args.demb)
        self.enc_dropout = nn.Dropout(args.dropout_emb, inplace=True)
        self.n_heads, self.n_layers, self.d_ff = args.encoder_heads, args.encoder_layers, args.demb
        self._engines = {}
        self._pool = EnginePool(self._pool_engine)

    def _pool_engine(self, key, slot):
        B, L, T, device = key
        key = (B, L, T, str(device)) if slot == 0 else (B, L, T, str(device), lease_slot(slot))
        eng = self._engines.get(key)
        if eng is None:
            params = {"encoder_vl." + n: p for n, p in self.named_parameters()}
            eng = ETEngine(params, self.n_heads, self.n_layers, self.d_ff, B, L, T, device,
                           with_frame_attn=False, with_heads=False)
            self._engines[key] = eng
        return eng

    def _dropout_config(self):
        """Train mode: nn.TransformerEncoderLayer's dropout p at its four sites (stateless hash masks,
        ``ETEngine.set_dropout``); the embedding dropout (dropout_emb, 0 in the reference's configs) is not
        implemented."""
        if not self.training:
            return 0.0, 0.0, 0
        if self.enc_dropout.p > 0:
            raise NotImplementedError("dropout_emb > 0 (EncoderVL's embedding dropout) is not implemented")
        self._drop_step = getattr(self, "_drop_step", 0) + 1
        seed = (torch.initial_seed() * 1000003 + self._drop_step) & 0xFFFFFFFFFFFFFFFF
        return float(self.enc_transformer.layers[0].dropout.p), 0.0, seed

    def forward(self, emb_lang, emb_frames, emb_directions, lengths):
        """enc_vl.py:34-69 -> (output [B,S,768], mask_pad [B,S] bool)."""
        _lib.require_cuda(emb_lang, emb_frames, emb_directions)
        B, L, _ = emb_lang.shape
        T = emb_frames.shape[1]
        # with grad enabled the engine is held until this forward's backward (``_lease.EnginePool``)
        eng, lease = self._pool.acquire((B, L, T, emb_lang.device), torch.is_grad_enabled())
        eng.set_dropout(*self._dropout_config())
        out = _EncoderFn.apply(self, eng, lease, list(lengths), emb_lang, emb_frames, emb_directions,
                               *[p for _, p in self.named_parameters()])
        return out, model_util.generate_pad_mask(lengths, L, emb_lang.device)


class _EncoderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, eng, lease, lengths, lang, frames, dirs, *params):
        eng.set_lengths(lengths)
        lang, frames, dirs = (t.detach().contiguous().float() for t in (lang, frames, dirs))
        x = eng.encode(lang, frames, dirs, True, mod.enc_pos.pe[0])
        ctx.mod, ctx.eng = mod, eng
        ctx.save_for_backward(lease)
        return x.view(eng.B, eng.S, E).clone()

    @staticmethod
    def backward(ctx, d_out):
        mod, eng = ctx.mod, ctx.eng
        eng.zero_grads()
        if not eng._bwd_ready:
            eng._build_bwd_plans_safe()
        dv0 = eng.backward_encoder(d_out.contiguous().float()).view(eng.B, eng.S, E)
        L, T = eng.L, eng.T
        grads = [eng.G["encoder_vl." + n].clone() for n, _ in mod.named_parameters()]
        return (None, None, None, None, dv0[:, :L].clone(), dv0[:, L:L + T].clone(), dv0[:, L + T:].clone(), *grads)
