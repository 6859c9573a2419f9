"""``ET`` -- the HAA-Transformer of AVDN, mirror of src/models/ET_haa.py:77-184.

Same constructor (``ET(args)``), same sub-module names and therefore the same
``state_dict`` keys (including the unused ``dec_action.*`` and
``attention_layer_vision.c.*`` parameters, which receive no gradient in the
reference either), same ``forward(**inputs) -> (output, pred_saliency)``.

All arithmetic runs on libavdn kernels through ``_et_engine.ETEngine``:
tcgen05 GEMMs (bf16 operands, fp32 accumulation) for every dense contraction,
warp-level kernels for the frame attention, embeddings, LayerNorm, masked
softmax and the heads.  Precision: bf16 tensor-core path (north_star tolerance
1e-2 relative on logits and loss).
"""
import numpy as np
import torch
from torch import nn

from .. import _lib
from ._et_engine import ETEngine, ETDecodeState, E, NCH, NSP
from ._lease import EnginePool, lease_slot
from .enc_vl import EncoderVL


class SoftDotAttention(nn.Module):
    """Parameter container of src/models/ET_haa.py:30-74 (``c`` is unused there too)."""

    def __init__(self, dim):
        super().__init__()
        self.linear_in = nn.Linear(dim, dim, bias=False)
        self.sm = nn.Softmax(dim=1)
        self.linear_out = nn.Linear(dim * 2, dim, bias=False)
        self.tanh = nn.Tanh()
        self.c = nn.Sequential(nn.Linear(768, 256), nn.ReLU(), nn.Dropout(0.2), nn.Linear(256, 32), nn.ReLU(),
                               nn.Dropout(0.2), nn.Linear(32, 4), nn.ReLU())


class ET(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.encoder_vl = EncoderVL(args)
        self.dataset_enc = None
        self.args = args
        self.dec_action = nn.Linear(args.demb, args.demb)
        self.decoder_2_action_full = nn.Sequential(nn.Linear(768, 256), nn.ReLU(), nn.Dropout(0.2),
                                                   nn.Linear(256, 32), nn.ReLU(), nn.Dropout(0.2), nn.Linear(32, 4))
        self.attention_layer_vision = SoftDotAttention(49)
        self.fc = nn.Sequential(nn.Linear(768, 64), nn.Dropout(0.2), nn.ReLU())
        self.direction_embedding = nn.Linear(2, 768)
        self.fc2 = nn.Linear(49, 768)
        self.init_weights()
        self._engines = {}
        self._pool = EnginePool(self._pool_engine)
        self._grad_arena = None          # name -> tensor, set by the optimiser arena (xview_et.agent)

    def init_weights(self, init_range=0.1):
        self.dec_action.bias.data.zero_()
        self.dec_action.weight.data.uniform_(-init_range, init_range)

    # names of the parameters the forward pass uses (everything else has grad None in the reference)
    def used_parameters(self):
        skip = ("dec_action.", "attention_layer_vision.c.")
        return {n: p for n, p in self.named_parameters() if not n.startswith(skip)}

    def engine(self, B, L, T, device, slot=0):
        """``slot`` separates engines of equal shape whose activations must coexist (pending forwards)."""
        key = (B, L, T, str(device)) if slot == 0 else (B, L, T, str(device), slot)
        eng = self._engines.get(key)
        if eng is None:
            a = self.args
            eng = ETEngine(self.used_parameters(), a.encoder_heads, a.encoder_layers, a.demb, B, L, T, device,
                           grads=self._grad_arena)
            self._engines[key] = eng
        return eng

    def _pool_engine(self, key, slot):
        return self.engine(*key, slot=lease_slot(slot))

    def decoder(self, B, L, Tmax, device):
        """Incremental inference state of a greedy rollout (``_et_engine.ETDecodeState``)."""
        key = ("dec", B, L, Tmax, str(device))
        d = self._engines.get(key)
        if d is None:
            d = ETDecodeState(self.engine(B, L, 1, device), Tmax)
            self._engines[key] = d
        return d

    HEAD_DROPOUT = 0.2                   # nn.Dropout(0.2) of decoder_2_action_full / fc (ET_haa.py:98-119)

    def dropout_config(self):
        """(p_encoder, p_heads, seed) of the next forward: the reference's train-mode dropout
        (nn.TransformerEncoderLayer(dropout=dropout_transformer_encoder), Dropout(0.2) in the heads), zeros
        in eval mode.  The seed advances every train-mode forward and derives from torch's global seed."""
        if not self.training:
            return 0.0, 0.0, 0
        if float(getattr(self.args, "dropout_emb", 0.0)) != 0.0:
            raise NotImplementedError("dropout_emb > 0 (EncoderVL's embedding dropout) is not implemented")
        self._drop_step = getattr(self, "_drop_step", 0) + 1
        seed = (torch.initial_seed() * 1000003 + self._drop_step + 0x9E3779B97F4A7C15 * int(getattr(self, 'drop_rank', 0))) \
            & 0xFFFFFFFFFFFFFFFF
        return float(self.args.dropout_transformer_encoder), self.HEAD_DROPOUT, seed

    def forward_features(self, **inputs):
        """Like ``forward`` but returns ``(output [B,4], h_sali [B,64])`` -- the 8x8
        saliency map before the 224x224 upsample, which ``avdn_loss`` fuses."""
        frames, lang, lang_cls, dirs = inputs["frames"], inputs["lang"], inputs["lang_cls"], inputs["directions"]
        _lib.require_cuda(frames, lang, lang_cls, dirs)
        B, T = frames.shape[:2]
        L = lang.shape[1]
        if tuple(frames.shape[2:]) != (NCH, NSP):
            raise ValueError("frames must be [B,T,512,49] (src/xview_et/agent.py:594,615)")
        lenths = [int(x) for x in inputs["lenths"]]
        # with grad enabled the engine is held until this forward's backward (``_lease.EnginePool``)
        eng, lease = self._pool.acquire((B, L, T, frames.device), torch.is_grad_enabled())
        eng.set_dropout(*self.dropout_config())
        return _ETFn.apply(self, eng, lease, lenths, frames, lang, lang_cls, dirs, *self.used_parameters().values())

    def forward(self, **inputs):
        """src/models/ET_haa.py:121-184: keys ``directions [B,T,2]``, ``frames [B,T,512,49]``,
        ``lenths list[int]``, ``lang [B,L,768]``, ``lang_cls [B,49]`` ->
        ``(output [B,4], pred_saliency [B,1,224,224])``."""
        output, h_sali = self.forward_features(**inputs)
        return output, _UpsampleFn.apply(h_sali)


class _ETFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, eng, lease, lenths, frames, lang, lang_cls, dirs, *params):
        f = frames.detach().contiguous().float().view(-1, NCH, NSP)
        lg = lang.detach().contiguous().float()
        lc = lang_cls.detach().contiguous().float()
        dr = dirs.detach().contiguous().float()
        output, h_sali = eng.forward(f, lg, lc, dr, lenths, mod.encoder_vl.enc_pos.pe[0])
        ctx.mod, ctx.eng = mod, eng
        ctx.save_for_backward(lease)
        ctx.frames_shape = frames.shape
        ctx.need_lang = lang.requires_grad
        ctx.need_cls = lang_cls.requires_grad
        ctx.need_frames = frames.requires_grad
        return output.clone(), h_sali.clone()

    @staticmethod
    def backward(ctx, d_output, d_h_sali):
        mod, eng = ctx.mod, ctx.eng
        own = mod._grad_arena is None
        if own:
            eng.zero_grads()
        d_output = torch.zeros_like(eng.output) if d_output is None else d_output.contiguous().float()
        d_h_sali = torch.zeros_like(eng.h_sali) if d_h_sali is None else d_h_sali.contiguous().float()
        d_cls = torch.zeros((eng.B, NSP), dtype=torch.float32, device=eng.dev) if ctx.need_cls else None
        d_frames, d_lang = eng.backward(d_output, d_h_sali, need_lang_grad=ctx.need_lang, d_lang_cls=d_cls)
        if own:
            grads = [eng.G[n].clone() for n in mod.used_parameters()]
        else:                            # gradients were accumulated straight into the optimiser arena
            grads = [None] * len(mod.used_parameters())
        return (None, None, None, None, d_frames.view(ctx.frames_shape) if ctx.need_frames else None, d_lang, d_cls, None,
                *grads)


class _UpsampleFn(torch.autograd.Function):
    """F.interpolate(h_sali.view(-1,1,8,8), (224,224), bilinear, align_corners=False) (ET_haa.py:166-167)."""

    @staticmethod
    def forward(ctx, h_sali):
        B = h_sali.shape[0]
        h = h_sali.detach().contiguous()
        pred = torch.empty((B, 1, 224, 224), dtype=torch.float32, device=h.device)
        _lib.call("avdn_upsample_saliency", _lib.ptr(h), B, _lib.ptr(pred))
        return pred

    @staticmethod
    def backward(ctx, d_pred):
        B = d_pred.shape[0]
        g = d_pred.contiguous().float()
        dh = torch.empty((B, 64), dtype=torch.float32, device=g.device)
        _lib.call("avdn_upsample_saliency_bwd", _lib.ptr(g), B, _lib.ptr(dh))
        return dh
