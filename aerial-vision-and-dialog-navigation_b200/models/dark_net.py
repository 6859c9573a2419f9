"""B200-native ``Darknet`` trunk — host-side mirror of the reference class
(``/root/reference/src/models/dark_net.py``): same constructor, same cfg format,
same ``state_dict`` keys (``module_list.{i}.conv_{i}.weight``,
``module_list.{i}.batch_norm_{i}.{weight,bias,running_mean,running_var,num_batches_tracked}``),
``forward`` returns the last layer's output ``[N, C, H/32, W/32]`` float32.

Device work: every 3x3 / 1x1 convolution (forward, dgrad, wgrad) is the tcgen05
implicit-GEMM kernel (``avdn_gemm_*``); BatchNorm(train) + LeakyReLU(0.01) +
shortcut add and their backward are the fused elementwise kernels of
``csrc/trunk.cu``.  Activations live in NHWC bf16 with channels padded to 64.
The nn.Conv2d / nn.BatchNorm2d sub-modules are parameter containers only (so
that reference checkpoints load); their ``forward`` is never called.

Scope: the layer types the truncated xview-yolov3 trunk contains
(``convolutional`` with batch_normalize=1 + leaky, ``shortcut``).  ``route``,
``upsample`` and ``yolo`` blocks are outside the hot path (SURVEY.md §2 #4) and
raise ``NotImplementedError``.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from .. import _lib
from .. import gemm as G
from ._lease import EnginePool, lease_slot

LEAKY_SLOPE = 0.01      # nn.LeakyReLU() default, dark_net.py:33
# AVDN_FUSE_BNB=1: BatchNorm-backward reductions fused into the epilogue of the data-gradient convolution that
# produces dA (avdn_gemm_core.bnb_*) instead of the separate reduction pass over (z, dA).  Off by default: measured
# on a B200 the separate pass reads dA out of L2 right after the dgrad wrote it and runs at > 6 TB/s, while the
# fused epilogue (four single-issue warps per CTA) makes the memory-bound 1x1 / stride-2 dgrads 1.7-2.5x slower
# and the tensor-bound 3x3 ones ~10 % slower -- net +3 ms per step (DESIGN.md, "measured and not kept").
FUSE_BNB = os.environ.get("AVDN_FUSE_BNB", "0") == "1"
# Block 0 in train mode: recompute path (avdn_conv0_fwd_stats / _fwd_apply / _bwd) -- its pre-activation z and its
# gradient dz (2 GB each at 640 views) are never stored.  AVDN_CONV0_RECOMPUTE=0 keeps the stored-z path.
CONV0_RECOMPUTE = os.environ.get("AVDN_CONV0_RECOMPUTE", "1") != "0"
# Thin 3x3 stride-1 blocks (32 -> 64 channels: module_list.3 at 112 x 112) run their forward and data gradient on the
# halo-tile kernel (csrc/conv3_halo.cu: three TMA boxes per tile instead of nine, resident filters) where it applies.
CONV_HALO = os.environ.get("AVDN_CONV_HALO", "1") != "0"
BN_EPS = 1e-5
BN_MOMENTUM = 0.1


def parse_model_config(path):
    """Same cfg grammar as the reference parser (dark_net.py:243-261): ``[type]``
    headers, ``key=value`` lines, ``#`` comments; conv blocks default
    ``batch_normalize`` to 0."""
    defs = []
    with open(path, "r") as f:
        for raw in f.read().split("\n"):
            line = raw.strip()
            if not line or line.startswith("#"):
                continue
            if line.startswith("["):
                d = {"type": line[1:-1].rstrip()}
                if d["type"] == "convolutional":
                    d["batch_normalize"] = 0
                defs.append(d)
            else:
                k, v = line.split("=")
                defs[-1][k.rstrip()] = v.strip()
    return defs


def _pad64(c):
    """Stored channel count: multiples of 64 (one 128-byte k-block), except that 32-channel tensors
    (trunk blocks 0 and 2) are stored as they are -- half the HBM traffic of a padded copy."""
    return 32 if c == 32 else (c + 63) // 64 * 64


class EmptyLayer(nn.Module):
    """Placeholder for 'shortcut' blocks (keeps module indices aligned with the cfg)."""


def create_modules(module_defs):
    hyper = module_defs.pop(0)
    filters_out = [int(hyper["channels"])]
    mods = nn.ModuleList()
    for i, d in enumerate(module_defs):
        seq = nn.Sequential()
        if d["type"] == "convolutional":
            bn = int(d["batch_normalize"])
            filters = int(d["filters"])
            k = int(d["size"])
            pad = (k - 1) // 2 if int(d["pad"]) else 0
            seq.add_module("conv_%d" % i, nn.Conv2d(filters_out[-1], filters, k, int(d["stride"]), pad, bias=not bn))
            if bn:
                seq.add_module("batch_norm_%d" % i, nn.BatchNorm2d(filters))
            if d["activation"] == "leaky":
                seq.add_module("leaky_%d" % i, nn.LeakyReLU())
        elif d["type"] == "shortcut":
            filters = filters_out[int(d["from"])]
            seq.add_module("shortcut_%d" % i, EmptyLayer())
        else:
            raise NotImplementedError(f"darknet block '{d['type']}' is outside the AVDN hot path")
        mods.append(seq)
        filters_out.append(filters)
    return hyper, mods


class _Layer:
    """Static description + device buffers of one convolutional block."""
    pass


class _Engine:
    """Per-batch-size execution state: activation / gradient buffers and GEMM plans."""

    def __init__(self, net: "Darknet", N: int, H: int, W: int, device):
        self.N, self.H, self.W, self.device = N, H, W, device
        import weakref
        self.net_ref = weakref.ref(net)
        bf, f32 = torch.bfloat16, torch.float32
        dev = device
        self.layers = []
        defs = net.module_defs
        out_of = {}                    # module index -> layer object producing that output
        cur = dict(C=3, Cp=4, H=H, W=W, layer=None)
        shapes = {}                    # module index -> (C, H, W)
        max_elems = 0
        for i, d in enumerate(defs):
            if d["type"] == "convolutional":
                conv = net.module_list[i][0]
                if int(d["batch_normalize"]) != 1 or d["activation"] != "leaky":
                    raise NotImplementedError("only conv+BN+leaky blocks are on the hot path")
                k, s = conv.kernel_size[0], conv.stride[0]
                if k not in (1, 3) or s not in (1, 2) or (k == 1 and s != 1) or conv.padding[0] != (k - 1) // 2:
                    raise NotImplementedError(f"conv k={k} s={s} pad={conv.padding[0]} is not supported")
                L = _Layer()
                L.idx, L.k, L.s = i, k, s
                L.Cin, L.Cout = conv.in_channels, conv.out_channels
                L.Cin_p = 4 if len(self.layers) == 0 else _pad64(L.Cin)
                L.Cout_p = _pad64(L.Cout)
                L.Hin, L.Win = cur["H"], cur["W"]
                L.Hout, L.Wout = L.Hin // s, L.Win // s
                L.src = cur["layer"]           # producing layer of the input (None = image)
                L.res = None                   # residual source layer (fused shortcut)
                L.first = len(self.layers) == 0
                L.halo = L.halo_dgrad = L.halo_wgrad = False
                if L.first and not (L.Cin == 3 and L.Cout == 32 and k == 3 and s == 1):
                    raise NotImplementedError("first layer must be the 3->32 3x3 stride-1 conv of yolov3")
                L.R = N * L.Hout * L.Wout
                L.flops = 2 * L.R * L.Cout * L.Cin * k * k          # algorithmic (un-padded) FLOPs
                self.layers.append(L)
                out_of[i] = L
                shapes[i] = (L.Cout, L.Hout, L.Wout)
                cur = dict(C=L.Cout, Cp=L.Cout_p, H=L.Hout, W=L.Wout, layer=L)
            elif d["type"] == "shortcut":
                frm = i + int(d["from"]) if int(d["from"]) < 0 else int(d["from"])
                prev = out_of.get(i - 1)
                srcl = out_of.get(frm)
                if prev is None or srcl is None or prev.idx != i - 1 or prev.res is not None:
                    raise NotImplementedError("shortcut must directly follow a convolutional block")
                if shapes[frm] != shapes[i - 1]:
                    raise ValueError("shortcut operands differ in shape")
                prev.res = srcl                # fuse: out[i] = leaky(bn(conv)) + out[frm]
                out_of[i] = prev
                shapes[i] = shapes[i - 1]
        self.last = self.layers[-1]
        # ---- buffers ----
        for L in self.layers:
            n_el = L.R * L.Cout_p
            if not (L.first and CONV0_RECOMPUTE):              # the recompute path of block 0 forms no dz
                max_elems = max(max_elems, n_el)
            L.recompute = bool(L.first and CONV0_RECOMPUTE)
            L.z = None if L.recompute else torch.empty((N, L.Hout, L.Wout, L.Cout_p), dtype=bf, device=dev)
            L.a = torch.empty((N, L.Hout, L.Wout, L.Cout_p), dtype=bf, device=dev)
            if L.recompute:
                L.zw = torch.zeros(L.Cout * 27, dtype=f32, device=dev)         # sum z * x  (forward pass 1)
                L.gw = torch.zeros(L.Cout * 27, dtype=f32, device=dev)         # sum g * x  (backward)
                L.xs9 = torch.zeros(36, dtype=torch.float64, device=dev)       # patch sums (tcgen05) / border sums of x
                L.mask = torch.zeros(L.R, dtype=torch.int32, device=dev)       # sign bits of a, one word per pixel
            L.scale = torch.zeros(L.Cout_p, dtype=f32, device=dev)
            L.shift = torch.zeros(L.Cout_p, dtype=f32, device=dev)
            L.mean = torch.zeros(L.Cout_p, dtype=f32, device=dev)
            L.rstd = torch.zeros(L.Cout_p, dtype=f32, device=dev)
            L.sums = torch.zeros(4 * L.Cout_p, dtype=torch.float64, device=dev)
            if not L.first:
                L.wf = torch.empty((L.Cout_p, L.k * L.k * L.Cin_p), dtype=bf, device=dev)
                L.wd = torch.empty((L.Cin_p, L.k * L.k * L.Cout_p), dtype=bf, device=dev)
            L.g = None                 # gradient buffer of L.a (allocated on first backward)
        self.x_in = None
        self.dz = None
        self._max_elems = max_elems
        self._fwd_plans = False
        self._eval_plans = False
        self._bwd_plans = False
        self.launches = 0

    # plans bake device pointers, so they are created once the buffers exist
    def build_fwd(self, x_nhwc4):
        if self._fwd_plans and self.x_in is x_nhwc4:
            return
        self.x_in = x_nhwc4
        if not self._fwd_plans:
            for L in self.layers:
                if L.first:
                    continue
                # two plans: train mode accumulates the BatchNorm batch statistics in the epilogue
                L.p_fwd = G.plan_conv_fwd(L.src.a, L.wf, L.z, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                          Cout=L.Cout_p, k=L.k, stride=L.s, flops=L.flops)
                L.p_fwd_stats = G.plan_conv_fwd(L.src.a, L.wf, L.z, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                                Cout=L.Cout_p, k=L.k, stride=L.s, flops=L.flops, stats=L.sums)
                L.halo = bool(CONV_HALO and L.k == 3 and L.s == 1 and
                              _lib.lib().avdn_conv3x3_thin_supported(L.Hin, L.Win, L.Cin_p, L.Cout_p))
            self._fwd_plans = True

    def conv_table(self, net):
        """Device array of ``avdn_conv_item`` (one per tcgen05 conv block, layer order) for the one-launch
        weight packing / gradient unpacking; rebuilt when a pointer changes (e.g. ``net.to()``)."""
        import ctypes as C
        import numpy as np
        tc = [L for L in self.layers if not L.first]
        sig = tuple((net.module_list[L.idx][0].weight.data_ptr(),
                     0 if getattr(L, "dwf", None) is None else L.dwf.data_ptr(),
                     0 if getattr(L, "dw", None) is None else L.dw.data_ptr()) for L in tc)
        if getattr(self, "_table_sig", None) != sig:
            arr = (_lib.ConvItem * len(tc))()
            for i, L in enumerate(tc):
                it = arr[i]
                it.w = net.module_list[L.idx][0].weight.data_ptr()
                it.wf, it.wd = L.wf.data_ptr(), L.wd.data_ptr()
                it.dwf, it.grad = sig[i][1] or None, sig[i][2] or None
                if getattr(L, "halo_wgrad", False):
                    it.dwf = None           # its weight gradient goes straight into grad (avdn_conv3x3_thin_wgrad)
                it.Cout, it.Cin, it.k, it.stride = L.Cout, L.Cin, L.k, L.s
                it.Cout_p, it.Cin_p = L.Cout_p, L.Cin_p
                it.pairs = 1 if getattr(L, "pairs", False) else 0
            raw = np.frombuffer(bytes(arr), dtype=np.uint8).copy()
            self._table = torch.from_numpy(raw).to(self.device)
            self._table_sig = sig
            self._table_n = len(tc)
        return self._table

    def build_fwd_eval(self):
        """Eval mode: the BN affine is known before the convolution runs, so BatchNorm + LeakyReLU +
        the shortcut add are the convolution's epilogue (no z round trip, no elementwise pass)."""
        if self._eval_plans:
            return
        for L in self.layers:
            if L.first:
                continue
            L.p_fwd_eval = G.plan_conv_fwd(L.src.a, L.wf, L.a, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                           Cout=L.Cout_p, k=L.k, stride=L.s, flops=L.flops,
                                           affine=(L.scale, L.shift, LEAKY_SLOPE),
                                           residual=L.res.a if L.res is not None else None)
        self._eval_plans = True

    def build_bwd(self, net=None):
        if self._bwd_plans:
            return
        arena = getattr(net, "_grad_arena", None) if net is not None else None
        bf, f32, dev = torch.bfloat16, torch.float32, self.device
        self.dz = torch.empty(self._max_elems, dtype=bf, device=dev)
        # gradient buffers: a fused-shortcut output shares its buffer with the residual source
        for L in reversed(self.layers):
            if L.g is None:
                L.g = torch.empty((self.N, L.Hout, L.Wout, L.Cout_p), dtype=bf, device=dev)
            if L.res is not None:
                assert L.res.g is None
                L.res.g = L.g
        # WGRAD outputs (fp32, split-K reduce-add targets) live in one arena: zeroed with one memset per step
        def dwf_shape(L):
            if L.Cin_p == 32 or L.Cout_p == 32:
                nblk = 6 if L.s == 2 else L.k * (3 if L.k == 3 else 1)
                return (L.Cout_p if L.s == 2 else 2 * L.Cout_p, nblk * 2 * L.Cin_p)
            return (L.Cout_p, L.k * L.k * L.Cin_p)
        tot = sum((dwf_shape(L)[0] * dwf_shape(L)[1] + 63) // 64 * 64 for L in self.layers if not L.first)
        # the fused BatchNorm-backward sums ([2, Cout_p] f64 per block) live behind the WGRAD outputs: the one
        # memset per step clears both
        n_bs = sum(4 * L.Cout_p for L in self.layers)
        self.dwf_arena = torch.zeros(tot + n_bs, dtype=f32, device=dev)
        bs_off = tot
        # the data gradient of a block's output is final once its FIRST consumer (in forward order) has run its
        # dgrad: that launch can reduce the BatchNorm-backward sums of the producing block in its epilogue
        first_consumer = {}
        for L in self.layers:
            for P in (L.src, L.res):
                if P is not None:
                    first_consumer[id(P)] = min(first_consumer.get(id(P), L.idx), L.idx)
        for L in self.layers:
            L.coef = L.sums[2 * L.Cout_p:].view(f32)               # [4, Cout_p] fp32 scratch of the backward apply
            L.bsums = self.dwf_arena[bs_off: bs_off + 4 * L.Cout_p].view(torch.float64)
            bs_off += 4 * L.Cout_p
            L.bnb_fused = False
            L.bnb_ready = False
        dwf_off = 0
        seen_as_input = set()
        for L in reversed(self.layers):
            dz = None if L.recompute else self.dz[: L.R * L.Cout_p].view(self.N, L.Hout, L.Wout, L.Cout_p)
            L.dz = dz
            if arena is not None:
                i = L.idx
                L.dgamma = arena[f"module_list.{i}.batch_norm_{i}.weight"]
                L.dbeta = arena[f"module_list.{i}.batch_norm_{i}.bias"]
                L.dw = arena[f"module_list.{i}.conv_{i}.weight"]
            else:
                L.dgamma = torch.zeros(L.Cout, dtype=f32, device=dev)
                L.dbeta = torch.zeros(L.Cout, dtype=f32, device=dev)
                L.dw = torch.zeros((L.Cout, L.Cin, L.k, L.k), dtype=f32, device=dev)
            if L.first:
                continue
            L.pairs = (L.Cin_p == 32 or L.Cout_p == 32)      # 32-channel operand: pixel-pair wgrad
            shp = dwf_shape(L)
            L.dwf = self.dwf_arena[dwf_off: dwf_off + shp[0] * shp[1]].view(shp)
            dwf_off += (shp[0] * shp[1] + 63) // 64 * 64
            if L.pairs:
                L.p_wgrad = G.plan_conv_wgrad_pairs(dz, L.src.a, L.dwf, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                                    Cout=L.Cout_p, k=L.k, stride=L.s, flops=L.flops)
            else:
                L.p_wgrad = G.plan_conv_wgrad(dz, L.src.a, L.dwf, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                              Cout=L.Cout_p, k=L.k, stride=L.s, flops=L.flops)
            # the input's gradient buffer already holds the skip gradient iff the input is a
            # residual source whose consumer (a later fused shortcut) was processed before
            acc = 1 if id(L.src) in seen_as_input else 0
            P = L.src
            bnb = None
            if FUSE_BNB and P.z is not None and first_consumer[id(P)] == L.idx and G.pick_bn(L.Cin_p) <= 128:
                bnb = (P.z, P.scale, P.shift, P.mean, P.bsums, LEAKY_SLOPE)
                P.bnb_fused = True
            L.p_dgrad = G.plan_conv_dgrad(dz, L.wd, L.src.g, N=self.N, H=L.Hin, W=L.Win, Cin=L.Cin_p,
                                          Cout=L.Cout_p, k=L.k, stride=L.s, accumulate=acc, flops=L.flops, bnb=bnb)
            L.halo_dgrad = bool(getattr(L, "halo", False) and acc == 0 and bnb is None)     # overwrite only
            L.halo_wgrad = bool(getattr(L, "halo", False))
            seen_as_input.add(id(L.src))
            if L.res is not None:
                seen_as_input.add(id(L.res))
        self._bwd_plans = True


def _trunk_forward(net, eng, x_nhwc4, train, out=None, frozen=False):
    """Forward of every block on libavdn kernels.  Returns ``[N, C_last, h, w]`` fp32.
    ``frozen`` (eval mode only): the parameters and running statistics have not changed since
    the previous call on this engine, so the bf16 weight operands and the BN affine
    coefficients are reused (the rollout of config 5 runs 20 trunk passes on fixed weights)."""
    call = _lib.call
    ptr = _lib.ptr
    eng.build_fwd(x_nhwc4)
    n = 0
    reuse = frozen and not train and getattr(eng, "_frozen_ready", False)
    eng._frozen_ready = (not train)
    if not train:
        eng.build_fwd_eval()
    if not reuse:
        # fp32 master weights -> bf16 GEMM operands (wf, wd) of every block, one launch
        tbl = eng.conv_table(net)
        call("avdn_pack_conv_weights", ptr(tbl), eng._table_n)
        n += 1
    for li, L in enumerate(eng.layers):
        conv = net.module_list[L.idx][0]
        bn = net.module_list[L.idx][1]
        if not train:
            # eval: affine from the running statistics first, then conv with the fused epilogue
            if not reuse:
                call("avdn_bn_eval_coeffs", L.Cout_p, L.Cout, ptr(bn.weight), ptr(bn.bias), ptr(bn.running_mean),
                     ptr(bn.running_var), BN_EPS, ptr(L.scale), ptr(L.shift))
                n += 1
            if L.first:
                call("avdn_conv0_fwd_eval", ptr(x_nhwc4), ptr(conv.weight), ptr(L.scale), ptr(L.shift), LEAKY_SLOPE,
                     ptr(L.a), eng.N, L.Hin, L.Win)
                n += 1
            else:
                L.p_fwd_eval.run()
                n += 1
            continue
        if L.first and L.recompute:
            # pass 1: batch statistics (+ the z-weighted input sums the backward needs); pass 2 below recomputes z
            call("avdn_conv0_fwd_stats", ptr(x_nhwc4), ptr(conv.weight), eng.N, L.Hin, L.Win, ptr(L.sums), ptr(L.zw),
                 ptr(L.xs9))
            n += 2                  # kernels only (memsets / symbol copies inside the ABI calls are not counted)
        elif L.first:
            call("avdn_conv0_fwd", ptr(x_nhwc4), ptr(conv.weight), ptr(L.z), eng.N, L.Hin, L.Win, ptr(L.sums))
            n += 1
        elif L.halo:
            call("avdn_conv3x3_thin_fwd", ptr(L.src.a), ptr(L.wf), ptr(L.z), eng.N, L.Hin, L.Win, L.Cin_p, L.Cout_p,
                 ptr(L.sums), flops=L.flops)
            n += 1
        else:
            L.p_fwd_stats.run()
            n += 1
        call("avdn_bn_finalize", ptr(L.sums), L.R, L.Cout_p, L.Cout, ptr(bn.weight), ptr(bn.bias),
             ptr(bn.running_mean), ptr(bn.running_var), BN_MOMENTUM, BN_EPS, ptr(L.scale),
             ptr(L.shift), ptr(L.mean), ptr(L.rstd))
        n += 1                      # finalize
        if L.first and L.recompute:
            call("avdn_conv0_fwd_apply", ptr(x_nhwc4), ptr(conv.weight), ptr(L.scale), ptr(L.shift), LEAKY_SLOPE,
                 ptr(L.a), ptr(L.mask), eng.N, L.Hin, L.Win)
        else:
            call("avdn_bn_apply", ptr(L.z), ptr(L.scale), ptr(L.shift), ptr(L.res.a) if L.res is not None else None,
                 ptr(L.a), L.R, L.Cout_p, LEAKY_SLOPE)
        n += 1
    if train:
        net._bump_batches_tracked()
    last = eng.last
    if out is None:
        out = torch.empty((eng.N, last.Cout, last.Hout, last.Wout), dtype=torch.float32, device=eng.device)
    call("avdn_nhwc_to_nchw_f32", ptr(last.a), ptr(out), eng.N, last.Hout * last.Wout, last.Cout_p)
    eng.launches += n + 1
    return out


def _trunk_forward_graphed(net, eng, x_nhwc4, out):
    """Eval-mode forward on frozen weights replayed from a CUDA graph (the rollouts run 19 of their 20 trunk
    passes on unchanged weights and fixed buffers; at rollout batch sizes the 58 launches of a pass are short
    enough for launch latency to show).  The first call for a (input, output) buffer pair captures
    ``_trunk_forward(frozen=True)``; the caller must have run one un-graphed pass since the weights last changed."""
    if _lib.PROFILE is not None:                  # per-kernel instrumentation needs real launches
        return _trunk_forward(net, eng, x_nhwc4, False, out=out, frozen=True)
    graphs = eng.__dict__.setdefault("_graphs", {})
    key = (x_nhwc4.data_ptr(), out.data_ptr())
    g = graphs.get(key)
    if g is None:
        assert getattr(eng, "_frozen_ready", False), "run one eval pass before graph capture"
        l0 = eng.launches
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            _trunk_forward(net, eng, x_nhwc4, False, out=out, frozen=True)
        graphs[key] = (g, eng.launches - l0)
        g = graphs[key]
    g[0].replay()
    eng.launches += g[1]
    return out


def _layer_backward(eng, L, unpack=True, zero=True):
    """Backward of one conv block: BN/LeakyReLU backward (dz, dgamma, dbeta), weight gradient,
    input gradient.  Returns the number of kernel launches.  ``unpack=False`` / ``zero=False``: the caller
    zeroes the WGRAD arena once and unpacks ranges of layers in one launch (``_trunk_backward``)."""
    call, ptr = _lib.call, _lib.ptr
    if L.first and L.recompute:
        # one pass over (x, dA): BatchNorm-backward sums and the weight gradient, z recomputed, dz never formed
        conv = eng.net_ref().module_list[L.idx][0]
        call("avdn_conv0_bwd", ptr(eng.x_in), ptr(conv.weight), ptr(L.g), ptr(L.mask), ptr(L.scale), ptr(L.shift), ptr(L.mean),
             ptr(L.rstd), LEAKY_SLOPE, eng.N, L.Hin, L.Win, ptr(L.zw), ptr(L.xs9), ptr(L.sums), ptr(L.gw), ptr(L.dw),
             ptr(L.dgamma), ptr(L.dbeta))
        return 2
    if L.bnb_fused and L.bnb_ready:
        # the sums were reduced by the epilogue of the dgrad that wrote L.g: coefficients + apply only
        call("avdn_bn_backward_apply", ptr(L.g), ptr(L.z), ptr(L.scale), ptr(L.shift), ptr(L.mean), ptr(L.rstd), L.R,
             L.Cout_p, L.Cout, LEAKY_SLOPE, ptr(L.bsums), ptr(L.coef), ptr(L.dz), ptr(L.dgamma), ptr(L.dbeta))
        L.bnb_ready = False
        n = 2
    else:
        call("avdn_bn_backward", ptr(L.g), ptr(L.z), ptr(L.scale), ptr(L.shift), ptr(L.mean), ptr(L.rstd), L.R,
             L.Cout_p, L.Cout, LEAKY_SLOPE, ptr(L.sums), ptr(L.dz), ptr(L.dgamma), ptr(L.dbeta))
        n = 3                       # reduce, coefficients, apply
    if L.first:
        call("avdn_conv0_wgrad", ptr(L.dz), ptr(eng.x_in), ptr(L.dw), eng.N, L.Hin, L.Win)
        return n + 1
    if L.halo_wgrad:
        call("avdn_conv3x3_thin_wgrad", ptr(L.dz), ptr(L.src.a), ptr(L.dw), eng.N, L.Hin, L.Win, L.Cin_p, L.Cout_p,
             flops=L.flops)
        n += 1
        unpack = False
    else:
        if zero:
            L.dwf.zero_()
            n += 1
        L.p_wgrad.run()
        n += 1
    if unpack:
        if L.pairs:
            call("avdn_unpack_conv_wgrad_pairs", ptr(L.dwf), L.Cout, L.Cin, L.k, L.s, L.Cout_p, L.Cin_p, ptr(L.dw))
        else:
            call("avdn_unpack_conv_wgrad", ptr(L.dwf), L.Cout, L.Cin, L.k, L.Cin_p, ptr(L.dw))
        n += 1
    if L.src.bnb_fused:
        if zero:
            L.src.bsums.zero_()
            n += 1
        L.src.bnb_ready = True
    if L.halo_dgrad:
        call("avdn_conv3x3_thin_dgrad", ptr(L.dz), ptr(L.wd), ptr(L.src.g), eng.N, L.Hin, L.Win, L.Cin_p,
             L.Cout_p, flops=L.flops)
        return n + 1
    for p in L.p_dgrad:
        p.run()
    return n + len(L.p_dgrad)


def _trunk_backward(net, eng, dout, after_layer=None, flush_layers=None):
    """Backward of every block; parameter gradients are ACCUMULATED into the
    engine's gradient tensors (``L.dw / L.dgamma / L.dbeta``: views of the optimiser
    arena when one is attached, engine-owned buffers otherwise).
    The WGRAD outputs are folded into the weight gradients in one launch per range of layers: at
    every layer index in ``flush_layers`` (the blocks that close a data-parallel bucket) and at the end.
    ``after_layer(i)`` is called once the gradients of conv block ``i`` (counted from
    the input) are complete -- the hook the data-parallel bucketing uses."""
    call, ptr = _lib.call, _lib.ptr
    eng.build_bwd(net)
    tbl = eng.conv_table(net)                      # now carries the dwf / grad pointers
    last = eng.last
    eng.dwf_arena.zero_()
    n = 2
    call("avdn_nchw_f32_to_nhwc", ptr(dout), ptr(last.g), eng.N, last.Hout * last.Wout, last.Cout_p)
    flush = set(flush_layers or ())
    hi = len(eng.layers) - 1                       # highest layer whose WGRAD output is still pending
    for li in reversed(range(len(eng.layers))):
        n += _layer_backward(eng, eng.layers[li], unpack=False, zero=False)
        if li in flush or li == 0:
            lo = max(li, 1)                        # layer 0 (conv0) writes its gradient directly
            if hi >= lo:
                call("avdn_unpack_conv_wgrads", ptr(tbl), lo - 1, hi - lo + 1)
                n += 1
            hi = li - 1
        if after_layer is not None:
            after_layer(li)
    eng.launches += n


class _TrunkFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, eng, lease, x_nhwc4, train, *params):
        out = _trunk_forward(net, eng, x_nhwc4, train)
        ctx.net, ctx.eng, ctx.train = net, eng, train
        ctx.save_for_backward(lease)     # holds the engine's activations until this node's graph is freed
        return out

    @staticmethod
    def backward(ctx, dout):
        net, eng = ctx.net, ctx.eng
        if not ctx.train:
            raise RuntimeError("Darknet backward is implemented for train mode (batch statistics) only")
        eng.build_bwd(net)
        own = net._grad_arena is None
        if own:
            for L in eng.layers:
                L.dw.zero_(); L.dgamma.zero_(); L.dbeta.zero_()
        _trunk_backward(net, eng, dout.contiguous().float())
        flat = []
        for L in eng.layers:
            flat += [L.dw.clone(), L.dgamma.clone(), L.dbeta.clone()] if own else [None, None, None]
        return (None, None, None, None, None, *flat)


class Darknet(nn.Module):
    """YOLOv3 trunk used as the 512x7x7 feature extractor (src/xview_et/agent.py:134-141,593)."""

    def __init__(self, config_path, img_size=416):
        super().__init__()
        self.module_defs = parse_model_config(config_path)
        self.module_defs[0]["height"] = img_size            # dark_net.py:207
        self.hyperparams, self.module_list = create_modules(self.module_defs)
        self.img_size = img_size
        self.loss_names = ["loss", "x", "y", "w", "h", "conf", "cls", "nGT", "TP", "FP", "FPe", "FN", "TC"]
        self._engines = {}
        self._pool = EnginePool(self._pool_engine)
        self._grad_arena = None          # name -> tensor, set by the optimiser arena (xview_et.agent)
        self._pending_batches = 0
        self.register_state_dict_pre_hook(lambda m, prefix, keep_vars: m._flush_batches_tracked())

    def _bump_batches_tracked(self):
        # nn.BatchNorm2d.num_batches_tracked: counted on the host, written to the 57 buffers only
        # when somebody looks (state_dict), instead of 57 one-element kernels per step
        self._pending_batches += 1

    def _flush_batches_tracked(self, *a, **k):
        if self._pending_batches:
            for i, d in enumerate(self.module_defs):
                if d["type"] == "convolutional":
                    self.module_list[i][1].num_batches_tracked += self._pending_batches
            self._pending_batches = 0

    def engine(self, N, H, W, device, slot=0):
        """``slot`` separates engines of equal shape whose activations must coexist (one trunk pass per time step of a
        training rollout, each kept for its own backward pass)."""
        return self._engine(N, H, W, device, slot)

    def _params(self):
        ps = []
        for i, d in enumerate(self.module_defs):
            if d["type"] == "convolutional":
                ps += [self.module_list[i][0].weight, self.module_list[i][1].weight, self.module_list[i][1].bias]
        return ps

    def _engine(self, N, H, W, device, slot=0):
        key = (N, H, W, str(device)) if slot == 0 else (N, H, W, str(device), slot)
        e = self._engines.get(key)
        if e is None:
            e = _Engine(self, N, H, W, device)
            self._engines[key] = e
        return e

    def _pool_engine(self, key, slot):
        return self._engine(*key, slot=lease_slot(slot))

    def forward_nhwc4(self, x_nhwc4):
        """Fast path: ``x`` is the renderer's ``norm_nhwc`` output ``[N,H,W,4]`` bf16
        (R,G,B,0).  Returns ``[N, C_last, H/32, W/32]`` float32.  A train-mode forward with grad enabled
        keeps its engine (and so its activations) until its backward: pending forwards of one shape each
        run on an engine of their own (``_lease.EnginePool``)."""
        _lib.require_cuda(x_nhwc4)
        assert x_nhwc4.dtype == torch.bfloat16 and x_nhwc4.shape[-1] == 4 and x_nhwc4.is_contiguous()
        N, H, W, _ = x_nhwc4.shape
        eng, lease = self._pool.acquire((N, H, W, x_nhwc4.device), self.training and torch.is_grad_enabled())
        return _TrunkFn.apply(self, eng, lease, x_nhwc4, self.training, *self._params())

    def forward(self, x, targets=None, requestPrecision=False, weight=None, epoch=None):
        """Reference signature (dark_net.py:212): ``x`` is ``[N,3,H,W]`` float32 NCHW."""
        if targets is not None:
            raise NotImplementedError("detection losses (YOLOLayer) are outside the AVDN hot path")
        _lib.require_cuda(x)
        N, C, H, W = x.shape
        assert C == 3
        x4 = torch.zeros((N, H, W, 4), dtype=torch.bfloat16, device=x.device)
        x4[..., :3] = x.permute(0, 2, 3, 1)          # layout glue of the compatibility entry point
        return self.forward_nhwc4(x4)
