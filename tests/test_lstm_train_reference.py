"""CPU: the reference of the LSTM training rollout (tests/lstm_rollout_reference.py) against the oracle's step."""
import types

import torch

from oracle import model_oracle as mo
import lstm_rollout_reference as ref


def _setup(B=3, T=1, L=7, seed=0):
    from avdn_b200.models.vln_model import ViT_LSTM
    torch.manual_seed(seed)
    m = ViT_LSTM(types.SimpleNamespace(), torch.nn.Identity())
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(seed + 1)
    inp = dict(frames=torch.randn(B, T, 512, 49, generator=g), directions=torch.randint(0, 360, (B, T), generator=g).float(),
               cls_hidden=torch.relu(torch.randn(B, 49, generator=g)), lang_feature=torch.randn(B, L, 768, generator=g),
               gt_xy=torch.rand(B, T, 2, generator=g) * 2 - 1, gt_alt=torch.rand(B, T, generator=g),
               gt_prog=torch.rand(B, T, generator=g))
    return sd, inp


def test_all_ones_masks_equal_eval_step_bit_for_bit():
    sd, x = _setup(T=2)
    B = x["frames"].shape[0]
    ones = dict(input=torch.ones(B, 49), h0=torch.ones(B, 256), h1=torch.ones(B, 32), fc=torch.ones(B, 128))
    state = None
    for t in range(2):
        a = ref.vit_lstm_step(sd, x["frames"][:, t], x["directions"][:, t:t + 1], x["cls_hidden"], x["lang_feature"],
                              state, drop=ones)
        b = mo.vit_lstm_step(sd, x["frames"][:, t], x["directions"][:, t:t + 1], x["cls_hidden"], x["lang_feature"],
                             state)
        for u, v in zip(a, b):
            assert torch.equal(u, v)
        state = a[:4]


def test_masks_change_the_step():
    sd, x = _setup()
    B = x["frames"].shape[0]
    drop = dict(input=torch.ones(B, 49), h0=torch.ones(B, 256), h1=torch.ones(B, 32), fc=torch.ones(B, 128))
    drop["fc"][:, :64] = 0.0
    a = ref.vit_lstm_step(sd, x["frames"][:, 0], x["directions"][:, :1], x["cls_hidden"], x["lang_feature"], drop=drop)
    b = mo.vit_lstm_step(sd, x["frames"][:, 0], x["directions"][:, :1], x["cls_hidden"], x["lang_feature"])
    assert torch.equal(a[4], b[4]) and not torch.equal(a[5], b[5])        # only the saliency branch saw the mask


def test_rollout_loss_at_one_step_is_the_step_loss():
    sd, x = _setup(T=1)
    B = x["frames"].shape[0]
    sal = torch.zeros(B, 1, 224, 224, dtype=torch.float64)
    sal[0, 0, 50:90, 60:120] = 1.0
    total = ref.rollout_loss(sd, gt_saliency=sal, nss_w=0.5, train_ml=0.2, **x)
    _, _, _, _, out, h_sali = mo.vit_lstm_step(sd, x["frames"][:, 0], x["directions"][:, :1], x["cls_hidden"],
                                               x["lang_feature"])
    pred = torch.nn.functional.interpolate(h_sali.view(-1, 1, 8, 8), size=(224, 224), mode="bilinear",
                                           align_corners=False)
    one = mo.step_loss(mo.et_loss(out, pred, x["gt_xy"][:, 0], x["gt_alt"][:, 0], x["gt_prog"][:, 0], sal[:, 0], 0.5),
                       0.2, B)
    assert torch.equal(total, one)
