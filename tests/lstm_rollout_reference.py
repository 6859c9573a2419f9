"""CPU reference of the LSTM baseline's teacher-forced training rollout (torch autograd), built on the oracle's
functions: the ViT_LSTM step with explicit train-mode dropout masks, and the rollout loss whose autograd is the
reference for every gradient of ``ViT_LSTM.train_engine``."""
import torch
import torch.nn.functional as F

from oracle import model_oracle as mo


def vit_lstm_step(sd, im_feature, current_direct, cls_hidden, lang_feature, state=None, drop=None):
    """``oracle.model_oracle.vit_lstm_step`` (src/models/vln_model.py:213-250) with ``drop`` = None (eval arithmetic;
    the oracle's own function is called) or a dict of keep-scale masks (0 or 1/(1-p)) of the four train-mode
    nn.Dropout sites: ``input`` [B,49] (self.drop on the input of vision_lstm; the saliency fc reads the undropped
    attention output), ``h0`` [B,256] / ``h1`` [B,32] (after the two hidden ReLUs of decoder_2_action_full), ``fc``
    [B,128] (after fc's first ReLU)."""
    if drop is None:
        return mo.vit_lstm_step(sd, im_feature, current_direct, cls_hidden, lang_feature, state)
    h0, c0, hh0, cc0 = state if state is not None else (None, None, None, None)
    inp, _ = mo.soft_dot_attention(cls_hidden, im_feature, sd["attention_layer_vision.linear_in.weight"],
                                   sd["attention_layer_vision.linear_out.weight"])
    hh1, cc1 = mo._lstm_cell(inp * drop["input"], hh0, cc0, sd["vision_lstm.weight_ih"], sd["vision_lstm.weight_hh"],
                             sd["vision_lstm.bias_ih"], sd["vision_lstm.bias_hh"])
    cd = current_direct / 180 * mo.PI_REF
    direction = torch.cat((torch.sin(cd), torch.cos(cd)), dim=1).float()
    demb = direction @ sd["direction_embedding.weight"].t() + sd["direction_embedding.bias"]
    h1, c1 = mo._lstm_cell(demb, h0, c0, sd["direct_lstm.weight_ih"], sd["direct_lstm.weight_hh"],
                           sd["direct_lstm.bias_ih"], sd["direct_lstm.bias_hh"])
    hcat = torch.cat((h1, hh1), 1)
    target = hcat @ sd["attention_layer_lang.linear_in.weight"].t()
    attn = torch.softmax(torch.bmm(lang_feature, target.unsqueeze(2)).squeeze(2), dim=1)
    weighted = torch.bmm(attn.unsqueeze(1), lang_feature).squeeze(1)
    act_in = torch.tanh(torch.cat((weighted, hcat), 1) @ sd["attention_layer_lang.linear_out.weight"].t())
    h = torch.relu(act_in @ sd["decoder_2_action_full.0.weight"].t() + sd["decoder_2_action_full.0.bias"]) * drop["h0"]
    h = torch.relu(h @ sd["decoder_2_action_full.3.weight"].t() + sd["decoder_2_action_full.3.bias"]) * drop["h1"]
    output = h @ sd["decoder_2_action_full.6.weight"].t() + sd["decoder_2_action_full.6.bias"]
    s = torch.relu(inp @ sd["fc.0.weight"].t() + sd["fc.0.bias"]) * drop["fc"]
    h_sali = torch.relu(s @ sd["fc.3.weight"].t() + sd["fc.3.bias"])
    return h1, c1, hh1, cc1, output, h_sali


def rollout_loss(sd, frames, directions, cls_hidden, lang_feature, gt_xy, gt_alt, gt_prog, gt_saliency=None,
                 nss_w=0.0, nss_r=0, train_ml=0.2, drop=None):
    """T chained steps with the recurrent state carried (zero state first, src/xview_lstm/agent.py:546-550), the
    loss ``et_loss(..., jitter=None)`` of every step scaled by ``train_ml / B`` (agent.py:636,883-885) and summed.
    ``frames`` [B,T,512,49]; ``directions`` [B,T] degrees; ``gt_xy`` [B,T,2]; ``gt_alt`` / ``gt_prog`` [B,T];
    ``gt_saliency`` float64 [B,T,224,224] or None; ``drop``: None or a list of T mask dicts."""
    B, T = frames.shape[:2]
    state, total = None, 0
    for t in range(T):
        h1, c1, hh1, cc1, out, h_sali = vit_lstm_step(sd, frames[:, t], directions[:, t:t + 1], cls_hidden,
                                                      lang_feature, state, None if drop is None else drop[t])
        pred = F.interpolate(h_sali.view(-1, 1, 8, 8), size=(224, 224), mode="bilinear", align_corners=False)
        sal = gt_saliency[:, t] if gt_saliency is not None else torch.zeros((B, 224, 224), dtype=torch.float64)
        total = total + mo.step_loss(mo.et_loss(out, pred, gt_xy[:, t], gt_alt[:, t], gt_prog[:, t], sal, nss_w,
                                                nss_r), train_ml, B)
        state = (h1, c1, hh1, cc1)
    return total
