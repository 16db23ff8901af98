"""fp64 CPU reference for per-utterance audio lengths.  TEST INFRASTRUCTURE ONLY.

The oracle (oracle/deer_oracle.py) restates the reference modules on rectangular batches.  This module extends the functions
of its audio path with an optional `lengths` [B] (default None: the oracle's own function, unchanged): sample b is the
utterance x[b, :L_b] and the result equals the oracle applied to that utterance alone.  It is batched -- the LSTM state is
reset to zero at every padded step t >= L_b in both directions (so the reverse direction starts at L_b - 1 from zero and
the padded outputs are 0, as pad_packed_sequence returns them) and the attention softmax is masked -- and
tests/test_lengths_oracle.py pins it against torch.nn.LSTM on a pack_padded_sequence batch and against the per-sample
truncated oracle.
"""
from __future__ import annotations

import torch

from oracle import deer_oracle as O


def valid_mask(lengths, B, T):
    """[B,T] bool: t < L_b."""
    return torch.arange(T).unsqueeze(0) < torch.as_tensor(lengths).reshape(B, 1)


def lstm_direction(x, w_ih, w_hh, b_ih, b_hh, reverse, lengths=None):
    if lengths is None:
        return O.lstm_direction(x, w_ih, w_hh, b_ih, b_hh, reverse)
    B, T, _ = x.shape
    H = w_hh.shape[1]
    valid = valid_mask(lengths, B, T)
    x = torch.where(valid.unsqueeze(-1), x, torch.zeros((), dtype=x.dtype))
    h = x.new_zeros(B, H)
    c = x.new_zeros(B, H)
    pre = O.linear(x, w_ih, b_ih + b_hh).unbind(1)
    outs = [None] * T
    w_hh_t = w_hh.t()
    zero = x.new_zeros(B, H)
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        g = pre[t] + h @ w_hh_t
        i_, f_, g_, o_ = g.split(H, dim=1)
        c_new = torch.sigmoid(f_) * c + torch.sigmoid(i_) * torch.tanh(g_)
        h_new = torch.sigmoid(o_) * torch.tanh(c_new)
        v = valid[:, t:t + 1]
        c = torch.where(v, c_new, zero)
        h = torch.where(v, h_new, zero)
        outs[t] = h
    return torch.stack(outs, dim=1)


def bilstm(x, sd, prefix="lstm.", num_layers=2, lengths=None):
    out = x
    for l in range(num_layers):
        f = lstm_direction(out, sd[f"{prefix}weight_ih_l{l}"], sd[f"{prefix}weight_hh_l{l}"],
                           sd[f"{prefix}bias_ih_l{l}"], sd[f"{prefix}bias_hh_l{l}"], False, lengths)
        r = lstm_direction(out, sd[f"{prefix}weight_ih_l{l}_reverse"], sd[f"{prefix}weight_hh_l{l}_reverse"],
                           sd[f"{prefix}bias_ih_l{l}_reverse"], sd[f"{prefix}bias_hh_l{l}_reverse"], True, lengths)
        out = torch.cat([f, r], dim=-1)
    return out


def attn_pool(x, w1, b1, w2, b2, lengths=None):
    if lengths is None:
        return O.attn_pool(x, w1, b1, w2, b2)
    B, T, _ = x.shape
    s = O.linear(torch.tanh(O.linear(x, w1, b1)), w2, b2)  # [B,T,1]
    s = s.masked_fill(~valid_mask(lengths, B, T).unsqueeze(-1), float("-inf"))
    w = torch.softmax(s, dim=1)
    return (x * w).sum(dim=1), w


def audio_encoder(x, sd, p="", lengths=None):
    if lengths is None:
        return O.audio_encoder(x, sd, p)
    h = bilstm(x, sd, p + "lstm.", lengths=lengths)
    pooled, _ = attn_pool(h, sd[p + "attention.0.weight"], sd[p + "attention.0.bias"],
                          sd[p + "attention.2.weight"], sd[p + "attention.2.bias"], lengths)
    y = torch.relu(O.linear(pooled, sd[p + "output_projection.0.weight"], sd[p + "output_projection.0.bias"]))
    y = O.linear(y, sd[p + "output_projection.3.weight"], sd[p + "output_projection.3.bias"])
    return O.layer_norm(y, sd[p + "output_projection.4.weight"], sd[p + "output_projection.4.bias"])


def sequence_model(audio, video, text, mask, ling, sd, training=True, lengths=None):
    if lengths is None:
        return O.sequence_model(audio, video, text, mask, ling, sd, training)
    a = audio_encoder(audio, sd, "audio_encoder.", lengths)
    v = O.video_encoder(video, sd, "video_encoder.", training)
    t = O.text_encoder(text, mask, ling, sd, "text_encoder.")
    fus = O.hierarchical_fusion(a, v, t, sd, "fusion.")
    out = O.multidim_deer(fus["fused_features"], sd, "deer.")
    out["fused_features"] = fus["fused_features"]
    out["audio_encoded"], out["video_encoded"], out["text_encoded"] = a, v, t
    return out


def sequence_model_loss(audio, video, text, mask, ling, y, sd, training=True, lengths=None):
    out = sequence_model(audio, video, text, mask, ling, sd, training, lengths)
    return out, O.multitask_deer_loss(out, y)
