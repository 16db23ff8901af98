"""fp64 CPU reference for per-clip video lengths. TEST INFRASTRUCTURE ONLY.

Extends the video path of the oracle (oracle/deer_oracle.py) with `lengths` [B]: sample b is the clip video[b, :L_b].
Each Conv1d sees the clip zero-padded at its own ends, BatchNorm in training takes its statistics over the valid frames
of the whole batch (nn.BatchNorm1d on them packed into one batch), BN+ReLU is 0 at padded frames and the pooling softmax
covers t < L_b. The audio path with lengths comes from tests/lengths_oracle.py. tests/test_video_lengths_oracle.py pins
this module against the oracle on each clip alone (eval) and against stock torch modules on the packed valid frames
(training).
"""
from __future__ import annotations

import torch

import lengths_oracle as LO
from oracle import deer_oracle as O


def _zero(x):
    return torch.zeros((), dtype=x.dtype)


def conv1d_k3(x, w, b, lengths=None):
    """nn.Conv1d(k=3, padding=1) on each clip x[b, :L_b] alone; 0 at padded frames."""
    if lengths is None:
        return O.conv1d_k3(x, w, b)
    valid = LO.valid_mask(lengths, x.shape[0], x.shape[1]).unsqueeze(-1)
    return torch.where(valid, O.conv1d_k3(torch.where(valid, x, _zero(x)), w, b), _zero(x))


def batchnorm_relu(x, g, b, running_mean, running_var, training, lengths=None, eps=1e-5, momentum=0.1, running=None,
                   prefix=""):
    """ReLU(nn.BatchNorm1d) over the valid frames of channels-last x [B,T,C] (all frames without lengths), 0 at padded
    frames.  Training: the batch statistics of the N valid frames; with a dict `running`, the updated running mean /
    variance (momentum, unbiased factor N / (N - 1)) and the num_batches_tracked increment go into it under prefix."""
    B, T, _ = x.shape
    valid = LO.valid_mask(lengths if lengths is not None else torch.full((B,), T), B, T)
    if training:
        xv = x[valid]
        n = xv.shape[0]
        mu = xv.mean(dim=0)
        var = ((xv - mu) ** 2).mean(dim=0)
        if running is not None:
            unb = var * (n / (n - 1)) if n > 1 else var
            running[prefix + "running_mean"] = (1 - momentum) * running_mean + momentum * mu.detach()
            running[prefix + "running_var"] = (1 - momentum) * running_var + momentum * unb.detach()
            running[prefix + "num_batches_tracked"] = 1
    else:
        mu, var = running_mean, running_var
    y = torch.relu((x - mu) / torch.sqrt(var + eps) * g + b)
    return torch.where(valid.unsqueeze(-1), y, _zero(x))


def video_encoder(x, sd, p="", training=True, lengths=None, running=None):
    """EnhancedVideoEncoder on the clips x[b, :L_b] (module docstring).  With T == 1 the oracle's one-frame shortcut runs and
    lengths have no effect.  `running` (dict): receives the BatchNorm running-statistic updates of a training forward
    (keys as in the state dict, num_batches_tracked as the increment)."""
    if x.shape[1] == 1 or (lengths is None and running is None):
        return O.video_encoder(x, sd, p, training)
    B, T, _ = x.shape
    if lengths is not None:
        x = torch.where(LO.valid_mask(lengths, B, T).unsqueeze(-1), x, _zero(x))
    h = torch.relu(O.linear(x, sd[p + "spatial_projection.0.weight"], sd[p + "spatial_projection.0.bias"]))
    for conv, bn in ((0, 1), (4, 5)):
        h = conv1d_k3(h, sd[f"{p}temporal_cnn.{conv}.weight"], sd[f"{p}temporal_cnn.{conv}.bias"], lengths)
        q = f"{p}temporal_cnn.{bn}."
        h = batchnorm_relu(h, sd[q + "weight"], sd[q + "bias"], sd[q + "running_mean"], sd[q + "running_var"], training,
                           lengths, running=running, prefix=q)
    pooled, _ = LO.attn_pool(h, sd[p + "temporal_attention.0.weight"], sd[p + "temporal_attention.0.bias"],
                             sd[p + "temporal_attention.2.weight"], sd[p + "temporal_attention.2.bias"], lengths)
    y = torch.relu(O.linear(pooled, sd[p + "output_projection.0.weight"], sd[p + "output_projection.0.bias"]))
    return O.layer_norm(y, sd[p + "output_projection.3.weight"], sd[p + "output_projection.3.bias"])


def sequence_model(audio, video, text, mask, ling, sd, training=True, audio_lengths=None, video_lengths=None,
                   running=None):
    """The sequence composite with audio lengths (tests/lengths_oracle.py) and video lengths; `running`: see
    video_encoder."""
    if video_lengths is None and running is None:
        return LO.sequence_model(audio, video, text, mask, ling, sd, training, audio_lengths)
    a = LO.audio_encoder(audio, sd, "audio_encoder.", audio_lengths)
    v = video_encoder(video, sd, "video_encoder.", training, video_lengths, running)
    t = O.text_encoder(text, mask, ling, sd, "text_encoder.")
    fus = O.hierarchical_fusion(a, v, t, sd, "fusion.")
    out = O.multidim_deer(fus["fused_features"], sd, "deer.")
    out["fused_features"] = fus["fused_features"]
    out["audio_encoded"], out["video_encoded"], out["text_encoded"] = a, v, t
    return out


def sequence_model_loss(audio, video, text, mask, ling, y, sd, training=True, audio_lengths=None, video_lengths=None,
                        running=None):
    out = sequence_model(audio, video, text, mask, ling, sd, training, audio_lengths, video_lengths, running)
    return out, O.multitask_deer_loss(out, y)
