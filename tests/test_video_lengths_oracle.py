"""CPU checks of per-clip video lengths in the fp64 reference (tests/video_lengths_oracle.py): in eval each clip's
encoding is the oracle's on the clip alone; in training the encoder equals stock torch modules (nn.Conv1d on each
truncated clip, nn.BatchNorm1d in train mode on the valid frames of the batch packed into one batch), running statistics
included; lengths = T is the rectangular oracle; the content of padded frames does not matter; shard_batch carries
video_lengths."""
import pytest
import torch
import torch.nn as nn

import deer_b200
import lengths_oracle as LO
import video_lengths_oracle as VLO
from gen_common import det_state_dict
from oracle import deer_oracle as O

DIN, D = 12, 16
P = "video_encoder."


def state_dict(seed):
    enc = deer_b200.EnhancedVideoEncoder({"hidden_dim": D, "dropout": 0.0, "frame_feature_dim": DIN})
    shapes = {k: tuple(v.shape) for k, v in enc.state_dict().items() if k != "temporal_cnn.1.num_batches_tracked"
              and k != "temporal_cnn.5.num_batches_tracked"}
    sd = det_state_dict(shapes, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for bn in ("temporal_cnn.1.", "temporal_cnn.5."):     # non-trivial running statistics (eval uses them)
        sd[bn + "running_mean"] = 0.1 * torch.randn(D, generator=g, dtype=torch.float64)
        sd[bn + "running_var"] = 0.5 + torch.rand(D, generator=g, dtype=torch.float64)
    return sd


def stock_encoder(sd):
    """The module tree of EnhancedVideoEncoder (stock nn.Linear / Conv1d / BatchNorm1d / ... modules), fp64, sd loaded."""
    enc = deer_b200.EnhancedVideoEncoder({"hidden_dim": D, "dropout": 0.0, "frame_feature_dim": DIN}).double()
    full = dict(sd)
    for bn in ("temporal_cnn.1.", "temporal_cnn.5."):
        full[bn + "num_batches_tracked"] = torch.tensor(0)
    enc.load_state_dict(full)
    return enc


def stock_forward(enc, x, lengths):
    """Each clip x[b, :L_b] through the stock modules; the BatchNorm layers (train or eval as enc is) see the valid
    frames of all clips concatenated into one [N, C] batch and split back."""
    sp, cnn, att, op = enc.spatial_projection, enc.temporal_cnn, enc.temporal_attention, enc.output_projection
    Ls = [int(v) for v in lengths]
    h = [sp(x[b, :L]) for b, L in enumerate(Ls)]                              # [L_b, D] each
    for conv, bn, relu in ((cnn[0], cnn[1], cnn[2]), (cnn[4], cnn[5], cnn[6])):
        h = [conv(hb.t().unsqueeze(0)).squeeze(0).t() for hb in h]            # nn.Conv1d on the truncated clip
        h = list(torch.split(relu(bn(torch.cat(h))), Ls))                     # nn.BatchNorm1d on the packed frames
    pooled = torch.stack([(hb * att(hb.unsqueeze(0))[0]).sum(dim=0) for hb in h])
    return op(pooled)


def ragged(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    L = torch.randint(1, T + 1, (B,), generator=g)
    L[0], L[1 % B], L[-1] = 1, min(2, T), T
    return L


@pytest.mark.parametrize("B,T", [(5, 9), (11, 17)])
def test_eval_clip_equals_the_clip_alone(B, T):
    sd = state_dict(B + T)
    L = ragged(B, T, B * T)
    x = torch.randn(B, T, DIN, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    got = VLO.video_encoder(x, sd, training=False, lengths=L)
    enc = stock_encoder(sd).eval()
    for b in range(B):
        Lb = int(L[b])
        if Lb >= 2:
            ref = O.video_encoder(x[b:b + 1, :Lb], sd, training=False)
        else:       # one frame inside a T > 1 batch: the temporal stack on that frame (no one-frame shortcut)
            with torch.no_grad():
                ref = stock_forward(enc, x[b:b + 1], L[b:b + 1])
        assert float((got[b] - ref[0]).abs().max()) < 1e-10, b


@pytest.mark.parametrize("B,T", [(5, 9), (11, 17)])
def test_training_equals_stock_modules_on_packed_frames(B, T):
    sd = state_dict(3 * B + T)
    L = ragged(B, T, B + T)
    x = torch.randn(B, T, DIN, dtype=torch.float64, generator=torch.Generator().manual_seed(4))
    running = {}
    got = VLO.video_encoder(x, sd, training=True, lengths=L, running=running)
    enc = stock_encoder(sd).train()
    with torch.no_grad():
        ref = stock_forward(enc, x, L)
    assert float((got - ref).abs().max()) < 1e-10
    ref_sd = enc.state_dict()
    for bn in ("temporal_cnn.1.", "temporal_cnn.5."):
        for k in ("running_mean", "running_var"):
            assert float((running[bn + k] - ref_sd[bn + k]).abs().max()) < 1e-10, bn + k
        assert int(ref_sd[bn + "num_batches_tracked"]) == running[bn + "num_batches_tracked"] == 1


def test_full_lengths_equal_the_rectangular_oracle():
    B, T = 6, 11
    sd = state_dict(1)
    x = torch.randn(B, T, DIN, dtype=torch.float64, generator=torch.Generator().manual_seed(5))
    full = torch.full((B,), T)
    for training in (False, True):
        got = VLO.video_encoder(x, sd, training=training, lengths=full)
        assert float((got - O.video_encoder(x, sd, training=training)).abs().max()) < 1e-10


@pytest.mark.parametrize("fill", ["nan", "noise"])
def test_padding_content_does_not_matter(fill):
    B, T = 7, 10
    sd = {k: v.clone().requires_grad_(True) for k, v in state_dict(6).items()}
    L = ragged(B, T, 8)
    x0 = torch.randn(B, T, DIN, dtype=torch.float64, generator=torch.Generator().manual_seed(9))
    pad = ~LO.valid_mask(L, B, T)
    x0[pad] = 0.0
    xf = x0.clone()
    xf[pad] = float("nan") if fill == "nan" else 1e3 * torch.randn(int(pad.sum()), DIN, dtype=torch.float64)
    res = []
    for x in (x0, xf):
        xg = x.clone().requires_grad_(True)
        running = {}
        y = VLO.video_encoder(xg, sd, training=True, lengths=L, running=running)
        y.sum().backward()
        res.append((y.detach(), {k: v.grad.clone() for k, v in sd.items() if v.grad is not None}, xg.grad, running))
        for v in sd.values():
            v.grad = None
    (y0, g0, d0, r0), (yf, gf, df, rf) = res
    assert torch.equal(y0, yf)
    assert all(torch.equal(g0[k], gf[k]) for k in g0)
    assert torch.equal(d0, df) and float(df[pad].abs().sum()) == 0.0
    assert all(torch.equal(torch.as_tensor(r0[k]), torch.as_tensor(rf[k])) for k in r0)
    with torch.no_grad():
        assert torch.equal(VLO.video_encoder(x0, sd, training=False, lengths=L),
                           VLO.video_encoder(xf, sd, training=False, lengths=L))


def test_one_frame_batch_ignores_lengths():
    sd = state_dict(2)
    x = torch.randn(4, 1, DIN, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    for training in (False, True):
        got = VLO.video_encoder(x, sd, training=training, lengths=torch.ones(4, dtype=torch.int64))
        assert torch.equal(got, O.video_encoder(x, sd, training=training))


def test_shard_batch_keeps_integer_video_lengths():
    from deer_b200.trainer import shard_batch
    batch = {"video_features": torch.zeros(8, 5, 256), "video_lengths": torch.arange(1, 9, dtype=torch.int64),
             "audio_lengths": torch.arange(1, 9, dtype=torch.int32), "targets": torch.zeros(8, 3)}
    sh = shard_batch(batch, 1, 2)
    assert sh["video_lengths"].dtype == torch.int64 and sh["video_lengths"].tolist() == [5, 6, 7, 8]
    assert sh["audio_lengths"].dtype == torch.int32
