"""CPU checks of per-utterance audio lengths: the fp64 reference (tests/lengths_oracle.py) against stock torch.nn.LSTM on a
pack_padded_sequence batch plus a per-utterance softmax, and against the oracle on each utterance alone; host-side
validation of lengths; shard_batch carrying an integer lengths tensor."""
import pytest
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

import lengths_oracle as LO
from deer_b200 import ops
from gen_common import det_state_dict
from oracle import deer_oracle as O

H, IN = 16, 12


def lstm_state_dict(seed, In=IN, hidden=H):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for l in range(2):
        i = In if l == 0 else 2 * hidden
        for sfx in ("", "_reverse"):
            sd[f"lstm.weight_ih_l{l}{sfx}"] = torch.randn(4 * hidden, i, generator=g, dtype=torch.float64) * 0.3
            sd[f"lstm.weight_hh_l{l}{sfx}"] = torch.randn(4 * hidden, hidden, generator=g, dtype=torch.float64) * 0.3
            sd[f"lstm.bias_ih_l{l}{sfx}"] = torch.randn(4 * hidden, generator=g, dtype=torch.float64) * 0.1
            sd[f"lstm.bias_hh_l{l}{sfx}"] = torch.randn(4 * hidden, generator=g, dtype=torch.float64) * 0.1
    return sd


def ragged(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    lengths = torch.randint(1, T + 1, (B,), generator=g)
    lengths[0], lengths[-1] = 1, T
    return lengths


@pytest.mark.parametrize("B,T", [(1, 1), (5, 9), (11, 17)])
def test_bilstm_lengths_equals_packed_nn_lstm(B, T):
    sd = lstm_state_dict(B + T)
    lengths = ragged(B, T, B * T) if B > 1 else torch.tensor([T])
    x = torch.randn(B, T, IN, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    x[~LO.valid_mask(lengths, B, T)] = 7.0        # padding content must not matter
    lstm = torch.nn.LSTM(IN, H, num_layers=2, batch_first=True, bidirectional=True).double()
    lstm.load_state_dict({k[len("lstm."):]: v for k, v in sd.items()})
    with torch.no_grad():
        packed = pack_padded_sequence(x, lengths, batch_first=True, enforce_sorted=False)
        ref, _ = pad_packed_sequence(lstm(packed)[0], batch_first=True, total_length=T)
        got = LO.bilstm(x, sd, lengths=lengths)
    assert float((got - ref).abs().max()) < 1e-10
    assert float(got[~LO.valid_mask(lengths, B, T)].abs().sum()) == 0.0


def test_attn_pool_lengths_is_a_per_utterance_softmax():
    B, T, D = 6, 10, 8
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, T, D, dtype=torch.float64, generator=g)
    w1, b1 = torch.randn(4, D, dtype=torch.float64, generator=g), torch.randn(4, dtype=torch.float64, generator=g)
    w2, b2 = torch.randn(1, 4, dtype=torch.float64, generator=g), torch.randn(1, dtype=torch.float64, generator=g)
    lengths = ragged(B, T, 2)
    out, w = LO.attn_pool(x, w1, b1, w2, b2, lengths)
    for b in range(B):
        L = int(lengths[b])
        ob, wb = O.attn_pool(x[b:b + 1, :L], w1, b1, w2, b2)
        assert float((out[b] - ob[0]).abs().max()) < 1e-10
        assert float((w[b, :L] - wb[0]).abs().max()) < 1e-10
        assert float(w[b, L:].abs().sum()) == 0.0


def test_audio_encoder_lengths_equals_truncated_oracle():
    B, T = 7, 13
    shapes = {"lstm.weight_ih_l0": (64, IN), "lstm.weight_hh_l0": (64, H), "lstm.bias_ih_l0": (64,),
              "lstm.bias_hh_l0": (64,), "lstm.weight_ih_l1": (64, 2 * H), "lstm.weight_hh_l1": (64, H),
              "lstm.bias_ih_l1": (64,), "lstm.bias_hh_l1": (64,),
              "attention.0.weight": (H, 2 * H), "attention.0.bias": (H,), "attention.2.weight": (1, H),
              "attention.2.bias": (1,), "output_projection.0.weight": (2 * H, 2 * H),
              "output_projection.0.bias": (2 * H,), "output_projection.3.weight": (2 * H, 2 * H),
              "output_projection.3.bias": (2 * H,), "output_projection.4.weight": (2 * H,),
              "output_projection.4.bias": (2 * H,)}
    for k in list(shapes):
        if k.startswith("lstm."):
            shapes[k + "_reverse"] = shapes[k]
    sd = det_state_dict(shapes, seed=9)
    lengths = ragged(B, T, 4)
    x = torch.randn(B, T, IN, dtype=torch.float64, generator=torch.Generator().manual_seed(8))
    got = LO.audio_encoder(x, sd, lengths=lengths)
    for b in range(B):
        ref = O.audio_encoder(x[b:b + 1, :int(lengths[b])], sd)
        assert float((got[b] - ref[0]).abs().max()) < 1e-10
    # every length == T is the rectangular oracle
    full = LO.audio_encoder(x, sd, lengths=torch.full((B,), T))
    assert float((full - O.audio_encoder(x, sd)).abs().max()) < 1e-10


def test_host_lengths_are_validated():
    dev = torch.device("cpu")
    assert ops.sequence_lengths(None, 4, 9, dev) is None
    with pytest.raises(ops._lib.DeerError):
        ops.sequence_lengths(torch.tensor([1.0, 2.0]), 2, 9, dev)          # not an integer tensor
    with pytest.raises(ops._lib.DeerError):
        ops.sequence_lengths(torch.tensor([3, 4, 5]), 2, 9, dev)           # not [B]
    with pytest.raises(ops._lib.DeerError):
        ops.sequence_lengths(torch.tensor([0, 4]), 2, 9, dev)              # a CPU length below 1
    with pytest.raises(ops._lib.DeerError):
        ops.sequence_lengths(torch.tensor([3, 10], dtype=torch.int32), 2, 9, dev)   # ... or beyond T


def test_shard_batch_keeps_integer_lengths():
    from deer_b200.trainer import shard_batch
    batch = {"audio_features": torch.zeros(8, 5, 84), "audio_lengths": torch.arange(1, 9, dtype=torch.int32),
             "targets": torch.zeros(8, 3)}
    sh = shard_batch(batch, 1, 2)
    assert sh["audio_lengths"].dtype == torch.int32
    assert sh["audio_lengths"].tolist() == [5, 6, 7, 8]
