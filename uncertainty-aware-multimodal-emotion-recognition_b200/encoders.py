"""B200 drop-in for the feature-input halves of the reference modality encoders.

Mirrors /root/reference/src/models/encoders.py (class names, config keys, state_dict keys, init):
  EnhancedAudioEncoder  :50-389   BiLSTM(84->256 x2 layers, bidirectional) + attention pooling + projection
  EnhancedVideoEncoder  :392-550  frame features -> Linear/ReLU -> Conv1d(k3)+BN+ReLU x2 -> attention pooling
  EnhancedTextEncoder   :553-761  token embeddings -> masked attention pooling -> projections
Out of scope here (SURVEY.md section 2 rows 2): the librosa waveform featuriser, the 2-D CNN backbone and BERT
itself.  The torch.nn modules below are *parameter containers* only (so names / shapes / initial values match the
reference); their forward() is never used - every FLOP runs in libdeer_b200.so.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn

from . import ops


def _xavier_linear_init(module: nn.Module):
    for m in module.modules():
        if isinstance(m, nn.Linear):
            nn.init.xavier_uniform_(m.weight)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LSTM):
            for name, p in m.named_parameters():
                if "weight" in name:
                    nn.init.xavier_uniform_(p.data)
                elif "bias" in name:
                    nn.init.constant_(p.data, 0)


def _scorer_pool(x_bt, x_rows, att: nn.Sequential, mask=None):
    """Linear-Tanh-Linear scorer + softmax-over-time pooling.  x_rows is any row view of the same data whose
    leading dims enumerate (b,t) or (t,b); x_bt is the [B,T,D] view handed to the pooling kernel."""
    hidden = ops.linear(x_rows, att[0].weight, att[0].bias, "tanh")
    s = ops.rowdot(hidden, att[2].weight.view(-1), att[2].bias)
    return hidden, s


def _scorer_and_pool(x, att: nn.Sequential, mask=None, time_major=False, precise=True, x_bf16=None, lengths=None):
    """Scorer + softmax-over-time pooling of x ([T,B,D] when time_major, else [B,T,D]) as one autograd node
    (ops.scorer_pool), or as the separate scorer / pooling ops when fusion is switched off.  `lengths` (device [B]):
    pooling over each sample's frames t < L_b only."""
    if ops.scorer_pool_fused():
        return ops.scorer_pool(x, att[0].weight, att[0].bias, att[2].weight, att[2].bias, mask, time_major, precise,
                               x_bf16, lengths=lengths)
    _, s = _scorer_pool(None, x, att)
    if time_major:
        return ops.attn_pool(x.permute(1, 0, 2), s.permute(1, 0), mask, lengths)
    return ops.attn_pool(x, s, mask, lengths)


class EnhancedAudioEncoder(nn.Module):
    def __init__(self, config: Optional[Dict] = None):
        super().__init__()
        config = config or {}
        self.sample_rate = config.get("sample_rate", 16000)
        self.hidden_dim = config.get("hidden_dim", 512)
        self.num_layers = config.get("num_layers", 2)
        self.dropout = config.get("dropout", 0.3)
        self.bidirectional = config.get("bidirectional", True)
        if not self.bidirectional:
            raise NotImplementedError("deer_b200: only the bidirectional configuration (the reference default) is built")
        self.enhanced_features_dim = 84
        self.lstm = nn.LSTM(input_size=self.enhanced_features_dim, hidden_size=self.hidden_dim // 2,
                            num_layers=self.num_layers, batch_first=True,
                            dropout=self.dropout if self.num_layers > 1 else 0, bidirectional=True)
        d = self.hidden_dim
        self.attention = nn.Sequential(nn.Linear(d, d // 2), nn.Tanh(), nn.Linear(d // 2, 1), nn.Softmax(dim=1))
        self.output_projection = nn.Sequential(nn.Linear(d, d), nn.ReLU(), nn.Dropout(self.dropout), nn.Linear(d, d),
                                               nn.LayerNorm(d))
        _xavier_linear_init(self)

    def _layer_weights(self, l):
        g = lambda n: getattr(self.lstm, n)
        return (g(f"weight_ih_l{l}"), g(f"weight_hh_l{l}"), g(f"bias_ih_l{l}"), g(f"bias_hh_l{l}"),
                g(f"weight_ih_l{l}_reverse"), g(f"weight_hh_l{l}_reverse"), g(f"bias_ih_l{l}_reverse"),
                g(f"bias_hh_l{l}_reverse"))

    def lstm_forward(self, features: torch.Tensor, return_bf16: bool = False, lengths=None):
        """[B,T,84] -> time-major LSTM output [T,B,hidden_dim] (and, on request, the BF16 copy of it that the last
        layer's recurrence kernel wrote for BPTT: the pooling scorer's weight-gradient GEMM reads it as well).
        `lengths` [B] (int32 / int64; see ops.sequence_lengths): self.lstm on pack_padded_sequence(features, lengths,
        batch_first=True, enforce_sorted=False); the output is ~0 (|h| <= 2^-83 ~ 1e-25) at padded frames t >= L_b."""
        lengths = ops.sequence_lengths(lengths, features.shape[0], features.shape[1], features.device)
        h = features            # batch_first: layer 0 permutes while casting its operands (ops.bilstm_layer)
        h16 = hb16 = None
        nodrop = not (self.training and self.dropout > 0.0)
        nodes = []
        for l in range(self.num_layers):
            # nn.LSTM(dropout=p): dropout on the OUTPUT of every layer but the last == on the input of layers >= 1.
            # Without dropout (inference) the recurrence kernel also writes the FP16 copy of h that the next layer's
            # input projection consumes, so the [T*B, 512] cast pass disappears.
            h, h16, hb16 = ops.bilstm_layer(h, *self._layer_weights(l), input_dropout=self.dropout if l > 0 else 0.0,
                                            training=self.training, x_f16=h16,
                                            emit_f16=nodrop and l + 1 < self.num_layers, return_bf16=True,
                                            x_batch_major=(l == 0), lengths=lengths)
            nodes.append(h.grad_fn)
        # autograd nodes of the layers, first layer first: layer l's weight gradients are complete when node l has run (the
        # data-parallel trainer exchanges the gradients of layers >= 1 beside the BPTT of layer 0)
        self.__dict__["_lstm_bwd_nodes"] = nodes
        return (h, hb16) if return_bf16 else h

    def forward(self, audio_input: torch.Tensor, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        """audio_input [B,T,84] frames.  `lengths` [B] (int32 / int64, CUDA or CPU; None: every sample is T frames long):
        sample b is the utterance audio_input[b, :L_b] and its encoding equals that of the utterance alone -- the LSTM
        runs as on a packed sequence and the attention softmax covers t < L_b only, so the content of the padded frames
        (zeros, noise, NaN) does not matter.  CUDA lengths are clamped to [1, T] on the device; CPU lengths outside that
        range raise."""
        if audio_input.shape[-1] != self.enhanced_features_dim:
            raise NotImplementedError("deer_b200: raw-waveform feature extraction (librosa, CPU) is outside the CUDA hot "
                                      "path; pass pre-extracted 84-D frames [B,T,84]")
        if audio_input.dim() == 2:
            audio_input = audio_input.unsqueeze(1)
        lengths = ops.sequence_lengths(lengths, audio_input.shape[0], audio_input.shape[1], audio_input.device)
        h_tm, hb16 = self.lstm_forward(audio_input, return_bf16=True, lengths=lengths)   # [T,B,D]
        pooled, _ = _scorer_and_pool(h_tm, self.attention, time_major=True, precise=False, x_bf16=hb16, lengths=lengths)
        op = self.output_projection
        y = ops.linear(pooled, op[0].weight, op[0].bias, "relu", dropout=self.dropout, training=self.training)
        y = ops.linear(y, op[3].weight, op[3].bias)
        return ops.layer_norm(y, op[4].weight, op[4].bias, op[4].eps)


class EnhancedVideoEncoder(nn.Module):
    def __init__(self, config: Optional[Dict] = None):
        super().__init__()
        config = config or {}
        self.hidden_dim = config.get("hidden_dim", 512)
        self.dropout = config.get("dropout", 0.3)
        self.max_frames = config.get("max_frames", 32)
        # width of the per-frame features fed to spatial_projection: 512 in the reference (its CNN backbone output),
        # 256 for the BASELINE.json sequence composite (SURVEY.md section 8a row V)
        self.frame_feature_dim = config.get("frame_feature_dim", 512)
        d = self.hidden_dim
        self.spatial_projection = nn.Sequential(nn.Linear(self.frame_feature_dim, d), nn.ReLU(), nn.Dropout(self.dropout))
        self.temporal_cnn = nn.Sequential(
            nn.Conv1d(d, d, kernel_size=3, padding=1), nn.BatchNorm1d(d), nn.ReLU(), nn.Dropout(self.dropout),
            nn.Conv1d(d, d, kernel_size=3, padding=1), nn.BatchNorm1d(d), nn.ReLU())
        self.temporal_attention = nn.Sequential(nn.Linear(d, d // 2), nn.Tanh(), nn.Linear(d // 2, 1), nn.Softmax(dim=1))
        self.output_projection = nn.Sequential(nn.Linear(d, d), nn.ReLU(), nn.Dropout(self.dropout), nn.LayerNorm(d))

    def _bn_relu(self, x, bn: nn.BatchNorm1d, lengths=None):
        return ops.batchnorm_relu(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked,
                                  self.training, bn.momentum, bn.eps, lengths=lengths)

    def forward(self, video_input: torch.Tensor, lengths: Optional[torch.Tensor] = None) -> torch.Tensor:
        """video_input [B,T,frame_feature_dim] per-frame features.  `lengths` [B] (int32 / int64, CUDA or CPU; None: every
        clip has all T frames): sample b is the clip video_input[b, :L_b].  Each Conv1d sees the clip zero-padded at its
        own ends, BatchNorm (training) takes its statistics over the valid frames of the batch only (nn.BatchNorm1d on
        them packed into one batch, running statistics included), BN+ReLU is 0 at padded frames and the attention
        softmax covers t < L_b -- so in eval a clip's encoding equals that of the clip alone, and the content of the
        padded frames (zeros, noise, NaN) changes no output or gradient; the input gradient is 0 there.  A clip with
        L_b = 1 in a batch with T > 1 still goes through the convolutions and BatchNorm (on its one frame); the
        reference's one-frame shortcut (no convolution, no BatchNorm) applies only when T itself is 1, and lengths then
        have no effect.  CUDA lengths are clamped to [1, T] on the device; CPU lengths outside that range raise."""
        if video_input.dim() == 2:
            video_input = video_input.unsqueeze(1)
        if video_input.dim() != 3:
            raise NotImplementedError("deer_b200: raw frames / the 2-D CNN backbone are outside the CUDA hot path; pass "
                                      "per-frame features [B,F,frame_feature_dim]")
        lengths = ops.sequence_lengths(lengths, video_input.shape[0], video_input.shape[1], video_input.device)
        if lengths is not None and video_input.shape[1] == 1:
            lengths = None
        if lengths is not None:
            # padded rows of the input become zero rows (never read): spatial_projection's dW = dz^T x takes no 0 * NaN
            video_input = ops.mask_padding(video_input, lengths)
        sp, cnn = self.spatial_projection, self.temporal_cnn
        p = ops.linear(video_input, sp[0].weight, sp[0].bias, "relu")
        # the autograd node that runs LAST in this encoder's backward: the data-parallel trainer hangs its early
        # gradient exchange on it (trainer._forward_backward)
        self.__dict__["_first_bwd_node"] = p.grad_fn
        if video_input.shape[1] > 1:
            # the two nn.Dropout layers in front of the convolutions ride on the convolutions' padding passes
            h = ops.conv1d_k3(p, cnn[0].weight, cnn[0].bias, self.dropout, self.training, lengths=lengths)
            h = self._bn_relu(h, cnn[1], lengths)
            h = ops.conv1d_k3(h, cnn[4].weight, cnn[4].bias, self.dropout, self.training, lengths=lengths)
            h = self._bn_relu(h, cnn[5], lengths)
            pooled, _ = _scorer_and_pool(h, self.temporal_attention, lengths=lengths)
        else:
            pooled = ops.dropout(p, self.dropout, self.training)[:, 0]
        op = self.output_projection
        y = ops.linear(pooled, op[0].weight, op[0].bias, "relu", dropout=self.dropout, training=self.training)
        return ops.layer_norm(y, op[3].weight, op[3].bias, op[3].eps)


class EnhancedTextEncoder(nn.Module):
    def __init__(self, config: Optional[Dict] = None):
        super().__init__()
        config = config or {}
        self.hidden_dim = config.get("hidden_dim", 512)
        self.dropout = config.get("dropout", 0.3)
        self.max_length = config.get("max_text_length", 128)
        self.bert = None
        self.bert_hidden_size = 768
        d, e = self.hidden_dim, self.bert_hidden_size
        self.token_attention = nn.Sequential(nn.Linear(e, e // 2), nn.Tanh(), nn.Linear(e // 2, 1), nn.Softmax(dim=1))
        self.bert_projection = nn.Sequential(nn.Linear(e, d), nn.ReLU(), nn.Dropout(self.dropout))
        self.linguistic_features_dim = 10
        self.linguistic_projection = nn.Sequential(nn.Linear(10, d // 4), nn.ReLU(), nn.Dropout(self.dropout))
        self.output_projection = nn.Sequential(nn.Linear(d + d // 4, d), nn.ReLU(), nn.Dropout(self.dropout),
                                               nn.LayerNorm(d))

    def extract_linguistic_features(self, input_ids: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
        """encoders.py:648-699: [B,T] int64 token ids -> [B,10] integer statistics, one kernel instead of a Python loop
        over the batch with device syncs."""
        return ops.linguistic_features(input_ids, attention_mask, self.max_length)

    def forward(self, token_embeddings: torch.Tensor, attention_mask: Optional[torch.Tensor] = None,
                linguistic_features: Optional[torch.Tensor] = None,
                input_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
        """token_embeddings [B,T,768] (what BERT's last_hidden_state would be), attention_mask [B,T] 0/1,
        linguistic_features [B,10] (encoders.py:648-699): given, or computed on the device from `input_ids` [B,T]
        int64, or zeros when both are omitted."""
        if not torch.is_floating_point(token_embeddings):
            raise NotImplementedError("deer_b200: BERT / token-id embedding is outside the CUDA hot path; pass 768-D token "
                                      "embeddings [B,T,768]")
        B, T, _ = token_embeddings.shape
        dev = token_embeddings.device
        if attention_mask is None:
            attention_mask = ops.constant(1.0, (B, T), dev)
        m = attention_mask.to(torch.float32)
        if linguistic_features is None and input_ids is not None:
            linguistic_features = self.extract_linguistic_features(input_ids, attention_mask)
        if linguistic_features is None:
            linguistic_features = ops.constant(0.0, (B, 10), dev)
        att = self.token_attention
        if ops.scorer_pool_fused() and not (token_embeddings.requires_grad and torch.is_grad_enabled()):
            # `token_embeddings * attention_mask` (encoders.py:733-735) inside the scorer's operand cast and the pooling
            # kernels: the masked copy is never written
            agg, _ = ops.scorer_pool(token_embeddings, att[0].weight, att[0].bias, att[2].weight, att[2].bias, m,
                                     premask=True)
        else:
            x = ops.rowscale(token_embeddings, m)
            agg, _ = _scorer_and_pool(x, att, mask=m)
        bp, lp, op = self.bert_projection, self.linguistic_projection, self.output_projection
        dr = dict(dropout=self.dropout, training=self.training)
        pb = ops.linear(agg, bp[0].weight, bp[0].bias, "relu", **dr)
        pl = ops.linear(linguistic_features, lp[0].weight, lp[0].bias, "relu", **dr)
        y = ops.linear([pb, pl], op[0].weight, op[0].bias, "relu", **dr)
        return ops.layer_norm(y, op[3].weight, op[3].bias, op[3].eps)


# names the reference driver imports (experiments/run_multimodal_deer.py:77)
AudioEncoder = EnhancedAudioEncoder
VideoEncoder = EnhancedVideoEncoder
TextEncoder = EnhancedTextEncoder


def create_encoders_from_config(config: Optional[Dict] = None):
    """encoders.py:936 counterpart: one encoder per modality from a shared config dict."""
    config = config or {}
    return {"audio": EnhancedAudioEncoder(config.get("audio", config)),
            "video": EnhancedVideoEncoder(config.get("video", config)),
            "text": EnhancedTextEncoder(config.get("text", config))}
