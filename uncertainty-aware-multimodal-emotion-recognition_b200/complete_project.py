"""B200 drop-in for /root/reference/src/models/complete_project.py (the POOLED-feature model, SURVEY.md section 3.2):
ModelConfig (:34), ResidualBlock (:61), EnhancedModalityEncoder (:77), MultiHeadAttention (:121),
UncertaintyEstimator (:186), UncertaintyAwareAttention (:215), HierarchicalFusionModule (:306),
DEERPredictionHead (:369), UncertaintyCalibrationLayer (:420), CompleteDEERModel (:462),
create_complete_deer_model (:605).  Same constructor signatures, state_dict keys and output dictionary; every
floating-point operation runs in libdeer_b200 (ops.*).

Algebra (checked against the reference in tests/golden/pooled_b16.npz): every attention in this model has ONE key
(sequence length 1, :240-270), so softmax == 1 and MultiHeadAttention reduces to output_proj(value_proj(value));
query_proj / key_proj receive exactly zero gradient.  In training the reference still applies Dropout(p) to that
single attention weight per (sample, head) (:172): reproduced by scaling the head slices of the value projection.

Superset API needed by the reference driver/trainer (SURVEY.md section 8b): forward accepts (audio, video, text) or
one dict {'audio','video','text'}; outputs additionally carry gamma/nu/alpha/beta [B,3]; compute_loss is
MultiTaskDEERLoss; ModelCheckpoint provides the save helpers training.py:415-448 calls."""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import ops
from .deer import EVIDENCE_KEY, nig_dict
from .losses import MultiTaskDEERLoss


@dataclass
class ModelConfig:
    audio_dim: int = 84
    video_dim: int = 256
    text_dim: int = 768
    encoder_dim: int = 256
    fusion_dim: int = 512
    emotion_dims: int = 3
    attention_heads: int = 8
    encoder_layers: int = 3
    dropout: float = 0.3
    evidence_weight: float = 1.0
    kl_weight: float = 0.1
    learning_rate: float = 1e-4
    weight_decay: float = 1e-5
    gradient_clip: float = 1.0


def _lin(x, m: nn.Linear, act="none", dropout: float = 0.0, training: bool = False):
    """nn.Linear (+ activation) (+ nn.Dropout, fused into the GEMM epilogue on the chain engine)."""
    return ops.linear(x, m.weight, m.bias, act, dropout=dropout, training=training)


def _ln(x, m: nn.LayerNorm):
    return ops.layer_norm(x, m.weight, m.bias, m.eps)


class ResidualBlock(nn.Module):
    def __init__(self, dim: int, dropout: float = 0.3):
        super().__init__()
        self.dropout = dropout
        self.layers = nn.Sequential(nn.Linear(dim, dim), nn.ReLU(inplace=True), nn.Dropout(dropout), nn.LayerNorm(dim))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        h = _lin(x, self.layers[0], "relu", self.dropout, self.training)
        return ops.add(x, _ln(h, self.layers[3]))


class EnhancedModalityEncoder(nn.Module):
    def __init__(self, input_dim: int, output_dim: int = 256, dropout: float = 0.3, num_layers: int = 3):
        super().__init__()
        self.input_projection = nn.Sequential(nn.Linear(input_dim, output_dim), nn.ReLU(inplace=True),
                                              nn.LayerNorm(output_dim))
        self.encoder_layers = nn.ModuleList([ResidualBlock(output_dim, dropout) for _ in range(num_layers)])
        self.output_projection = nn.Linear(output_dim, output_dim)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        h = _ln(_lin(x, self.input_projection[0], "relu"), self.input_projection[2])
        for layer in self.encoder_layers:
            h = layer(h)
        return _lin(h, self.output_projection)


class MultiHeadAttention(nn.Module):
    """Single-key form of complete_project.py:121-183 (the only form the model uses)."""

    def __init__(self, feature_dim: int, num_heads: int = 8, dropout: float = 0.1):
        super().__init__()
        assert feature_dim % num_heads == 0, "feature_dim must be divisible by num_heads"
        self.feature_dim, self.num_heads = feature_dim, num_heads
        self.head_dim = feature_dim // num_heads
        self.scale = math.sqrt(self.head_dim)
        self.query_proj = nn.Linear(feature_dim, feature_dim)
        self.key_proj = nn.Linear(feature_dim, feature_dim)
        self.value_proj = nn.Linear(feature_dim, feature_dim)
        self.output_proj = nn.Linear(feature_dim, feature_dim)
        self.dropout = nn.Dropout(dropout)

    def forward(self, query: torch.Tensor, key: torch.Tensor, value: torch.Tensor,
                mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        squeeze = value.dim() == 2
        v_in = value if squeeze else value.reshape(-1, self.feature_dim)
        if not squeeze and value.shape[1] != 1:
            raise NotImplementedError("deer_b200 MultiHeadAttention implements the single-key case the model uses")
        v = _lin(v_in, self.value_proj)
        p = self.dropout.p
        if self.training and p > 0.0:
            B = v.shape[0]
            ones = torch.ones((B, self.num_heads), device=v.device, dtype=torch.float32)
            m = ops.dropout(ones, p, True).detach()           # attention weight 1 -> {0, 1/(1-p)} per (sample, head)
            v = ops.rowscale(v.view(B * self.num_heads, self.head_dim), m.view(-1)).view(B, self.feature_dim)
        out = _lin(v, self.output_proj)
        return out if squeeze else out.view(value.shape[0], 1, self.feature_dim)


class UncertaintyEstimator(nn.Module):
    def __init__(self, feature_dim: int):
        super().__init__()
        self.estimator = nn.Sequential(nn.Linear(feature_dim, feature_dim // 2), nn.ReLU(inplace=True), nn.Dropout(0.2),
                                       nn.Linear(feature_dim // 2, feature_dim // 4), nn.ReLU(inplace=True),
                                       nn.Linear(feature_dim // 4, 1), nn.Sigmoid())

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        e = self.estimator
        h = _lin(x, e[0], "relu", e[2].p, self.training)
        return _lin(_lin(h, e[3], "relu"), e[5], "sigmoid")


class UncertaintyAwareAttention(nn.Module):
    def __init__(self, feature_dim: int, num_heads: int = 8, dropout: float = 0.1):
        super().__init__()
        self.feature_dim, self.num_heads, self.dropout = feature_dim, num_heads, dropout
        self.self_attention = MultiHeadAttention(feature_dim, num_heads, dropout)
        self.cross_attention = MultiHeadAttention(feature_dim, num_heads, dropout)
        self.uncertainty_estimator = UncertaintyEstimator(feature_dim)
        self.weight_network = nn.Sequential(nn.Linear(feature_dim * 3 + 3, feature_dim), nn.ReLU(inplace=True),
                                            nn.Dropout(dropout), nn.Linear(feature_dim, 3), nn.Softmax(dim=1))

    def forward(self, audio: torch.Tensor, video: torch.Tensor, text: torch.Tensor) -> Dict[str, torch.Tensor]:
        ua, uv, ut = (self.uncertainty_estimator(z) for z in (audio, video, text))
        sa, sv, st = (self.self_attention(z, z, z) for z in (audio, video, text))
        # cross attention with text as the query: the value token decides the result (one key)
        ca, cv, ct = (self.cross_attention(text, z, z) for z in (audio, video, text))
        unc = torch.cat([ua, uv, ut], dim=1)
        wn = self.weight_network
        w = ops.linear([sa, sv, st, unc], wn[0].weight, wn[0].bias, "relu", dropout=self.dropout, training=self.training)
        w = ops.softmax_rows(_lin(w, wn[3]))
        return {"audio": ops.mix(w[:, 0], unc[:, 0], sa, ca), "video": ops.mix(w[:, 1], unc[:, 1], sv, cv),
                "text": ops.mix(w[:, 2], unc[:, 2], st, ct), "attention_weights": w, "modality_uncertainties": unc}


class HierarchicalFusionModule(nn.Module):
    def __init__(self, feature_dim: int = 256, fusion_dim: int = 512, dropout: float = 0.3):
        super().__init__()
        self.dropout = dropout

        def stage(in_dim):
            return nn.Sequential(nn.Linear(in_dim, fusion_dim), nn.ReLU(inplace=True), nn.Dropout(dropout),
                                 nn.LayerNorm(fusion_dim), nn.Linear(fusion_dim, fusion_dim), nn.ReLU(inplace=True))
        self.av_fusion = stage(feature_dim * 2)
        self.trimodal_fusion = stage(fusion_dim + feature_dim)
        self.fusion_gate = nn.Sequential(nn.Linear(fusion_dim + feature_dim, fusion_dim), nn.Sigmoid())

    def _stage(self, seq, xs):
        h = ops.linear(xs, seq[0].weight, seq[0].bias, "relu", dropout=self.dropout, training=self.training)
        return _lin(_ln(h, seq[3]), seq[4], "relu")

    def forward(self, audio: torch.Tensor, video: torch.Tensor, text: torch.Tensor) -> torch.Tensor:
        av = self._stage(self.av_fusion, [audio, video])
        g = ops.linear([av, text], self.fusion_gate[0].weight, self.fusion_gate[0].bias, "sigmoid")
        tri = self._stage(self.trimodal_fusion, [av, text])
        return ops.gate(g, tri, av)


class DEERPredictionHead(nn.Module):
    def __init__(self, input_dim: int, hidden_dim: int = 256, dropout: float = 0.3):
        super().__init__()
        self.dropout = dropout
        self.evidence_network = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU(inplace=True), nn.Dropout(dropout),
                                              nn.Linear(hidden_dim, hidden_dim // 2), nn.ReLU(inplace=True),
                                              nn.Dropout(dropout), nn.Linear(hidden_dim // 2, 4))

    def evidence(self, x):
        n = self.evidence_network
        h = _lin(x, n[0], "relu", self.dropout, self.training)
        h = _lin(h, n[3], "relu", self.dropout, self.training)
        return _lin(h, n[6])

    def forward(self, x: torch.Tensor) -> Dict[str, torch.Tensor]:
        nig = ops.nig_head(self.evidence(x))          # [7,B]
        keys = ("mu", "nu", "alpha", "beta", "aleatoric_uncertainty", "epistemic_uncertainty", "uncertainty")
        return {k: nig[i] for i, k in enumerate(keys)}


class UncertaintyCalibrationLayer(nn.Module):
    def __init__(self, num_dimensions: int = 3):
        super().__init__()
        self.temperature = nn.Parameter(torch.ones(num_dimensions))
        self.calibration_network = nn.Sequential(nn.Linear(1, 32), nn.ReLU(inplace=True), nn.Linear(32, 16),
                                                 nn.ReLU(inplace=True), nn.Linear(16, 1), nn.Sigmoid())

    def forward(self, uncertainties: torch.Tensor) -> torch.Tensor:
        B, D = uncertainties.shape
        scaled = ops.coldiv(uncertainties, self.temperature)
        n = self.calibration_network
        # the per-dimension loop of the reference (:452-457) shares one MLP: run it on the [B*D,1] column instead
        h = _lin(_lin(scaled.reshape(B * D, 1), n[0], "relu"), n[2], "relu")
        return _lin(h, n[4], "sigmoid").view(B, D)


class CompleteDEERModel(nn.Module):
    DIMS = ("valence", "arousal", "dominance")

    def __init__(self, config: Optional[ModelConfig] = None):
        super().__init__()
        config = config or ModelConfig()
        self.config = config
        c = config
        self.audio_encoder = EnhancedModalityEncoder(c.audio_dim, c.encoder_dim, c.dropout, c.encoder_layers)
        self.video_encoder = EnhancedModalityEncoder(c.video_dim, c.encoder_dim, c.dropout, c.encoder_layers)
        self.text_encoder = EnhancedModalityEncoder(c.text_dim, c.encoder_dim, c.dropout, c.encoder_layers)
        self.attention_module = UncertaintyAwareAttention(c.encoder_dim, c.attention_heads, c.dropout)
        self.fusion_module = HierarchicalFusionModule(c.encoder_dim, c.fusion_dim, c.dropout)
        self.prediction_heads = nn.ModuleDict({d: DEERPredictionHead(c.fusion_dim, 256, c.dropout) for d in self.DIMS})
        self.calibration_layer = UncertaintyCalibrationLayer(c.emotion_dims)
        self.loss_fn = MultiTaskDEERLoss()
        self._initialize_weights()

    def _initialize_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.LayerNorm):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)

    def forward(self, audio_features, video_features=None, text_features=None) -> Dict[str, torch.Tensor]:
        if isinstance(audio_features, dict):
            d = audio_features
            audio_features = d.get("audio", d.get("audio_features"))
            video_features = d.get("video", d.get("video_features"))
            text_features = d.get("text", d.get("text_features"))
        ops.begin_step()
        a = self.audio_encoder(audio_features)
        v = self.video_encoder(video_features)
        t = self.text_encoder(text_features)
        att = self.attention_module(a, v, t)
        fused = self.fusion_module(att["audio"], att["video"], att["text"])
        # the three heads as grouped GEMMs into one [B,3,*] buffer, then one fused NIG kernel
        nets = [self.prediction_heads[d].evidence_network for d in self.DIMS]
        p = self.config.dropout
        D = len(nets)
        dr = dict(dropout=p, training=self.training)
        h = ops.grouped_linear([fused] * D, [n[0].weight for n in nets], [n[0].bias for n in nets], "relu", **dr)
        h = ops.grouped_linear(h, [n[3].weight for n in nets], [n[3].bias for n in nets], "relu", **dr)
        ev = ops.grouped_linear(h, [n[6].weight for n in nets], [n[6].bias for n in nets])
        out = nig_dict(ev, ops.nig_head(ev), self.DIMS, trailing_dim=False)
        out["calibrated_uncertainty"] = self.calibration_layer(out["uncertainty_all"])
        out["attention_weights"] = att["attention_weights"]
        out["modality_uncertainties"] = att["modality_uncertainties"]
        out["fused_features"] = fused
        return out

    def compute_loss(self, predictions: Dict[str, torch.Tensor], targets: torch.Tensor,
                     target_mask: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """`target_mask` (targets' shape, bool / uint8, nonzero = labelled): partially labelled batch, see losses."""
        if target_mask is None:
            return self.loss_fn(predictions, targets)
        return self.loss_fn(predictions, targets, target_mask=target_mask)

    def get_predictions_and_uncertainties(self, outputs: Dict[str, torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
        return outputs["mu_all"], outputs.get("calibrated_uncertainty", outputs["uncertainty_all"])


def create_complete_deer_model(config: Optional[ModelConfig] = None) -> CompleteDEERModel:
    model = CompleteDEERModel(config or ModelConfig())
    total = sum(p.numel() for p in model.parameters())
    print(f"Complete DEER model created: {total:,} parameters "
          f"({model.config.encoder_layers}-layer encoders, {model.config.attention_heads}-head attention)")
    return model


class ModelCheckpoint:
    """The helper src/training/training.py:31,415-448 imports from the (non-existent) `complete_model` module."""

    @staticmethod
    def save_checkpoint(model: nn.Module, optimizer, epoch: int, loss: float, path: str):
        torch.save({"model_state_dict": model.state_dict(),
                    "optimizer_state_dict": optimizer.state_dict() if optimizer is not None else None,
                    "epoch": epoch, "loss": loss}, path)

    @staticmethod
    def save_model_for_inference(model: nn.Module, path: str):
        torch.save({"model_state_dict": model.state_dict(), "config": getattr(model, "config", None)}, path)

    @staticmethod
    def load_checkpoint(model: nn.Module, path: str, map_location=None):
        ck = torch.load(path, map_location=map_location, weights_only=False)
        model.load_state_dict(ck["model_state_dict"])
        return ck
