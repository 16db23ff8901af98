"""The sequence composite named by BASELINE.json `north_star`: audio BiLSTM encoder (84-D x T frames), video (256-D
x F) and text (768-D x L) feature encoders, hierarchical attention fusion, evidential NIG head for valence / arousal
/ dominance, DEER multitask loss.  The reference never wires these modules together itself (SURVEY.md section 0);
the wiring below follows its call stack (section 3.3) and its trainer-facing API (`forward(a,v,t)` or one dict,
`compute_loss`, `get_predictions_and_uncertainties`; section 8b)."""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn

from . import chain, ops
from .deer import MultiDimensionalDEER, nig_dict
from .encoders import EnhancedAudioEncoder, EnhancedTextEncoder, EnhancedVideoEncoder
from .fusion import HierarchicalMultimodalFusion
from .losses import MultiTaskDEERLoss


class SequenceDEERModel(nn.Module):
    def __init__(self, hidden_dim: int = 512, video_feature_dim: int = 256, dropout: float = 0.3,
                 attention_heads: int = 8, emotion_dims: int = 3):
        super().__init__()
        self.audio_encoder = EnhancedAudioEncoder({"hidden_dim": hidden_dim, "dropout": dropout})
        self.video_encoder = EnhancedVideoEncoder({"hidden_dim": hidden_dim, "dropout": dropout,
                                                   "frame_feature_dim": video_feature_dim})
        self.text_encoder = EnhancedTextEncoder({"hidden_dim": hidden_dim, "dropout": dropout})
        self.fusion = HierarchicalMultimodalFusion(hidden_dim, hidden_dim, hidden_dim, fusion_dim=hidden_dim,
                                                   intermediate_dim=hidden_dim // 2,
                                                   num_attention_heads=attention_heads, dropout=dropout)
        self.deer = MultiDimensionalDEER(hidden_dim, emotion_dims, hidden_dim // 2, dropout)
        self.loss_fn = MultiTaskDEERLoss()

    def forward(self, audio, video=None, text=None, attention_mask: Optional[torch.Tensor] = None,
                linguistic_features: Optional[torch.Tensor] = None,
                audio_lengths: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """`audio_lengths` [B] (int32 / int64; also read from the batch dict key "audio_lengths"): frames of each audio
        utterance, see EnhancedAudioEncoder.forward.  None: every sample has all T frames."""
        if isinstance(audio, dict):
            d = audio
            audio = d.get("audio", d.get("audio_features"))
            video = d.get("video", d.get("video_features"))
            text = d.get("text", d.get("text_features"))
            attention_mask = d.get("attention_mask", attention_mask)
            linguistic_features = d.get("linguistic_features", linguistic_features)
            audio_lengths = d.get("audio_lengths", audio_lengths)
        ops.begin_step()
        # training: up to 512 samples the recurrence is ONE wave of clusters; beyond that the second wave of the
        # (gate / cell storing) kernels competes with the side work for SMs.  Inference forwards (no stores for BPTT,
        # dual sub-tile kernel) gain at every size (B = 1024: 5.28 -> 5.11 ms).
        if ops.branch_streams_enabled() and audio.is_cuda and (
                audio.shape[0] <= ops.branch_max_batch() or not torch.is_grad_enabled()):
            # The three encoders are independent until the fusion.  The audio LSTM recurrence is a latency-bound
            # persistent kernel (128 of 148 SMs, one CTA each, mostly waiting on the cluster exchange), so it runs on
            # its own HIGH-PRIORITY stream (its CTAs and the second wave of a large batch are placed first) while the
            # video and text encoders fill the rest of the machine from the calling stream: forked here, joined
            # before the fusion; autograd replays each node's backward on the stream its forward ran on, which
            # overlaps BPTT the same way.  Fork / join are event edges, so the pattern is captured unchanged into
            # the CUDA graph of a step.
            main = torch.cuda.current_stream()
            side = self._branch_stream()
            side.wait_stream(main)
            ops.mark("step_start")
            with torch.cuda.stream(side):
                a = ops.mark_tensor(self.audio_encoder(ops.mark_tensor(audio, "audio_in"), audio_lengths), "audio_out")
            tside = self._branch_stream("text", 0) if ops.text_stream_enabled() else None
            if tside is not None:
                # the text encoder (one scorer GEMM, small kernels) on a third stream: with the first LSTM layer's input
                # projection inside the recurrence kernel the audio branch ends first, and video + text in sequence had
                # become the longest chain of the forward (and of the backward, where autograd replays the same streams)
                tside.wait_stream(main)      # fork point: BEFORE the video encoder's launches enter the calling stream
            # program order video -> text (whatever the streams): the video encoder's first node keeps the lowest sequence
            # number behind the audio block, so autograd runs it LAST in backward -- the trainer's early gradient exchange
            # hangs its "everything behind the audio block is complete" hook on it
            v = ops.mark_tensor(self.video_encoder(ops.mark_tensor(video, "video_in")), "video_out")
            if tside is None:
                t = ops.mark_tensor(self.text_encoder(ops.mark_tensor(text, "text_in"), attention_mask,
                                                      linguistic_features), "text_out")
            else:
                with torch.cuda.stream(tside):
                    t = ops.mark_tensor(self.text_encoder(ops.mark_tensor(text, "text_in"), attention_mask,
                                                          linguistic_features), "text_out")
                main.wait_stream(tside)
                t.record_stream(main)
            main.wait_stream(side)
            a.record_stream(main)
            ops.mark("joined")
        else:
            a = self.audio_encoder(audio, audio_lengths)
            v = self.video_encoder(video)
            t = self.text_encoder(text, attention_mask, linguistic_features)
        if chain.enabled() and a.is_cuda and chain.supported(self.fusion, self.deer, a, v, t):
            # fusion + NIG head as ONE persistent-kernel launch (and one in backward): csrc/chain.cu
            fused, _av, _tri, attw, ev = chain.fusion_head_chain(self.fusion, self.deer, a, v, t)
            ops.mark_tensor(fused, "fused")
            ops.mark("head_out_chain")
            out = nig_dict(ev, ops.nig_head(ev), self.deer.dimension_names)
            out["fused_features"] = fused
            out["audio_encoded"], out["video_encoded"], out["text_encoded"] = a, v, t
            out["attention_weights"] = attw
            return out
        fus = self.fusion(a, v, t)
        out = self.deer(ops.mark_tensor(fus["fused_features"], "fused"))
        out["fused_features"] = fus["fused_features"]
        out["audio_encoded"], out["video_encoded"], out["text_encoded"] = a, v, t
        out["attention_weights"] = fus["trimodal_attention_weights"]
        return out

    def branch_streams(self):
        """The side streams this model has forked onto so far (the trainer's early gradient exchange waits for them)."""
        return list(self.__dict__.get("_side_streams", {}).values())

    def _branch_stream(self, name: str = "audio", priority: int = -1):
        dev = torch.cuda.current_device()
        st = self.__dict__.setdefault("_side_streams", {})
        if (dev, name) not in st:
            st[(dev, name)] = torch.cuda.Stream(device=dev, priority=priority)
        return st[(dev, name)]

    def compute_loss(self, predictions: Dict[str, torch.Tensor], targets: torch.Tensor) -> Dict[str, torch.Tensor]:
        return self.loss_fn(predictions, targets)

    @staticmethod
    def get_predictions_and_uncertainties(outputs: Dict[str, torch.Tensor]):
        return outputs["mu_all"], outputs.get("calibrated_uncertainty", outputs["uncertainty_all"])
