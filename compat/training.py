"""Flat module name imported by run_multimodal_deer.py:74 (`from training import DEERTrainer, TrainingConfig`).

Mirrors the trainer-facing contract of src/training/training.py (TrainingConfig :39-72, DEERTrainer :75-535):
AdamW with the 0.5x LR group for parameters whose name contains "encoder" (:121-150), CosineAnnealingLR that anneals
every group from its own base value to eta_min 1e-6 (:152-159), gradient clipping (:219), the per-batch dataset loss
weight `weighted_loss = total_loss * dataset_weights[name]` (:59-61, :211-212), the curriculum batch iterator
(:456-484), early stopping (:384-392), per-epoch history.  The step itself is deer_b200's fused trainer step (flat
buffers, NCCL all-reduce when launched under torch.distributed, fused clip+AdamW kernel, CUDA-graph replay); host
batches -- the reference's dicts (:201-204) or the driver's 4-tuples (run_multimodal_deer.py:342) -- are staged to the
device by deer_b200.data.DevicePrefetcher so the H2D copy of batch i+1 overlaps step i."""
import math
import time
from dataclasses import dataclass, field
from typing import Dict, List

import numpy as np
import torch

import _path  # noqa: F401
from deer_b200.data import DevicePrefetcher
from deer_b200.trainer import GROUP_DEFAULT, GROUP_ENCODER, DEERDataParallelTrainer
from evaluation import collect_predictions
from metrics import DEERMetrics


@dataclass
class TrainingConfig:
    """Field names and defaults of training.py:39-72; the last block are additions of this implementation."""
    learning_rate: float = 1e-4
    weight_decay: float = 1e-5
    gradient_clip: float = 1.0
    batch_size: int = 32
    num_epochs: int = 100
    scheduler_type: str = "cosine"
    warmup_epochs: int = 5
    patience: int = 10
    evidence_weight: float = 1.0
    kl_weight: float = 0.1
    attention_reg_weight: float = 0.1
    dataset_weights: Dict[str, float] = field(default_factory=lambda: {"iemocap": 1.0, "ravdess": 0.8, "meld": 0.6})
    curriculum_learning: bool = True
    val_frequency: int = 5
    save_frequency: int = 10
    early_stopping: bool = True
    output_dir: str = "./results"
    log_dir: str = "./logs"
    checkpoint_dir: str = "./checkpoints"
    # --- deer_b200 additions
    min_lr: float = 1e-6               # CosineAnnealingLR eta_min (hard-coded 1e-6 in the reference, :158)
    use_cuda_graph: bool = True        # replay the captured step (one launch) instead of ~150 kernel launches per batch
    prefetch_depth: int = 2            # device buffer sets of the H2D stager
    curriculum_seed: int = 0           # the reference draws np.random.random() per batch (:483); seeded here


class DEERTrainer:
    def __init__(self, model, config: TrainingConfig, device=None):
        self.config = config
        self.device = torch.device(device) if device is not None else next(model.parameters()).device
        self.model = model.to(self.device)
        self.step = DEERDataParallelTrainer(self.model, learning_rate=config.learning_rate,
                                            weight_decay=config.weight_decay, gradient_clip=config.gradient_clip)
        self.metrics = DEERMetrics()
        self.current_epoch = 0
        self.best_val_loss = float("inf")
        self.patience_counter = 0
        self._rng = np.random.RandomState(config.curriculum_seed + 9973 * getattr(self.step, "world", 1))
        self.history: Dict[str, List[float]] = {"train_loss": [], "val_loss": [], "val_ccc": [], "learning_rate": [],
                                                "epoch_time": []}

    # ------------------------------------------------------------------ schedule (training.py:152-174)
    def _group_lrs(self, epoch: int) -> Dict[int, float]:
        """CosineAnnealingLR(T_max=num_epochs, eta_min) applied to each group's base learning rate."""
        c = self.config
        base = {GROUP_ENCODER: 0.5 * c.learning_rate, GROUP_DEFAULT: c.learning_rate}
        if c.scheduler_type == "exponential":
            return {g: b * (0.95 ** epoch) for g, b in base.items()}
        if c.scheduler_type != "cosine" or c.num_epochs <= 1:
            return base
        f = 0.5 * (1.0 + math.cos(math.pi * epoch / c.num_epochs))
        return {g: c.min_lr + (b - c.min_lr) * f for g, b in base.items()}

    # ------------------------------------------------------------------ curriculum iterator (training.py:456-484)
    def _curriculum_probabilities(self) -> Dict[str, float]:
        c = self.config
        if not c.curriculum_learning:
            return {n: 1.0 for n in c.dataset_weights}
        progress = self.current_epoch / max(c.num_epochs, 1)
        if progress < 0.3:
            return {"iemocap": 0.7, "ravdess": 0.2, "meld": 0.1}
        if progress < 0.6:
            return {"iemocap": 0.5, "ravdess": 0.3, "meld": 0.2}
        return {"iemocap": 0.4, "ravdess": 0.3, "meld": 0.3}

    def _batches(self, train_loaders):
        """(host batch, dataset name): every loader in turn, each batch kept with its dataset's probability (names the
        curriculum does not know -- e.g. the driver's `synthetic_train` -- are always kept, as `.get(name, 1.0)`)."""
        probs = self._curriculum_probabilities()
        for name, loader in train_loaders.items():
            p = probs.get(name, 1.0)
            for batch in loader:
                if p >= 1.0 or self._rng.random_sample() < p:
                    yield batch, name

    def train_epoch(self, train_loaders) -> float:
        self.model.train()
        c = self.config
        total = torch.zeros((), device=self.device)
        n = 0
        names: List[str] = []

        def host_batches():
            for batch, name in self._batches(train_loaders):
                names.append(name)
                yield batch

        stager = DevicePrefetcher(host_batches(), self.device, depth=c.prefetch_depth)
        for i, b in enumerate(stager):
            w = float(c.dataset_weights.get(names[i], 1.0))          # training.py:211-212
            if c.use_cuda_graph:
                losses = self.step.train_step_auto(b, loss_weight=w, static_inputs=True)
            else:
                losses = self.step.train_step(b, loss_weight=w)
            total += losses[-1]            # stays on the device: no per-step host sync (cf. training.py:228-230)
            n += 1
        return float(total) / max(n, 1)

    @torch.no_grad()
    def validate_epoch(self, val_loaders) -> Dict[str, float]:
        preds, uncs, tgts = collect_predictions(self.model, val_loaders, self.device)
        m = self.metrics.compute_all_metrics(tgts, preds, uncs)
        self.model.eval()
        total, n = torch.zeros((), device=self.device), 0
        for b in DevicePrefetcher((x for loader in val_loaders.values() for x in loader), self.device):
            total += self.model.compute_loss(self.model(b), b["targets"], b.get("target_mask"))["total_loss"]
            n += 1
        self.model.train()
        return {"val_loss": float(total) / max(n, 1), "val_ccc": m["mean_ccc"], **m}

    def train(self, train_loaders, val_loaders=None) -> Dict[str, List[float]]:
        c = self.config
        for epoch in range(c.num_epochs):
            t0 = time.time()
            self.current_epoch = epoch
            self.step.set_group_lrs(self._group_lrs(epoch))
            self.history["train_loss"].append(self.train_epoch(train_loaders))
            self.history["learning_rate"].append(self.step.lr)
            stop = False
            if val_loaders and ((epoch + 1) % c.val_frequency == 0 or epoch == c.num_epochs - 1):
                v = self.validate_epoch(val_loaders)
                self.history["val_loss"].append(v["val_loss"])
                self.history["val_ccc"].append(v["val_ccc"])
                if v["val_loss"] < self.best_val_loss:           # training.py:384-392
                    self.best_val_loss, self.patience_counter = v["val_loss"], 0
                else:
                    self.patience_counter += 1
                    stop = c.early_stopping and self.patience_counter >= c.patience
            self.history["epoch_time"].append(time.time() - t0)
            if stop:
                break
        return self.history

    def evaluate_model(self, test_loaders) -> Dict[str, float]:
        preds, uncs, tgts = collect_predictions(self.model, test_loaders, self.device)
        return self.metrics.compute_all_metrics(tgts, preds, uncs)
