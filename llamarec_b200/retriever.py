"""Host-side mirror of the hot-path methods of LRUTrainer (reference: trainer/lru.py:30-175).

`LRURetriever.calculate_metrics(batch, exclude_history)` and `generate_candidates(path)` keep the
reference's names, arguments, metric aggregation and `retrieved.pkl` schema (consumed unchanged by
dataloader/llm.py:131-149), but run one fused GPU pass per batch instead of a per-user Python loop
with L scatters, a full argsort and ~17 host syncs per user (SURVEY section 0, fact 3).
"""
from __future__ import annotations

import pickle
from typing import Dict, List, Optional, Sequence

import torch

from .metrics import absolute_metrics_batch_wrapper, metrics_from_sums


class LRURetriever:
    def __init__(self, args, model, val_loader=None, test_loader=None, device: Optional[str] = None):
        self.args = args
        self.model = model
        self.val_loader = val_loader
        self.test_loader = test_loader
        self.metric_ks: List[int] = list(getattr(args, "metric_ks", None) or [1, 5, 10, 20, 50])
        self.device = torch.device(device) if device else next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("LRURetriever needs the model on a CUDA device (no CPU fallback)")

    def to_device(self, batch):
        return [x.to(self.device, non_blocking=True) for x in batch]

    # ---- trainer/lru.py:22-28 -------------------------------------------------------------------
    def calculate_loss(self, batch, dropout: bool = False) -> torch.Tensor:
        """Training loss of one batch; with autograd enabled `loss.backward()` fills the parameters' gradients
        (fused forward + backward train step, see LRURec.ce_loss).  `dropout=True` applies the reference's
        train-mode dropout while the model is in training mode (LRURec.ce_loss)."""
        seqs, labels = batch
        return self.model.ce_loss(seqs, labels, dropout=dropout)

    # ---- trainer/lru.py:30-42 -------------------------------------------------------------------
    def calculate_metrics(self, batch, exclude_history: bool = True) -> Dict[str, float]:
        """Batch-mean Recall/MRR/NDCG@ks, keys in the reference's order (k descending)."""
        seqs, labels = batch
        ks = self.metric_ks
        res = self.model.retrieve(seqs, k=max(ks), exclude_history=exclude_history, labels=labels.view(-1), ks=ks)
        m = metrics_from_sums(res["metric_sums"], ks, seqs.shape[0])
        return {key: m[key] for k in sorted(ks, reverse=True)
                for key in ("Recall@%d" % k, "MRR@%d" % k, "NDCG@%d" % k)}

    # ---- trainer/lru.py:44-175 ------------------------------------------------------------------
    def _sweep(self, loader, want_probs: bool):
        ks = self.metric_ks
        kmax = max(ks)
        k_cand = int(getattr(self.args, "llm_negative_sample_size", 19)) + 1
        k = max(kmax, k_cand)
        sums = torch.zeros(len(ks), 3, dtype=torch.float64)
        users: List[int] = []
        candidates: List[List[int]] = []
        non_users: List[int] = []
        probs: List[List[int]] = []
        all_labels: List[int] = []
        seen = 0
        for batch in loader:
            seqs, labels = self.to_device(batch)
            labels = labels.view(-1)
            res = self.model.retrieve(seqs, k=k, exclude_history=True, labels=labels, ks=ks)
            sums += res["metric_sums"].double().cpu()
            ids = res["ids"].cpu()
            rank = res["label_rank"].cpu()
            B = seqs.shape[0]
            hit = (rank >= 0) & (rank < k_cand)        # `label in top_indices` (trainer/lru.py:86, 128)
            pos = torch.arange(seen + 1, seen + B + 1)  # 1-based position in loader order (:85, :127)
            users.extend(pos[hit].tolist())
            candidates.extend(ids[hit][:, :k_cand].tolist())
            non_users.extend(pos[~hit].tolist())
            if want_probs:
                probs.extend(ids[:, :kmax].tolist())
                all_labels.extend(labels.cpu().tolist())
            seen += B
        metrics: Dict[str, float] = {}
        denom = float(self.args.num_users)               # summed per user, divided by num_users (:90-93)
        host = (sums / denom).tolist()
        for kk in sorted(ks, reverse=True):
            r, m, n = host[ks.index(kk)]
            metrics["Recall@%d" % kk] = r
            metrics["MRR@%d" % kk] = m
            metrics["NDCG@%d" % kk] = n
        return metrics, users, candidates, non_users, probs, all_labels

    def _subset_metrics(self, probs, labels, users) -> Dict[str, float]:
        ks = self.metric_ks
        if len(users) == 0:
            return {f"{n}@{k}": float("nan") for k in sorted(ks, reverse=True) for n in ("Recall", "MRR", "NDCG")}
        idx = torch.tensor(users) - 1
        p = torch.tensor(probs)[idx].to(self.device)
        l = torch.tensor(labels)[idx].to(self.device)
        return absolute_metrics_batch_wrapper(p, l, ks, num_classes=self.args.num_items + 1, preprocessed=True)

    @torch.no_grad()
    def generate_candidates(self, retrieved_data_path: Optional[str] = None) -> Dict:
        self.model.eval()
        val_metrics, val_users, val_candidates, _, _, _ = self._sweep(self.val_loader, want_probs=False)
        test_metrics, test_users, test_candidates, non_test_users, test_probs, test_labels = \
            self._sweep(self.test_loader, want_probs=True)
        test_retrieval = {
            "original_size": len(test_probs),
            "retrieval_size": len(test_candidates),
            "original_metrics": test_metrics,
            "retrieval_metrics": self._subset_metrics(test_probs, test_labels, test_users),
            "non_retrieval_metrics": self._subset_metrics(test_probs, test_labels, non_test_users),
        }
        payload = {
            "val_metrics": val_metrics,
            "val_users": val_users,
            "val_candidates": val_candidates,
            "test_probs": test_probs,
            "test_labels": test_labels,
            "test_metrics": test_metrics,
            "test_users": test_users,
            "test_candidates": test_candidates,
            "non_test_users": non_test_users,
            "test_retrieval": test_retrieval,
        }
        if retrieved_data_path is not None:
            with open(retrieved_data_path, "wb") as f:
                pickle.dump(payload, f)
        return payload
