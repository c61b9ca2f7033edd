"""Evaluation loop + report writer (SURVEY §8f rank 1).

Restates ``evaluate_model_with_confusion`` (R/training/utils.py:284-466) for the B200 path: the inference
loop of :311-320 runs through ``HostPredictor`` (double-buffered H2D, kernels, D2H of the class indices),
the confusion counts are accumulated ON THE DEVICE with one ``bincount`` per batch, and the text report is
written in exactly the format of :391-401 so that ``compare_models.py``'s ``ClassificationReportParser``
(TT/compare_models.py:39,44,49) reads it unchanged.  Plots (matplotlib/seaborn are not installed here) are
out of scope; the confusion matrices are returned and saved as ``.npy`` instead of PNGs.
"""
from __future__ import annotations

from pathlib import Path
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .modules import _AMCBase
from .trainer import HostPredictor, predict

TARGET_SNRS = (-8, 0, 8)          # R/training/utils.py:349


def _report_from_confusion(cm: np.ndarray, class_names: Sequence[str], digits: int = 4) -> str:
    """sklearn.metrics.classification_report(..., digits=4) computed from a confusion matrix
    (rows = true class).  Same layout and rounding as sklearn's text report."""
    support = cm.sum(1)
    tp = np.diag(cm).astype(np.float64)
    pred = cm.sum(0).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        prec = np.where(pred > 0, tp / pred, 0.0)
        rec = np.where(support > 0, tp / support, 0.0)
        f1 = np.where(prec + rec > 0, 2 * prec * rec / (prec + rec), 0.0)
    total = int(support.sum())
    acc = tp.sum() / max(total, 1)
    headers = ["precision", "recall", "f1-score", "support"]
    width = max(max(len(c) for c in class_names), len("weighted avg"), digits)
    head_fmt = "{:>{width}s} " + " {:>9}" * len(headers)
    out = head_fmt.format("", *headers, width=width) + "\n\n"
    row_fmt = "{:>{width}s} " + " {:>9.{digits}f}" * 3 + " {:>9}\n"
    for i, name in enumerate(class_names):
        out += row_fmt.format(name, prec[i], rec[i], f1[i], int(support[i]), width=width, digits=digits)
    out += "\n"
    acc_fmt = "{:>{width}s} " + " {:>9}" * 2 + " {:>9.{digits}f}" + " {:>9}\n"
    out += acc_fmt.format("accuracy", "", "", acc, total, width=width, digits=digits)
    w = support / max(total, 1)
    out += row_fmt.format("macro avg", prec.mean(), rec.mean(), f1.mean(), total, width=width, digits=digits)
    out += row_fmt.format("weighted avg", float((prec * w).sum()), float((rec * w).sum()), float((f1 * w).sum()),
                          total, width=width, digits=digits)
    return out


@torch.no_grad()
def evaluate_model_with_confusion(model: _AMCBase, batches: Iterable[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]],
                                  class_names: List[str], save_dir, prefix: str = "test",
                                  device: Optional[torch.device] = None, attack=None) -> Dict:
    """``batches`` yields (images, labels, snrs) like the reference DataLoader (host tensors, or device tensors).
    Returns overall / per-SNR accuracy and confusion matrices and writes ``{prefix}_classification_report.txt``.

    ``attack`` (an ``adversarial.PGDAttack`` on ``model``): robust evaluation.  Each batch is moved to the device and
    replaced by ``attack(images, labels)`` before the prediction; the report has the same format."""
    if attack is not None and attack.model is not model:
        raise ValueError("the attack must be bound to the model being evaluated (a transfer attack crafts the frames "
                         "beforehand and evaluates them without attack=)")
    save_dir = Path(save_dir)
    save_dir.mkdir(parents=True, exist_ok=True)
    model.eval()
    dev = device or model.flat_parameters().device
    C = len(class_names)
    cm_all = torch.zeros(C * C, dtype=torch.int64, device=dev)
    cm_snr = {s: torch.zeros(C * C, dtype=torch.int64, device=dev) for s in TARGET_SNRS}
    hp = None
    pending = None          # (labels, snrs) of the batch whose predictions arrive one call later

    def account(pred_dev, labels, snrs):
        labels = labels.to(dev, non_blocking=True)
        snrs = snrs.to(dev, non_blocking=True).float()
        idx = labels * C + pred_dev
        cm_all.add_(torch.bincount(idx, minlength=C * C))
        for s in TARGET_SNRS:
            sel = (snrs - s).abs() <= 0.5
            cm_snr[s].add_(torch.bincount(idx[sel], minlength=C * C))

    for images, labels, snrs in batches:
        if attack is not None:      # the attack runs no autograd, so no_grad does not get in its way
            images = attack(images.to(dev, non_blocking=True).contiguous(), labels.to(dev, non_blocking=True))
        if images.is_cuda:
            account(predict(model, images.contiguous()), labels, snrs)
            continue
        if hp is None or tuple(hp.x[0].shape) != tuple(images.shape):
            if hp is not None and pending is not None:
                account(hp.flush().to(dev), *pending)
                pending = None
            hp = HostPredictor(model, tuple(images.shape))
        images = images if images.is_pinned() else images.pin_memory()
        prev = hp.predict(images)
        if prev is not None and pending is not None:
            account(prev.to(dev, non_blocking=True), *pending)
        pending = (labels, snrs)
    if hp is not None and pending is not None:
        account(hp.flush().to(dev), *pending)

    cm = cm_all.view(C, C).cpu().numpy()
    acc_overall = float(np.trace(cm)) / max(int(cm.sum()), 1)
    snr_accuracies: Dict[int, float] = {}
    snr_cms: Dict[int, np.ndarray] = {}
    for s in TARGET_SNRS:
        c = cm_snr[s].view(C, C).cpu().numpy()
        if c.sum() == 0:
            continue
        snr_cms[s] = c
        snr_accuracies[s] = float(np.trace(c)) / int(c.sum())
    report = _report_from_confusion(cm, class_names, digits=4)
    report_path = save_dir / f"{prefix}_classification_report.txt"
    with open(report_path, "w") as f:                     # R/training/utils.py:391-401, verbatim layout
        f.write(f"Classification Report - {prefix.capitalize()} Set\n")
        f.write("=" * 80 + "\n\n")
        f.write(f"Overall Accuracy: {acc_overall*100:.2f}%\n\n")
        f.write("Accuracy by SNR:\n")
        for snr, acc in snr_accuracies.items():
            f.write(f"  SNR {snr:+3d} dB: {acc*100:.2f}%\n")
        f.write("\n" + "=" * 80 + "\n\n")
        f.write(report)
    np.save(save_dir / f"{prefix}_confusion_matrix.npy", cm)
    for s, c in snr_cms.items():
        np.save(save_dir / f"{prefix}_confusion_matrix_snr_{s}dB.npy", c)
    return {"overall_accuracy": acc_overall, "snr_accuracies": snr_accuracies, "confusion_matrix": cm,
            "snr_confusion_matrices": snr_cms, "report_path": str(report_path)}
