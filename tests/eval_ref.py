"""NumPy reference of the evaluation metrics (the reference's eval(), train.py:71-109): BCELoss(weight) with logs clamped at
-100, argmax accuracy, and roc_auc_score(argmax(y), pred[:, 1]) as the exact Mann-Whitney pair count."""
import numpy as np


def auc(labels, scores):
    """(#pairs with s_pos > s_neg + 0.5 #ties) / (P N) over positive / negative pairs; NaN when a class is absent."""
    labels, scores = np.asarray(labels), np.asarray(scores, dtype=np.float64)
    pos, neg = scores[labels == 1], scores[labels == 0]
    if len(pos) == 0 or len(neg) == 0:
        return float("nan")
    neg = np.sort(neg)
    below = np.searchsorted(neg, pos, side="left")          # negatives strictly below each positive
    ties = np.searchsorted(neg, pos, side="right") - below
    return float((2 * below.sum() + ties.sum()) / (2.0 * len(pos) * len(neg)))


def metrics(pred, y, class_w=None):
    """(bce, acc, auc) of pred [n, 2] against the one-hot y [n, 2], in float64."""
    p, t = np.asarray(pred, dtype=np.float64), np.asarray(y, dtype=np.float64)
    w = np.ones(2) if class_w is None else np.asarray(class_w, dtype=np.float64).reshape(2)
    with np.errstate(divide="ignore"):
        l1, l0 = np.maximum(np.log1p(-p), -100.0), np.maximum(np.log(p), -100.0)
    bce = float((w[None, :] * ((t - 1.0) * l1 - t * l0)).mean())
    labels = np.argmax(t, axis=1)
    acc = float((np.argmax(p, axis=1) == labels).mean())
    return bce, acc, auc(labels, p[:, 1])
