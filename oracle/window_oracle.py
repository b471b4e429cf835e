"""Sliding-window inference restated in numpy / torch on the CPU: the window grid, the window -> scan coordinate
map and the merge of per-window detections (csrc/windows.cu, ``LSSD3D.predict_scans``).

The merge is ``ssd3d_oracle.detect_from_decoded`` over the scan's "virtual prior list": row j = t * K + r is entry
r of window t (rows past the window's count and label-0 placeholders have probability 0 everywhere), with
probability score_j in class label_j and 0 elsewhere, and the mapped box as its decoded box."""
import math

import numpy as np
import torch

from oracle import ssd3d_oracle as O


def grid(scan_shape, window, overlap):
    """-> (n per axis, origins (T, 3) int64), W fastest."""
    strides = [max(1, int(math.floor(w * (1.0 - overlap)))) for w in window]
    axes = []
    for s, w, st in zip(scan_shape, window, strides):
        n = -(-(s - w) // st) + 1
        axes.append(np.array([min(i * st, s - w) for i in range(n)], dtype=np.int64))
    o = np.array([[a, b, c] for a in axes[0] for b in axes[1] for c in axes[2]], dtype=np.int64)
    return tuple(len(a) for a in axes), o


def map_boxes(boxes, origin, scan_shape, window):
    """(n, 6) fp32 window-fractional boxes -> scan-fractional: x' = fp32(fp32(x * fp32(w/S)) + fp32(o/S))."""
    b = np.asarray(boxes, dtype=np.float32).reshape(-1, 6)
    out = np.empty_like(b)
    for k in range(3):
        scale = np.float32(window[k] / scan_shape[k])
        off = np.float32(origin[k] / scan_shape[k])
        out[:, k] = (b[:, k] * scale) + off
        out[:, k + 3] = (b[:, k + 3] * scale) + off
    return out


def merge(win_boxes, win_labels, win_scores, scan_shape, window, overlap, n_classes, min_score, max_overlap, top_k):
    """Per-window detection lists of ONE scan (T lists, window order) -> (boxes, labels, scores) of the scan."""
    _, origins = grid(scan_shape, window, overlap)
    t_count = len(win_boxes)
    assert t_count == origins.shape[0]
    k = max(1, max(int(np.asarray(b).reshape(-1, 6).shape[0]) for b in win_boxes))
    p = t_count * k
    probs = torch.zeros((1, p, n_classes), dtype=torch.float32)
    decoded = torch.zeros((1, p, 6), dtype=torch.float32)
    for t in range(t_count):
        b = np.asarray(win_boxes[t], dtype=np.float32).reshape(-1, 6)
        lab = np.asarray(win_labels[t]).reshape(-1)
        sc = np.asarray(win_scores[t], dtype=np.float32).reshape(-1)
        mapped = map_boxes(b, origins[t], scan_shape, window)
        for r in range(b.shape[0]):
            if 1 <= int(lab[r]) < n_classes:
                probs[0, t * k + r, int(lab[r])] = float(sc[r])
                decoded[0, t * k + r] = torch.from_numpy(mapped[r])
    ob, ol, os_ = O.detect_from_decoded(probs, decoded, min_score, max_overlap, top_k)
    return ob[0], ol[0], os_[0]
