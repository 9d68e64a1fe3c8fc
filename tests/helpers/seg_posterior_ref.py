"""
numpy restatement of the segmentation posterior (csrc/irs_segpost.cu, ops.label_counts_update / ops.label_posterior), the
reference the GPU tests compare the kernels with; itself checked against plain loops in tests/test_seg_posterior.py.
  labels: 1..32 distinct non-zero values; any other voxel value is the class "other"
  counts (L, V) int32: counts[l][v] = number of segmentations whose voxel v is labels[l]
  prob = float32(counts) / float32(n);  majority = the largest of the L + 1 class counts, ties to "other" (0), then to the
  earlier label;  entropy = -sum_k p_k ln p_k over the L + 1 classes (float64 here);  summary (L, 3) int64 = (S, O, U)
"""
import numpy as np


def label_counts(segs, labels):
    """segs (N, ...) integer volumes -> counts (L, V) int32"""
    segs = np.asarray(segs).reshape(len(segs), -1)
    return np.stack([(segs == lab).sum(0) for lab in labels]).astype(np.int32)


def label_posterior(counts, n, labels, seg_fixed=None):
    """counts (L, V) -> (prob (L, V) float32, majority (V,) int16, entropy (V,) float64, summary (L, 3) int64)"""
    counts = np.asarray(counts, dtype=np.int64)
    labels = np.asarray(labels, dtype=np.int64)
    prob = counts.astype(np.float32) / np.float32(n)
    classes = np.vstack([(n - counts.sum(0))[None], counts])      # row 0 = "other": np.argmax keeps the first maximum
    best = np.argmax(classes, axis=0)
    majority = np.where(best == 0, 0, labels[np.maximum(best - 1, 0)]).astype(np.int16)
    p = classes / float(n)
    with np.errstate(divide='ignore', invalid='ignore'):
        entropy = -np.where(p > 0, p * np.log(p), 0.0).sum(0)
    fixed = np.zeros(counts.shape[1], np.int64) if seg_fixed is None else np.asarray(seg_fixed).reshape(-1)
    summary = np.stack([counts.sum(1), (counts * (fixed[None] == labels[:, None])).sum(1),
                        ((counts > 0) & (counts < n)).sum(1)], axis=1).astype(np.int64)
    return prob, majority, entropy, summary
