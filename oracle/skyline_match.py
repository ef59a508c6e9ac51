"""Host restatement of the skyline match rule of horizonator_skyline_match* (include/horizonator-batch.h), for the tests:
numpy float32, an explicit loop over the samples in their order, vectorised over views x headings.  Every operation
is one float32 rounding, as in k_skyline_score, so the scores must agree bit for bit.  Not used by the product."""
import numpy as np

#: horizonator_skyline_sample_t
SAMPLE_DTYPE = np.dtype([("dx", np.int32), ("y", np.float32)])


def samples(pairs):
    """(dx, y) pairs -> SAMPLE_DTYPE array."""
    a = np.asarray(pairs, np.float64).reshape(-1, 2)
    out = np.empty(len(a), SAMPLE_DTYPE)
    out["dx"], out["y"] = a[:, 0], a[:, 1]
    return out


def scores(rows, smp, clip_rows, wrap):
    """rows: (n, W) skyline rows (image row of the topmost terrain pixel, -1 = all sky); smp: SAMPLE_DTYPE array of m >= 1
    samples.  Returns (n, W) float32: scores[k, h] = (sum over i in order of d_i) / m with
    d_i = fmin(|(s - 0.5) - y_i|, clip_rows), s = rows[k, c_i], c_i = h + dx_i (mod W with wrap; outside [0, W)
    missing), and d_i = clip_rows for a missing or all-sky column."""
    rows = np.asarray(rows, np.int64)
    n, W = rows.shape
    m = len(smp)
    assert m >= 1
    clip = np.float32(clip_rows)
    half = np.float32(0.5)
    h = np.arange(W, dtype=np.int64)
    total = np.zeros((n, W), np.float32)
    for i in range(m):
        c = h + np.int64(smp["dx"][i])
        if wrap:
            c = np.mod(c, W)
        missing = (c < 0) | (c >= W)
        s = rows[:, np.clip(c, 0, W - 1)]
        d = np.fmin(np.abs((s.astype(np.float32) - half) - np.float32(smp["y"][i])), clip)
        d = np.where(missing[None, :] | (s < 0), clip, d).astype(np.float32)
        total = (total + d).astype(np.float32)
    return (total / np.float32(m)).astype(np.float32)
