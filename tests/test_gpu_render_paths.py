"""The batch calls when no batch view set can get scratch: they render one view at a time through the context's own
view set, and must give what lone renders give.  Run on the B200 box: pytest -m gpu."""
import gc

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON

pytestmark = pytest.mark.gpu

# A view of a batch set needs about 110 MB of scratch at 3600x600 (the image-sized queues and buffers; R is small), and
# a set takes scratch only while it fits into half of the free device memory.  With 150 MB left free no set gets any,
# while the context's own set, allocated with the context, still renders.
W, H, R = 3600, 600, 180
LEAVE_FREE = 150 << 20
# five eyes around the centre of the loaded square, wide windows (one chain shape for all); not exactly 360 degrees,
# which would place no label
VIEWS = [(C1_LAT + 0.01 * (k - 2), C1_LON - 0.008 * (k - 2), -180.0 + 7.0 * k, 179.8 + 7.0 * k) for k in range(5)]


def test_batch_calls_without_memory_for_a_set_equal_lone_renders(tiles_c1):
    import torch
    import horizonator_b200 as hz
    from tools.pois import summits
    h = hz.horizonator(C1_LAT, C1_LON, W, H, dir_dems=tiles_c1, render_radius_cells=R)
    h.set_zextents(100., 60000.)
    pois = summits(h, 300, seed=3)
    n = len(VIEWS)
    want_i, want_r = np.zeros((n, H, W, 3), np.uint8), np.zeros((n, H, W), np.float32)
    for k, (la, lo, a0, a1) in enumerate(VIEWS):
        h.move(la, lo)
        h.pan_zoom(a0, a1)
        h.render_into(want_i[k], want_r[k])
    assert (want_r > 0).any()
    lone_launches = h.last_render_stats()["launches"]
    # the skylines of the lone renders (horizon_profile_device()'s rule: the topmost pixel with a range > 0), and an
    # observed skyline made of view 0's: every third column from 1000 on
    terrain = want_r > 0
    want_rows = np.where(terrain.any(axis=1), terrain.argmax(axis=1), -1).astype(np.int32)
    want_range = np.where(want_rows >= 0, np.take_along_axis(want_r, np.maximum(want_rows, 0)[:, None, :], 1)[:, 0],
                          -1).astype(np.float32)
    samples = [(c - 1000, float(want_rows[0, c]) + 0.25) for c in range(1000, 1600, 3) if want_rows[0, c] >= 0]
    assert samples
    di = torch.zeros((n, H, W, 3), dtype=torch.uint8, device="cuda")
    dr = torch.zeros((n, H, W), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    gc.collect()                    # contexts of earlier tests that are still to be freed would free memory later
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    hold = torch.empty(max(free - LEAVE_FREE, 0), dtype=torch.uint8, device="cuda")
    try:
        assert torch.cuda.mem_get_info()[0] < 2 * LEAVE_FREE
        bi, br = h.render_batch(VIEWS)
        assert h.last_render_stats()["launches"] == lone_launches       # the lone chain: the context's own set
        h.render_batch_device(VIEWS, di.data_ptr(), dr.data_ptr())
        assert h.last_render_stats()["launches"] == lone_launches
        labels = h.annotate(VIEWS, pois)
        rows, rng = h.skyline(VIEWS)
        scores, score_rows = h.skyline_match(VIEWS, samples, rows=True)
        match_launches = h.last_render_stats()["launches"]
    finally:
        del hold
        torch.cuda.empty_cache()

    assert np.array_equal(bi, want_i) and np.array_equal(br, want_r)
    assert np.array_equal(di.cpu().numpy(), want_i) and np.array_equal(dr.cpu().numpy(), want_r)
    assert np.array_equal(rows, want_rows) and np.array_equal(rng.view(np.uint32), want_range.view(np.uint32))
    assert np.array_equal(score_rows, want_rows)
    # the same calls with memory to spare render on the batch sets (the batch chain: more launches)
    want_labels = h.annotate(VIEWS, pois)
    assert h.last_render_stats()["launches"] != lone_launches
    assert (want_labels["range_rendered_m"] > 0).any()
    assert np.array_equal(labels.view(np.uint32), want_labels.view(np.uint32))
    assert all(np.array_equal(a, b) for a, b in zip(h.skyline(VIEWS), (rows, rng)))
    want_scores, _ = h.skyline_match(VIEWS, samples, rows=True)
    assert h.last_render_stats()["launches"] != match_launches
    assert (want_scores[0] < 1.).any()
    assert np.array_equal(scores.view(np.uint32), want_scores.view(np.uint32))
