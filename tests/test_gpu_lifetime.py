"""Lifetime of a context's device resources: a render target that cannot be allocated, and the recovery after it.
Run on the B200 box: pytest -m gpu."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import C1_LAT, C1_LON

pytestmark = pytest.mark.gpu

W, H, R = 640, 200, 200
# 37 views: four batch sets, the last chunk ragged; every eye within a few cells of the centre of the loaded square
VIEWS = [(C1_LAT + 0.001 * (k % 5), C1_LON - 0.001 * (k % 3), -60.0 - 3 * k, 60.0 + 2 * k) for k in range(37)]
QUEUE_CAPACITIES = ("HORIZONATOR_TRI_CAPACITY", "HORIZONATOR_BIG_CAPACITY", "HORIZONATOR_BIGTRI_CAPACITY")


def _windowed(hb, tiles):
    ctx = hb.context_t()
    assert hb.lib.horizonator_init(C.byref(ctx), C1_LAT, C1_LON, None, 0, 0, R, -1.0, False, False, False,
                                   os.fsencode(tiles), None, None, None, False)
    return ctx


def _wedge(hb, ctx):
    image, ranges = np.zeros((H, W, 3), np.uint8), np.zeros((H, W), np.float32)
    ok = hb.lib.horizonator_render_wedge_host(C.byref(ctx), 0, W, image.ctypes.data, ranges.ctypes.data)
    return ok, image, ranges


def _batch(hb, ctx, width, height):
    n = len(VIEWS)
    images, ranges = np.zeros((n, height, width, 3), np.uint8), np.zeros((n, height, width), np.float32)
    assert hb.lib.horizonator_render_batch(C.byref(ctx), n, hb.horizonator._views(VIEWS),
                                           images.ctypes.data, ranges.ctypes.data)
    return images, ranges


def test_failed_resize_then_recovery(tiles_c1, monkeypatch):
    """A resize whose buffers cannot be allocated leaves the context without a target: it reports failure and renders
    nothing.  The next resize restores it, and its renders are then those of a fresh context of that size."""
    import horizonator_b200 as hb
    ctx = _windowed(hb, tiles_c1)
    try:
        _batch(hb, ctx, 1024, 1024)               # the batch sets exist, at the default window size
        # With the queues shrunk to one entry every image-sized buffer asks for more than the device has (the keys
        # alone take 1 TB), so each request is refused at once whatever the order of the allocations.  Without them
        # the capped queues (about 40 GB) could be allocated first.
        for name in QUEUE_CAPACITIES:
            monkeypatch.setenv(name, "1")
        assert not hb.lib.horizonator_resized(C.byref(ctx), 2000000000, 64)
        assert not hb.lib.horizonator_redraw(C.byref(ctx))
        assert not _wedge(hb, ctx)[0]
        for name in QUEUE_CAPACITIES:
            monkeypatch.delenv(name)

        assert hb.lib.horizonator_resized(C.byref(ctx), W, H)
        ok, image, ranges = _wedge(hb, ctx)
        assert ok
        images, batch_ranges = _batch(hb, ctx, W, H)
    finally:
        hb.lib.horizonator_deinit(C.byref(ctx))
        hb.lib.horizonator_deinit(C.byref(ctx))      # idempotent

    fresh = _windowed(hb, tiles_c1)
    try:
        assert hb.lib.horizonator_resized(C.byref(fresh), W, H)
        ok, want_image, want_ranges = _wedge(hb, fresh)
        assert ok
        want_images, want_batch_ranges = _batch(hb, fresh, W, H)
    finally:
        hb.lib.horizonator_deinit(C.byref(fresh))
    assert (want_ranges > 0).any() and (want_batch_ranges > 0).any()
    assert np.array_equal(image, want_image) and np.array_equal(ranges, want_ranges)
    assert np.array_equal(images, want_images) and np.array_equal(batch_ranges, want_batch_ranges)
