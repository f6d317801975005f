"""CPU tests of the canvas bookkeeping of ``ops.EncodeBuffers``: which occupancy bitmaps each native call receives, and
when the canvas counts as unknown (the whole canvas is then written again)."""
import pytest
import torch

from lidar_vision_vqa_b200 import ops


class FakeLib:
    def __init__(self):
        self.calls = []

    def pillars_set_canvas_occupancy(self, prev, nxt):
        self.calls.append((prev, nxt))
        return 0


@pytest.fixture()
def bufs():
    grid = ops.GridSpec.from_range((-3.2, -3.2, -5.0, 3.2, 3.2, 3.0), (0.2, 0.2, 8.0), 32, 1000)
    with torch.inference_mode():  # the canvas must still get a version counter
        return ops.EncodeBuffers(100, 3, grid, 64, "cpu")


def _call(bufs, lib, rc=0):
    return ops._encode_canvas(bufs, lib, lambda: rc)


def test_bitmaps_alternate_and_start_all_dirty(bufs):
    assert bufs._occupancy.shape == (2, 3, 4) and bool((bufs._occupancy == -1).all())
    lib = FakeLib()
    a, b = bufs._occupancy[0].data_ptr(), bufs._occupancy[1].data_ptr()
    for _ in range(2):
        assert _call(bufs, lib) == 0
    assert lib.calls == [(a, b), (b, a)]


def test_torch_writes_and_invalidate_make_the_canvas_unknown(bufs):
    lib = FakeLib()
    _call(bufs, lib)
    bufs.bev[:, :, 3:5].zero_()          # through a view
    _call(bufs, lib)
    _call(bufs, lib)
    with torch.inference_mode():
        bufs.bev.add_(1)                 # in place under inference mode
    _call(bufs, lib)
    torch.add(bufs.bev, 1, out=bufs.bev)  # out=
    _call(bufs, lib)
    bufs.invalidate_canvas()             # a write the counter cannot see
    _call(bufs, lib)
    _call(bufs, lib)
    assert [p is None for p, _ in lib.calls] == [False, True, False, True, True, True, False]


def test_failed_call_makes_the_canvas_unknown(bufs):
    lib = FakeLib()
    _call(bufs, lib)
    assert _call(bufs, lib, rc=7) == 7
    _call(bufs, lib)

    def boom():
        raise RuntimeError("launch")

    with pytest.raises(RuntimeError):
        ops._encode_canvas(bufs, lib, boom)
    _call(bufs, lib)
    _call(bufs, lib)
    assert [p is None for p, _ in lib.calls] == [False, False, True, False, True, False]
    # a failed call leaves the parity alone: the bitmap it may have written is the one the next call writes again
    assert lib.calls[1][1] == lib.calls[2][1]


def test_no_buffers_no_hook():
    lib = FakeLib()
    assert ops._encode_canvas(None, lib, lambda: 0) == 0
    assert lib.calls == []
