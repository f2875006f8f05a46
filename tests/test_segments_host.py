"""Host-side validation of ``Segments`` (no GPU needed): bad layouts are rejected with ValueError before anything
reaches the device."""
import numpy as np
import pytest

from pyxfocus_b200 import Segments


def test_starts_are_the_exclusive_scan_of_the_sizes():
    s = Segments([3, 0, 5, 1], device="cuda:0")
    assert s.start.dtype == np.int64
    assert list(s.start) == [0, 3, 3, 8, 9]
    assert s.nseg == 4 and s.num == 9
    assert list(s.sizes()) == [3, 0, 5, 1]


@pytest.mark.parametrize("sizes", [[-1, 2], [4, -4], [], [[1, 2]], [1.5, 2]])
def test_bad_sizes_raise(sizes):
    with pytest.raises(ValueError):
        Segments(sizes, device="cuda:0")


def test_length_and_device_mismatch_raise():
    s = Segments([2, 2], device="cuda:0")
    s.check(4, "cuda:0")
    with pytest.raises(ValueError):
        s.check(5, "cuda:0")
    with pytest.raises(ValueError):
        s.check(4, "cuda:1")


def test_after_rejects_bad_flags():
    import torch
    s = Segments([2, 2], device="cuda:0")
    with pytest.raises(ValueError):
        s.after(torch.ones(4, dtype=torch.float64))
    with pytest.raises(ValueError):
        s.after(torch.ones(5, dtype=torch.uint8))       # a CPU tensor of the wrong length: both checks fail first
