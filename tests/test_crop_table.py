"""CPU: the crop table tepose_b200.hmr.make_crop_table builds is the 24-byte tp_crop of include/tepose_b200.h."""
import ctypes

import pytest
import torch

from tepose_b200 import _native as nv
from tepose_b200.hmr import make_crop_table


def test_crop_struct_is_24_bytes():
    assert ctypes.sizeof(nv.Crop) == 24
    assert [f for f, _ in nv.Crop._fields_] == ["frame", "cx", "cy", "w", "h", "scale"]


def test_table_rows_read_back_as_tp_crop():
    rows = [(0, 960.25, 540.5, 180.0, 420.0, 1.2), (3, -12.75, 7.125, 0.5, 3000.0, 0.9)]
    table = make_crop_table(rows, "cpu")
    assert table.dtype == torch.int32 and table.shape == (2, 6) and table.is_contiguous()
    raw = (nv.Crop * 2).from_buffer_copy(table.numpy().tobytes())
    for got, want in zip(raw, rows):
        assert got.frame == want[0]
        for name, v in zip(("cx", "cy", "w", "h", "scale"), want[1:]):
            assert getattr(got, name) == torch.tensor(v, dtype=torch.float32).item(), name


@pytest.mark.parametrize("rows", [[(0, 1.0, 2.0, 3.0, 4.0)], [], [[(0, 1, 2, 3, 4, 5)]]])
def test_table_rejects_malformed_rows(rows):
    with pytest.raises(ValueError):
        make_crop_table(rows, "cpu")


def test_table_rejects_fractional_frame_index():
    with pytest.raises(ValueError):
        make_crop_table([(0.5, 1.0, 2.0, 3.0, 4.0, 1.0)], "cpu")
