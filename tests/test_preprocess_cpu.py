"""CPU: the host side of device preprocessing -- the reference's longest-side rounding, and the image table that
es3_preprocess_images reads (strides for CHW / HWC, staging planes and chunk widths, tap records for mixed sizes and dtypes)."""
import numpy as np
import pytest
import torch

from efficientsam3_b200.stage1 import transforms as T


def _reference_shape(oldh, oldw, long_side):
    # ResizeLongestSide.get_preprocess_shape, restated
    scale = long_side * 1.0 / max(oldh, oldw)
    return int(oldh * scale + 0.5), int(oldw * scale + 0.5)


@pytest.mark.parametrize("h,w,s,expect", [
    (1500, 2250, 1024, (683, 1024)),      # SA-1B landscape
    (2250, 1500, 1024, (1024, 683)),      # portrait
    (1500, 2250, 1008, (672, 1008)),
    (768, 1024, 1024, (768, 1024)),       # already at the target
    (1024, 1024, 1024, (1024, 1024)),
    (3, 2048, 1024, (2, 1024)),           # 1.5 rounds up: ties at .5 go up
    (1, 2048, 1024, (1, 1024)),           # 0.5 -> 1
    (6000, 4000, 1024, (1024, 683)),
    (17, 9, 1024, (1024, 542)),           # upscale
    (2250, 1, 1024, (1024, 0)),
])
def test_get_preprocess_shape_matches_the_reference_rounding(h, w, s, expect):
    assert T.get_preprocess_shape(h, w, s) == _reference_shape(h, w, s) == expect
    assert T.ResizeLongestSide(s).target_size(h, w) == expect
    assert T.ResizeLongestSide.get_preprocess_shape(h, w, s) == expect


def test_preprocess_shape_over_a_grid_of_sizes():
    for h in range(1, 300, 7):
        for w in range(1, 300, 11):
            for s in (64, 100, 1008, 1024):
                assert T.get_preprocess_shape(h, w, s) == _reference_shape(h, w, s)


def test_layout_of_chw_and_hwc_tensors():
    chw = torch.zeros(3, 40, 50, dtype=torch.uint8)
    assert T.image_layout(chw.shape, chw.stride(), hwc=False) == (40, 50, 2000, 50, 1)
    hwc = np.zeros((40, 50, 3), dtype=np.uint8)
    t = torch.from_numpy(hwc)
    assert T.image_layout(t.shape, t.stride(), hwc=True) == (40, 50, 1, 150, 3)
    view = torch.zeros(40, 50, 3).permute(2, 0, 1)          # HWC storage seen as CHW: same strides either way
    assert T.image_layout(view.shape, view.stride(), hwc=False) == (40, 50, 1, 150, 3)
    with pytest.raises(ValueError):
        T.image_layout((4, 40, 50), (2000, 50, 1), hwc=False)
    with pytest.raises(ValueError):
        T.image_layout((40, 50), (50, 1), hwc=False)


def test_descriptor_fields_for_interleaved_and_planar_images():
    # HWC uint8: one staged span per row holds all three channels: 768 - 15 bytes -> 251 pixels
    d = T.describe(0x1000, 0, 1500, 2250, 1, 6750, 3, (683, 1024))
    assert list(d[:T.F_KY + 1]) == [0x1000, 1, 6750, 3, 1500, 2250, 683, 1024, 0, 1, 251, 7, 7]
    span = ((d[T.F_XC] - 1) * 3 + 2 + 1)
    assert span <= T.SLOT_ROW - 15 < span + 3
    # CHW uint8: a span per channel plane (256 bytes each)
    d = T.describe(0, 0, 1500, 2250, 1500 * 2250, 2250, 1, (683, 1024))
    assert d[T.F_PLANES] == 3 and d[T.F_XC] == 256 - 15
    # fp32 HWC: 4-byte elements
    d = T.describe(0, 1, 17, 9, 1, 27, 3, (1024, 542))
    assert d[T.F_PLANES] == 1 and d[T.F_XC] == ((753 // 4) - 1 - 2) // 3 + 1
    assert d[T.F_KX] == 3 and d[T.F_KY] == 3          # upscale: support 1 -> 3 taps
    # a downscale by more than 5: taps = ceil(scale) * 2 + 1
    assert T.describe(0, 0, 6000, 4000, 1, 12000, 3, (1024, 683))[[T.F_KX, T.F_KY]].tolist() == [13, 13]


def test_table_lays_tap_records_out_back_to_back():
    rows = [T.describe(0x1000, 0, 1500, 2250, 1, 6750, 3, (683, 1024)),
            T.describe(0x2000, 1, 17, 9, 153, 9, 1, (1024, 542)),
            T.describe(0x3000, 0, 768, 1024, 768 * 1024, 1024, 1, (768, 1024))]
    table, taps, max_out = T.build_table(rows)
    assert table.shape == (3, T.TABLE_FIELDS) and table.dtype == np.int64
    expect, off = [], 0
    for d in table:
        expect.append((off, off + d[T.F_OUT_W] * (d[T.F_KX] + 2)))
        off += d[T.F_OUT_W] * (d[T.F_KX] + 2) + d[T.F_OUT_H] * (d[T.F_KY] + 2)
    assert [tuple(r) for r in table[:, [T.F_TAPX, T.F_TAPY]].tolist()] == expect and taps == off
    assert max_out == 1024
    assert table[:, T.F_PTR].tolist() == [0x1000, 0x2000, 0x3000] and table[:, T.F_DTYPE].tolist() == [0, 1, 0]


def test_preprocessor_affine_and_output_sizes():
    p = T.ImagePreprocessor(1024)
    assert p.output_size(1500, 2250) == (683, 1024)
    a = p._affine[0]
    np.testing.assert_allclose(a[:3], 1 / np.array([58.395, 57.12, 57.375]), rtol=1e-7)
    np.testing.assert_allclose(a[3:], -np.array([123.675, 116.28, 103.53]) / np.array([58.395, 57.12, 57.375]), rtol=1e-7)
    sam2 = T.ImagePreprocessor(1008, (127.5,) * 3, (127.5,) * 3, square=True, float_scale=255.0)
    assert sam2.output_size(300, 420) == (1008, 1008)
    np.testing.assert_allclose(sam2._affine[0], [1 / 127.5] * 3 + [-1.0] * 3, rtol=1e-7)
    np.testing.assert_allclose(sam2._affine[1], [2.0] * 3 + [-1.0] * 3, rtol=1e-7)      # ToTensor floats: (x - 0.5) / 0.5
    arr, hwc = T.ImagePreprocessor._as_tensor(np.zeros((5, 6, 3), dtype=np.float64))
    assert arr.dtype == np.float32 and hwc
    t, hwc = T.ImagePreprocessor._as_tensor(torch.zeros(3, 5, 6, dtype=torch.uint8))
    assert not hwc
    with pytest.raises(TypeError):
        T.ImagePreprocessor._as_tensor(np.zeros((5, 6, 3), dtype=np.int16))
