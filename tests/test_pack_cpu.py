"""CPU: the packed-code format of include/mhaq_fq.h, pinned with a numpy packer and decoder, and
the GPU-free parts of the new entry points (row stride, argument errors)."""
import ctypes

import numpy as np
import pytest

from tests import pack_ref as R

INNER = (1, 2, 3, 4, 5, 7, 9, 31, 33, 4095, 4096, 4097)


@pytest.mark.parametrize("bits", R.WIDTHS)
@pytest.mark.parametrize("n_inner", INNER)
def test_numpy_pack_round_trip_and_zero_padding(bits, n_inner):
    rng = np.random.default_rng(bits * 10007 + n_inner)
    codes = rng.integers(0, 1 << bits, size=(3, n_inner), dtype=np.uint32)
    data = R.pack(codes, bits)
    assert data.shape == (3, R.row_bytes(n_inner, bits))
    assert data.shape[1] % 16 == 0
    assert np.array_equal(R.unpack(data, bits, n_inner), codes)
    # padding bits of the last code byte and every byte after it are zero
    used = n_inner * bits
    full = np.unpackbits(data, axis=1, bitorder="little")
    assert not full[:, used:].any()
    # an all-ones tensor sets exactly the used bits
    ones = R.pack(np.full((1, n_inner), (1 << bits) - 1, np.uint32), bits)
    assert np.unpackbits(ones, bitorder="little").sum() == used


def test_bit_layout_by_hand():
    # b = 4: code j in nibble j % 2 of byte j // 2, low nibble first
    assert list(R.pack(np.array([[1, 2, 3]]), 4)[0, :3]) == [0x21, 0x03, 0]
    # b = 2: four codes per byte, code 0 in bits 0-1
    assert R.pack(np.array([[3, 0, 1, 2]]), 2)[0, 0] == 0b10_01_00_11
    # b = 1: code j is bit j % 8 of byte j // 8
    assert list(R.pack(np.array([[1, 0, 0, 0, 0, 0, 0, 1, 1]]), 1)[0, :2]) == [0x81, 0x01]
    # b = 16: little-endian uint16
    assert list(R.pack(np.array([[0x1234]]), 16)[0, :2]) == [0x34, 0x12]
    # b = 8: one byte per code
    assert list(R.pack(np.array([[7, 255]]), 8)[0, :3]) == [7, 255, 0]


def test_saturation_counts_nan_and_out_of_range():
    c, bad = R.saturate(np.array([0.0, 3.0, 4.0, -1.0, np.nan, 2.0]), 2)
    assert list(c) == [0, 3, 3, 0, 0, 2] and bad == 3


def test_packed_row_bytes_matches_the_library():
    from mhaq_b200 import _lib, ops
    L = _lib.lib
    for bits in R.WIDTHS:
        for n in INNER + (0, 1 << 20, (1 << 31) + 3):
            assert L.mhaq_fq_packed_row_bytes(n, bits) == R.row_bytes(n, bits)
            assert ops.packed_row_bytes(n, bits) == R.row_bytes(n, bits)
    for bad in (0, 3, 5, 6, 7, 32, -1):
        assert L.mhaq_fq_packed_row_bytes(16, bad) == -1
    assert L.mhaq_fq_packed_row_bytes(-1, 8) == -1
    with pytest.raises(ValueError):
        ops.packed_row_bytes(16, 3)


def test_pack_unpack_argument_errors_without_gpu():
    from mhaq_b200 import _lib
    L = _lib.lib
    d = ctypes.c_void_p(16)
    pack = lambda x, p, bits, sc, zp, lo, mode, rows, ch, ss=0: L.mhaq_fq_pack_f32(
        x, p, bits, sc, zp, lo, None, ss, 0, 0, 0, mode, rows, 8, ch, None, None)
    assert pack(None, d, 4, d, d, None, 0, 1, 1) == -2               # NULL input
    assert pack(d, None, 4, d, d, None, 0, 1, 1) == -2               # NULL code buffer
    assert pack(d, d, 4, None, d, None, 0, 1, 1) == -2               # NULL scale
    for bad in (0, 3, 5, 7, 32):
        assert pack(d, d, bad, d, d, None, 0, 1, 1) == -1            # unsupported width
    assert pack(d, d, 4, d, d, None, 0, 5, 2, ss=1) == -1            # rows not divisible by channels
    assert pack(d, d, 4, d, d, None, 0, 1, 1, ss=2) == -1            # bad stride
    assert pack(d, d, 4, d, d, None, 1, 1, 1) == -2                  # ACT_LOG without log_act_q
    assert pack(d, d, 4, d, d, d, 1, 2, 2) == -1                     # ACT_LOG with channels
    assert pack(d, d, 4, d, d, None, 9, 1, 1) == -1                  # unknown parameter mode
    unpack = lambda p, bits, y, sc, zp, mode, rows, ch, ss=0: L.mhaq_fq_unpack_f32(
        p, bits, y, sc, zp, ss, 0, mode, rows, 8, ch, None)
    assert unpack(None, 4, d, d, d, 0, 1, 1) == -2                   # NULL codes
    assert unpack(d, 4, None, d, d, 0, 1, 1) == -2                   # NULL output
    assert unpack(d, 4, d, d, None, 0, 1, 1) == -2                   # NULL zero point
    assert unpack(d, 6, d, d, d, 0, 1, 1) == -1                      # unsupported width
    assert unpack(d, 4, d, d, d, 0, 6, 4, ss=1) == -1                # rows not divisible by channels
    assert unpack(d, 4, d, d, d, 0, 1, 1, ss=3) == -1                # bad stride
    assert unpack(d, 4, d, d, d, 1, 2, 2) == -1                      # ACT_LOG with channels
    assert unpack(d, 4, d, d, d, 4, 1, 1) == -1                      # unknown parameter mode
    # zero-sized tensors launch nothing
    assert L.mhaq_fq_pack_f32(d, d, 4, d, d, None, None, 0, 0, 0, 0, 0, 0, 8, 1, None, None) == 0
    assert L.mhaq_fq_unpack_f32(d, 4, d, d, d, 0, 0, 0, 1, 0, 1, None) == 0
