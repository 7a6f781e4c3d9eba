"""The check vgl_submit runs on the FORMAT blocks of a VGL_HOST_BCF input record (csrc/tables.cpp bcf_fmt_blocks_tile): the
device walks n_fmt blocks (typed-integer key, type descriptor with the vector size, S vectors each) from fmt_off on, so the
record is accepted only when exactly n_fmt blocks tile its fmt_len bytes, and nothing is read outside them."""
import ctypes as C
import os
import struct
import sys

import numpy as np
import pytest

from test_tables import shim  # noqa: F401  (the fixture that builds tests/tables_shim.cpp)

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import bcf_oracle as bo  # noqa: E402

S = 3


@pytest.fixture(scope="module")
def tiles(shim):  # noqa: F811
    f = shim.shim_bcf_fmt_blocks_tile
    f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_int64]

    def call(data, n_fmt, n_samples=S):
        buf = np.frombuffer(data + b"\0" * 16, np.uint8)     # bytes past the record that a bounds error would read as valid
        return f(buf.ctypes.data, len(data), n_fmt, n_samples) == 1
    return call


def block(key, values, typ=bo.BT_INT8):
    """one FORMAT block: key, descriptor, S vectors of len(values) // S values"""
    fmt = {bo.BT_INT8: "<b", bo.BT_INT16: "<h", bo.BT_INT32: "<i", bo.BT_FLOAT: "<f"}[typ]
    return bo.enc_int1(key) + bo.enc_size(len(values) // S, typ) + b"".join(struct.pack(fmt, v) for v in values)


GQ = block(60, [10, 20, 30])
AF = block(61, [0.5] * 6, bo.BT_FLOAT)
WIDE = block(300, list(range(18 * S)), bo.BT_INT16)      # 18 values per sample: the size as a typed integer after the descriptor


def test_exact_tiling_is_accepted(tiles):
    assert tiles(GQ, 1)
    assert tiles(GQ + AF + WIDE, 3)
    assert tiles(bo.enc_int1(62) + bo.enc_size(0, bo.BT_NULL), 1)      # an empty vector


def test_fewer_blocks_than_n_fmt_are_rejected(tiles):
    # the first blocks fill fmt_len exactly, but the record promises more: the device would parse past the range
    assert not tiles(GQ + AF, 3)
    assert not tiles(GQ, 2)


def test_more_blocks_or_trailing_bytes_are_rejected(tiles):
    assert not tiles(GQ + AF, 1)
    assert not tiles(GQ + b"\x00", 1)


@pytest.mark.parametrize("cut", range(1, len(WIDE)))
def test_a_block_cut_anywhere_is_rejected(tiles, cut):
    # key, descriptor, typed size (cut inside its bytes too) and the values, truncated at the end of fmt_len
    assert not tiles(GQ + WIDE[:cut], 2)


def test_typed_size_truncated_at_the_end(tiles):
    head = bo.enc_int1(63) + bytes([15 << 4 | bo.BT_INT8])
    assert not tiles(head, 1)                                  # the size's type byte is missing
    assert not tiles(head + bytes([bo.BT_INT32 | 1 << 4]) + b"\x01\x00", 1)   # int32 size with two of its four bytes


def test_negative_vector_size_is_rejected(tiles):
    for size in (b"\x11\xff", b"\x12\xfe\xff", b"\x13\x00\x00\x00\x80"):    # -1 (int8), -2 (int16), INT32_MIN
        assert not tiles(bo.enc_int1(63) + bytes([15 << 4 | bo.BT_INT8]) + size, 1)


def test_int32_vector_size(tiles):
    n = 40000
    body = bo.enc_int1(64) + bytes([15 << 4 | bo.BT_INT8]) + bytes([1 << 4 | bo.BT_INT32]) + struct.pack("<i", n)
    assert tiles(body + b"\x01" * (n * S), 1)
    assert not tiles(body + b"\x01" * (n * S - 1), 1)
    # a size whose product with S and the value width does not fit 64 bits must not wrap around to a small length
    big = bo.enc_int1(64) + bytes([15 << 4 | bo.BT_INT32]) + bytes([1 << 4 | bo.BT_INT32]) + struct.pack("<i", 2 ** 31 - 1)
    assert not tiles(big + b"\x00" * 64, 1, n_samples=2 ** 62)
