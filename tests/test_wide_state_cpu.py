"""CPU tests of the portable stream-state header of wide engines (more than 128 matched-filter taps): each filter
section holds T = max(128, ntaps) taps and the header is 164 + 16 T + 12 bytes (include/same_engine.h).  same_state_info
accepts a header built here from that layout and rejects one whose size disagrees with the configuration's tap count."""
import struct
import zlib

import numpy as np
import pytest

import sameold_b200 as sb

BLOB_BYTES = 3240


def ntaps(rate):
    """floor(rate / 520.83) in f32, as the engine computes it"""
    return int(np.floor(np.float32(rate) / np.float32(520.83)))


def header_bytes(rate):
    return 164 + 16 * max(128, ntaps(rate)) + 12


def record_bytes(n_words):
    return (8 + 4 * n_words + 15) // 16 * 16 + (BLOB_BYTES + 4 + 15) // 16 * 16


def n_words(rate, dc_len, nff=6, nfb=4):
    return 34 + 2 * dc_len + ntaps(rate) + 64 + 2 * (nff + nfb)


def make_header(cfg, n_records, words, size=None):
    hb = header_bytes(cfg.input_rate) if size is None else size
    h = bytearray(hb)
    struct.pack_into("<10I", h, 0, 0x54534D53, 1, 0x01020304, hb, n_records, words, BLOB_BYTES, 1024,
                     record_bytes(words), 0)
    h[40:116] = bytes(cfg)
    struct.pack_into("<I", h, hb - 4, zlib.crc32(bytes(h[:hb - 4])))
    return h


@pytest.mark.parametrize("rate,size", [(22050, 2224), (66666, 2224), (96000, 3120), (192000, 6064), (266666, 8368)])
def test_documented_header_size(rate, size):
    assert header_bytes(rate) == size


@pytest.mark.parametrize("rate", [88200, 96000, 192000])
@pytest.mark.parametrize("n", [0, 2])
def test_state_info_accepts_a_wide_header(rate, n):
    cfg = sb.SameReceiverBuilder.samedec(rate).config()
    words = n_words(rate, int(np.float32(0.38) * (np.float32(rate) / np.float32(520.83))))
    buf = bytes(make_header(cfg, n, words)) + bytes(n * record_bytes(words))
    got, n_records = sb.state_info(buf)
    assert n_records == n and got.input_rate == rate and bytes(got) == bytes(cfg)


@pytest.mark.parametrize("rate,size", [(96000, 2224), (96000, 3120 + 16), (22050, 3120), (192000, 3120)])
def test_state_info_rejects_a_header_size_that_disagrees_with_the_tap_count(rate, size):
    cfg = sb.SameReceiverBuilder.samedec(rate).config()
    h = make_header(cfg, 0, n_words(rate, 70), size=size)
    with pytest.raises(sb.SameEngineError) as ei:
        sb.state_info(bytes(h))
    assert ei.value.code == 1   # SAME_ERR_INVALID_ARG
