"""CPU tests of the portable stream-state header (include/same_engine.h, "Portable stream state"): same_state_info reads a
header built here from the documented layout and rejects malformed ones.  No GPU needed."""
import struct
import zlib

import pytest

import sameold_b200 as sb
from sameold_b200 import _lib

HEADER_BYTES = 2224
BLOB_BYTES = 3240
N_WORDS_22050 = 192
RECORD_22050 = 4032


def record_bytes(n_words):
    w = (8 + 4 * n_words + 15) // 16 * 16
    b = (BLOB_BYTES + 4 + 15) // 16 * 16
    return w + b


def make_header(cfg, n_records, n_words=N_WORDS_22050, magic=0x54534D53, version=1, bom=0x01020304):
    h = bytearray(HEADER_BYTES)
    struct.pack_into("<10I", h, 0, magic, version, bom, HEADER_BYTES, n_records, n_words, BLOB_BYTES, 1024,
                     record_bytes(n_words), 0)
    h[40:116] = bytes(cfg)              # same_config: 19 little-endian 4-byte fields
    struct.pack_into("<I", h, 2220, zlib.crc32(bytes(h[:2220])))
    return h


def samedec_cfg():
    return sb.SameReceiverBuilder.samedec(22050).config()


def test_record_size_matches_the_documented_22050_figure():
    assert record_bytes(N_WORDS_22050) == RECORD_22050


@pytest.mark.parametrize("n", [0, 3])
def test_state_info_accepts_a_header_built_from_the_documented_layout(n):
    cfg = samedec_cfg()
    buf = bytes(make_header(cfg, n)) + bytes(n * RECORD_22050)
    got, n_records = sb.state_info(buf)
    assert n_records == n
    assert bytes(got) == bytes(cfg)
    assert got.agc_gain_max == cfg.agc_gain_max and got.input_rate == 22050


@pytest.mark.parametrize("what", ["magic", "version", "byte_order", "header_crc"])
def test_state_info_rejects_a_bad_header(what):
    cfg = samedec_cfg()
    if what == "magic":
        h = make_header(cfg, 0, magic=0x54534D54)
    elif what == "version":
        h = make_header(cfg, 0, version=2)
    elif what == "byte_order":
        h = make_header(cfg, 0, bom=0x04030201)
    else:
        h = make_header(cfg, 0)
        h[100] ^= 1
    with pytest.raises(sb.SameEngineError) as ei:
        sb.state_info(bytes(h))
    assert ei.value.code == 1   # SAME_ERR_INVALID_ARG


@pytest.mark.parametrize("cut", [0, 8, 40, HEADER_BYTES - 1, HEADER_BYTES + RECORD_22050 - 1, HEADER_BYTES + 2 * RECORD_22050 + 1])
def test_state_info_rejects_a_truncated_or_overlong_buffer(cut):
    buf = bytes(make_header(samedec_cfg(), 2)) + bytes(2 * RECORD_22050)
    data = buf[:cut] if cut <= len(buf) else buf + bytes(cut - len(buf))
    with pytest.raises(sb.SameEngineError) as ei:
        sb.state_info(data)
    assert ei.value.code == 1


def test_state_info_rejects_an_inconsistent_record_size():
    h = make_header(samedec_cfg(), 0)
    struct.pack_into("<I", h, 32, RECORD_22050 + 16)
    struct.pack_into("<I", h, 2220, zlib.crc32(bytes(h[:2220])))
    with pytest.raises(sb.SameEngineError) as ei:
        sb.state_info(bytes(h))
    assert ei.value.code == 1


def test_new_calls_are_bound():
    for name in ("same_engine_state_bytes", "same_engine_export_streams", "same_engine_import_streams", "same_state_info",
                 "same_multi_state_bytes", "same_multi_export_streams", "same_multi_import_streams"):
        assert name in _lib.API
        assert hasattr(_lib.load(), name)
