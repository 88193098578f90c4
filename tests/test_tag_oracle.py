"""SURVEY.md 8(f3), oracle side: music CRC / byte count kept by copy_buffer, the Xing / Info / LAME tag frame and the WAV
header reader of oracle/lj_vbrtag.cpp against what REAL lamejs computed under the engine
(tests/golden/lamejs_tag_golden.json, made by tests/golden/make_lamejs_tag_golden.py; seeded uniform-noise cases in
tests/golden/lamejs_seeded_golden.json, made by tests/golden/make_lamejs_seeded_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from synth import make_signal

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "lamejs_tag_golden.json")))
ENGINE = json.load(open(os.path.join(HERE, "golden", "lamejs_seeded_golden.json")))["engine"]

# VBRTag.js:113-145: entries of crc16Lookup as printed in the reference, and the SHA-256 of all 256 (big-endian 16-bit)
CRC_ROWS = {0: 0x0000, 1: 0xC0C1, 2: 0xC181, 3: 0x0140, 4: 0xC301, 8: 0xC601, 127: 0xE041, 128: 0xA001, 252: 0x4100, 253: 0x81C1, 254: 0x8081, 255: 0x4040}
CRC_TABLE_SHA256 = "4052764821e02d264bca5dfa3b5cd61eb2e8fcb335277af5726a319480245a4d"


def _sig(c):
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], seed=c["seed"])
    return l, (r if c["channels"] == 2 else None)


def test_crc_table_and_check_value(oracle):
    L = oracle.lib()
    for i, v in CRC_ROWS.items():
        assert L.lj_crc16_table(i) == v
    tab = [L.lj_crc16_table(i) for i in range(256)]
    assert hashlib.sha256(bytes(b for v in tab for b in (v >> 8, v & 255))).hexdigest() == CRC_TABLE_SHA256
    assert oracle.crc16(b"123456789") == 0xBB3D          # CRC-16/ARC check value
    assert oracle.crc16(b"") == 0 and oracle.crc16(b"6789", oracle.crc16(b"12345")) == 0xBB3D


@pytest.mark.parametrize("name", sorted(GOLD["hot"]))
def test_music_crc_and_byte_count_match_lamejs(oracle, name):
    """gfc.nMusicCRC / nBytesWritten of an ordinary Mp3Encoder run: part of the hot path's state in lamejs."""
    c = GOLD["hot"][name]
    l, r = _sig(c)
    enc = oracle.OracleEncoder(c["channels"], c["samplerate"], c["kbps"])
    out = bytearray()
    step = c["chunk"] or max(len(l), 1)
    for i in range(0, len(l), step):
        out += enc.encode_buffer(l[i:i + step], None if r is None else r[i:i + step])
    out += enc.flush()
    assert hashlib.sha256(bytes(out)).hexdigest() == c["sha256"]
    assert enc.music_crc() == c["music_crc"] == oracle.crc16(bytes(out))
    assert enc.bytes_written() == c["bytes_written"] == len(out)
    enc.close()


def _js_view(tag, js_tag, sideinfo_len):
    """Our tag as the JavaScript would have written it: `0xff & "I"` is 0, `0xff & "3"` is 3 (VBRTag.js:867-870,746-748), and
    the tag CRC follows from those bytes."""
    t = bytearray(tag)
    m = sideinfo_len
    t[m:m + 4] = js_tag[m:m + 4]
    v = m + 120
    t[v:v + 9] = js_tag[v:v + 9]
    return t, v


@pytest.mark.parametrize("name", sorted(GOLD["tagged"]))
def test_tag_frame_matches_lamejs(oracle, name):
    c = GOLD["tagged"][name]
    l, r = _sig(c)
    data, sizes, info = oracle.encode_stream_tagged(c["channels"], c["samplerate"], c["kbps"], l, r, chunk=c["chunk"] or None)
    plain, psizes, _ = oracle.encode_stream(c["channels"], c["samplerate"], c["kbps"], l, r, chunk=c["chunk"] or None)
    assert info["tag_on"] == c["write_tag"]
    assert info["music_crc"] == c["music_crc"] and info["bytes_written"] == c["bytes_written"] == len(plain)
    assert info["encoder_padding"] == c["encoder_padding"]
    if not c["write_tag"]:            # InitVbrTag: the frame cannot hold the tag (VBRTag.js:508-513)
        assert data == plain and info["tag"] == b"" and c["tag_ret"] == 0
        assert hashlib.sha256(data).hexdigest() == c["sha256"]
        return
    tfs = len(info["tag"])
    assert tfs == int(c["total_frame_size"])                       # Java: integer quotient
    assert data[tfs:] == plain and data[:4] == bytes.fromhex(c["first_bytes"])[:4] and not any(data[4:tfs])
    assert sizes[0] == psizes[0] + tfs and sizes[1:] == psizes[1:]
    if c["total_frame_size"] == tfs:                               # integer frame size: the JavaScript stream is the same stream
        assert hashlib.sha256(data).hexdigest() == c["sha256"] and sizes == c["sizes"]
    assert info["frames"] == c["frames"] and c["sum"] == c["frames"] * c["preset"]
    js = bytes.fromhex(c["tag"])
    m = c["sideinfo_len"]
    tag = info["tag"]
    assert tag[m:m + 4] == b"Info" and tag[m + 120:m + 129] == b"LAME3.98r"
    ours_as_js, v = _js_view(tag, js, m)
    crc_at = m + 116 + 38
    if c["frames"] < 400:
        # every byte JavaScript computes the way Java does is the same byte (header, flags, counts, TOC, LAME fields, music CRC)
        assert ours_as_js[:crc_at] == js[:crc_at]
        # ... and so is the tag CRC once the string bytes are what JavaScript wrote
        crc = oracle.crc16(bytes(ours_as_js[:crc_at]))
        assert bytes([crc >> 8, crc & 255]) == js[crc_at:crc_at + 2]
    else:
        # > 400 frames: `bag[i / 2]` (VBRTag.js:161-163) does not compact the bag in JavaScript; only the TOC may differ
        toc = slice(m + 16, m + 116)
        assert ours_as_js[:toc.start] == js[:toc.start] and ours_as_js[toc.stop:crc_at] == js[toc.stop:crc_at]
        t = tag[toc]
        assert all(t[i] <= t[i + 1] for i in range(99)) and t[0] == 0
    crc = oracle.crc16(tag[:crc_at])
    assert tag[crc_at:crc_at + 2] == bytes([crc >> 8, crc & 255]) and not any(tag[crc_at + 2:])


def test_tag_fields_decode(oracle):
    """Independent read-back of the frame (the layout every Xing / LAME tag reader uses)."""
    l, r = make_signal("noise", 70 * 1152, 44100, seed=77)
    data, _, info = oracle.encode_stream_tagged(2, 44100, 128, l, r, chunk=1152)
    tag = info["tag"]
    assert len(tag) == 417 and tag[:4] == bytes([0xFF, 0xFB, 0x90, 0x04])
    x = 4 + 32
    assert tag[x:x + 4] == b"Info" and int.from_bytes(tag[x + 4:x + 8], "big") == 0xF
    frames, nbytes = int.from_bytes(tag[x + 8:x + 12], "big"), int.from_bytes(tag[x + 12:x + 16], "big")
    assert frames == info["frames"] and nbytes == len(data) == info["bytes_written"] + 417
    toc = tag[x + 16:x + 116]
    assert toc[0] == 0 and toc[50] in (127, 128, 129)
    lame = x + 116
    assert int.from_bytes(tag[lame:lame + 4], "big") == 57 and tag[lame + 4:lame + 13] == b"LAME3.98r"
    assert tag[lame + 13] == 1 and tag[lame + 14] == 170              # CBR, lowpass 17000 Hz
    delay = (tag[lame + 25] << 4) | (tag[lame + 26] >> 4)
    padding = ((tag[lame + 26] & 15) << 8) | tag[lame + 27]
    assert delay == 576 and padding == info["encoder_padding"]
    assert (70 * 1152 + delay + padding) % 1152 == 0 and (70 * 1152 + delay + padding) // 1152 == frames
    assert int.from_bytes(tag[lame + 32:lame + 36], "big") == nbytes
    assert int.from_bytes(tag[lame + 36:lame + 38], "big") == oracle.crc16(data[417:])


@pytest.mark.parametrize("name", sorted(GOLD["wav"]))
def test_wav_header_matches_lamejs(oracle, name):
    c = GOLD["wav"][name]
    b, want = bytes.fromhex(c["hex"]), c["result"]
    if "throws" in want:
        with pytest.raises(IndexError if want["throws"] == "RangeError" else ValueError):
            oracle.wav_read_header(b)
    elif "undefined" in want:
        assert oracle.wav_read_header(b) is None
    else:
        assert oracle.wav_read_header(b) == want


def _engine_pcm(c):
    """Uniform PCM in [-20000, 20000), drawn as tests/golden/make_lamejs_seeded_golden.py drew it."""
    rng = np.random.default_rng(c["pcm_seed"])
    l = rng.integers(-20000, 20000, c["samples"]).astype(np.int16)
    r = rng.integers(-20000, 20000, c["samples"]).astype(np.int16) if c["channels"] == 2 else None
    return l, r


def test_live_against_the_engine(oracle):
    """Cases drawn at random once (configuration, length, chunking, full-band PCM) and run through lamejs: hot-path bytes,
    music CRC and byte count, and the tag frame."""
    assert len(ENGINE) >= 8
    for c in ENGINE:
        ch, sr, kbps, n, chunk = c["channels"], c["samplerate"], c["kbps"], c["samples"], c["chunk"]
        l, r = _engine_pcm(c)
        enc = oracle.OracleEncoder(ch, sr, kbps)
        out = bytearray()
        for i in range(0, n, chunk):
            out += enc.encode_buffer(l[i:i + chunk], None if r is None else r[i:i + chunk])
        out += enc.flush()
        assert hashlib.sha256(bytes(out)).hexdigest() == c["sha256"], (ch, sr, kbps, n, chunk)
        assert enc.music_crc() == c["music_crc"] and enc.bytes_written() == c["bytes_written"], (ch, sr, kbps, n, chunk)
        enc.close()
        _, _, info = oracle.encode_stream_tagged(ch, sr, kbps, l, r, chunk=chunk)
        assert info["tag_on"] == c["write_tag"] and info["music_crc"] == c["tag_crc"] and info["frames"] == c["frames"]
        if info["tag_on"]:
            js = bytes.fromhex(c["tag"])
            t, _ = _js_view(info["tag"], js, c["sideinfo_len"])
            k = c["sideinfo_len"] + 154
            assert len(js) == k and t[:k] == js, (ch, sr, kbps, n, chunk)
