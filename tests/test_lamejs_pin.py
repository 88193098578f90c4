"""The pin against the reference itself.  tests/golden/lamejs_golden.json holds SHA-256 / length / per-call sizes
of the bytes REAL lamejs produced (unmodified lamejs executed by Qt's QJSEngine, see tools/jsrun/ and
tests/golden/make_lamejs_golden.py).  The oracle must reproduce every fixture it supports on CPU; the CUDA path must
reproduce them through the C-ABI on the B200.  tests/golden/lamejs_seeded_golden.json (make_lamejs_seeded_golden.py)
adds lamejs's bytes for seeded random configurations, for its three loaders, and its intermediates of one more input."""
import hashlib
import json
import os

import numpy as np
import pytest

from synth import make_signal

HERE = os.path.dirname(os.path.abspath(__file__))
_GOLD = json.load(open(os.path.join(HERE, "golden", "lamejs_golden.json")))
FIX = _GOLD["cases"]
TAPS = _GOLD["taps"]     # lamejs's own intermediates (SHA-256 per array): MDCT spectrum, masking, block types, quantised lines ...
SEEDED = json.load(open(os.path.join(HERE, "golden", "lamejs_seeded_golden.json")))


def _supported(oracle, c):
    try:
        e = oracle.OracleEncoder(c["channels"], c["samplerate"], c["kbps"])
    except ValueError:
        return False
    e.close()
    return True


def _check(c, data, sizes):
    assert len(data) == c["bytes"]
    assert data[:48].hex() == c["head"]
    assert hashlib.sha256(data).hexdigest() == c["sha256"]
    if sizes is not None:
        assert len(sizes) == c["calls"]
        assert hashlib.sha256(json.dumps([int(s) for s in sizes]).encode()).hexdigest() == c["sizes_sha256"]


NAMES = sorted(k for k, v in FIX.items() if "error" not in v)


def test_fixture_inventory():
    assert len(NAMES) >= 250 and not [k for k, v in FIX.items() if "error" in v]


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_lamejs(oracle, name):
    c = FIX[name]
    if not _supported(oracle, c):
        pytest.skip("configuration needs the resampler / MPEG-2 row")
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    data, sizes, _ = oracle.encode_stream(c["channels"], c["samplerate"], c["kbps"], l, r if c["channels"] == 2 else None,
                                          chunk=c["chunk"] or None)
    _check(c, data, sizes)


def test_oracle_supports_every_native_rate_fixture(oracle):
    """No silent skips: every MPEG-1 configuration without resampling must be checked above."""
    n = sum(1 for k in NAMES if _supported(oracle, FIX[k]))
    assert n >= 70, n


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_matches_lamejs(name):
    import lamejs_b200 as M

    c = FIX[name]
    try:
        enc = M.Mp3Encoder(c["channels"], c["samplerate"], c["kbps"])
    except M.Mp3B200Error:
        pytest.skip("configuration needs the resampler / MPEG-2 row")
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    n = len(l)
    step = c["chunk"] or max(n, 1)
    out, sizes = bytearray(), []
    for i in range(0, n, step):
        b = enc.encodeBuffer(l[i:i + step], r[i:i + step] if c["channels"] == 2 else None)
        sizes.append(len(b))
        out += b
    b = enc.flush()
    sizes.append(len(b))
    out += b
    enc.close()
    _check(c, bytes(out), sizes)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_live_lamejs_on_random_inputs(oracle, seed):
    """Inputs drawn at random once: configuration, signal kind, length and chunking (make_lamejs_seeded_golden.py)."""
    c = SEEDED["random_inputs"][str(seed)]
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    got, sizes, _ = oracle.encode_stream(c["channels"], c["samplerate"], c["kbps"], l, r if c["channels"] == 2 else None,
                                         chunk=c["chunk"] or None)
    _check(c, got, sizes)


def test_loader_and_libm_independence(oracle):
    """lame.all.js and the src/js modules gave the same bytes; so did swapping the engine's libm for fdlibm; the oracle
    reproduces them."""
    c = SEEDED["loaders"]
    assert c["bundle"] == c["modules"] == c["fdlibm"]
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    data, _, _ = oracle.encode_stream(c["channels"], c["samplerate"], c["kbps"], l, r)
    assert hashlib.sha256(data).hexdigest() == c["bundle"]


def _tap_hash(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("name", sorted(TAPS))
def test_oracle_intermediates_match_lamejs(oracle, name):
    """Not only the bytes: the MDCT spectrum, the masking energies / thresholds (float32 bit patterns), block types, ATH
    adjustment, quantised lines and side info that REAL lamejs held in every frame (recorded through two one-line hooks,
    tools/jsrun/ref_lamejs.encode_with_taps) equal the oracle's trace bit for bit."""
    c = TAPS[name]
    ch, G = c["channels"], c["granules"]
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    data, _, tr = oracle.encode_stream(ch, c["samplerate"], c["kbps"], l, r if ch == 2 else None, trace_frames=c["frames"] + 2)
    assert hashlib.sha256(data).hexdigest() == c["sha256"] and len(tr) == c["frames"]
    for k, want in c["taps"].items():
        a = tr[k] if k == "ath_adjust" else tr[k][:, :G, :ch]
        assert _tap_hash(a) == want, k


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TAPS))
def test_gpu_intermediates_match_lamejs(name):
    """The CUDA stage taps against lamejs's own intermediates directly (no oracle in between): relative tolerance 0."""
    import lamejs_b200 as M

    c = TAPS[name]
    ch = c["channels"]
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    g = M.debug_stages(ch, c["samplerate"], c["kbps"], l, r if ch == 2 else None,
                       want=("xr", "blocktype", "en_l", "thm_l", "en_s", "thm_s", "ath_adjust", "l3_enc", "ginfo", "bytes"))
    assert hashlib.sha256(g["bytes"].tobytes()).hexdigest() == c["sha256"]
    gi = {k: g["ginfo"][..., j] for j, k in enumerate(["global_gain", "part2_3_length", "part2_length", "big_values", "count1", "scalefac_compress"])}
    for k, want in c["taps"].items():
        a = gi[k] if k in gi else g[k]
        assert _tap_hash(a) == want, k


def test_live_intermediates_on_a_random_input(oracle):
    c = SEEDED["taps"]
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    data, _, tr = oracle.encode_stream(c["channels"], c["samplerate"], c["kbps"], l, r, trace_frames=40)
    assert hashlib.sha256(data).hexdigest() == c["sha256"] and len(tr) == c["frames"]
    for k, want in c["taps"].items():
        a = tr[k] if k == "ath_adjust" else tr[k][:, :2, :2]
        assert _tap_hash(a) == want, k
