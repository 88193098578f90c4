#!/usr/bin/env python3
"""Generates tests/golden/lamejs_seeded_golden.json: what REAL lamejs (unmodified sources under Qt's QJSEngine,
tools/jsrun/) produced for the seeded cross-checks of tests/test_lamejs_pin.py and tests/test_tag_oracle.py, so that
those tests compare the oracle with lamejs on any machine, without the engine or the lamejs sources:

  random_inputs  six seeded draws of configuration, signal kind, length and chunking (bytes and per-call sizes)
  loaders        one burst stream through lame.all.js, through the src/js modules, and with fdlibm's Math
  taps           lamejs's per-frame intermediates (SHA-256 per array) of one burst stream
  engine         eight seeded draws of uniform-noise PCM: the hot path's music CRC / byte count and the Info / LAME tag

  python tests/golden/make_lamejs_seeded_golden.py      # ~1 minute
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tools", "jsrun"))
from synth import make_signal  # noqa: E402


def _sha(b):
    return hashlib.sha256(b).hexdigest()


def _tap_hash(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def random_inputs(R):
    out = {}
    for seed in range(6):
        rng = np.random.default_rng(0xA11CE + seed)
        ch = int(rng.integers(1, 3))
        sr = int(rng.choice([32000, 44100, 48000]))
        kbps = int(rng.choice([128, 160, 192, 224, 256, 320]))
        kind = str(rng.choice(["noise", "white", "octave", "burst"]))
        n = int(rng.integers(5, 40)) * 1152 + int(rng.integers(0, 1152))
        chunk = [None, 1152, int(rng.integers(1, 4000))][int(rng.integers(0, 3))]
        c = dict(channels=ch, samplerate=sr, kbps=kbps, kind=kind, samples=n, seed=1000 + seed, chunk=chunk or 0)
        l, r = make_signal(kind, n, sr, c["seed"])
        data, sizes, _ = R.encode(ch, sr, kbps, l, r, chunk=chunk)
        out[str(seed)] = dict(c, bytes=len(data), head=data[:48].hex(), sha256=_sha(data), calls=len(sizes),
                              sizes_sha256=_sha(json.dumps([int(s) for s in sizes]).encode()))
    return out


def loaders(R):
    c = dict(channels=2, samplerate=44100, kbps=128, kind="burst", samples=30 * 1152, seed=77)
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    for name, kw in (("bundle", {}), ("modules", {"loader": "modules"}), ("fdlibm", {"fdlibm": True})):
        data, _, _ = R.encode(2, 44100, 128, l, r, **kw)
        c[name] = _sha(data)
    return c


def taps(R):
    c = dict(channels=2, samplerate=44100, kbps=128, kind="burst", samples=20 * 1152 + 3, seed=4242)
    l, r = make_signal(c["kind"], c["samples"], c["samplerate"], c["seed"])
    data, t = R.encode_with_taps(2, 44100, 128, l, r)
    c["sha256"] = _sha(data)
    c["frames"] = int(t["xr"].shape[0])
    c["taps"] = {k: _tap_hash(t[k]) for k in ("xr", "en_l", "thm_l", "en_s", "thm_s", "blocktype", "l3_enc", "global_gain", "ath_adjust")}
    return c


def engine_pcm(c):
    """Uniform PCM in [-20000, 20000) of an `engine` case (tests/test_tag_oracle.py draws it the same way)."""
    rng = np.random.default_rng(c["pcm_seed"])
    l = rng.integers(-20000, 20000, c["samples"]).astype(np.int16)
    r = rng.integers(-20000, 20000, c["samples"]).astype(np.int16) if c["channels"] == 2 else None
    return l, r


def engine(T):
    out = []
    for seed in range(8):
        rng = np.random.default_rng(0x7A60 + seed)
        ch = int(rng.integers(1, 3))
        sr, kbps = [(48000, 192), (32000, 96), (44100, 160), (24000, 48), (22050, 64)][int(rng.integers(0, 5))]
        n = int(rng.integers(5, 30)) * 1152 + int(rng.integers(0, 1152))
        chunk = int(rng.integers(500, 6000))
        c = dict(channels=ch, samplerate=sr, kbps=kbps, samples=n, chunk=chunk, pcm_seed=0x7A60 + seed)
        l, r = engine_pcm(c)
        js, crc, nb = T.hot_path_crc(ch, sr, kbps, l, r, chunk=chunk)
        o = T.tagged(ch, sr, kbps, l, r, chunk=chunk)
        k = o["sideinfo_len"] + 154
        out.append(dict(c, sha256=_sha(js), music_crc=crc, bytes_written=nb, write_tag=o["write_tag"], tag_crc=o["crc"],
                        frames=o["frames"], sideinfo_len=o["sideinfo_len"], tag=bytes(o["tag"][:k]).hex()))
    return out


def main():
    import ref_lamejs as R
    import tag_probe as T
    assert R.available(), "needs the lamejs sources and the Qt JavaScript engine (tools/jsrun/)"
    out = {"random_inputs": random_inputs(R), "loaders": loaders(R), "taps": taps(R), "engine": engine(T)}
    with open(os.path.join(HERE, "lamejs_seeded_golden.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print({k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
