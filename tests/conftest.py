import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    d = {k: z[k] for k in z.files}
    if "meta" in d:
        d["meta"] = json.loads(str(d["meta"]))
    return d


CAPTURES = ["fsk", "ask", "ask_short", "psk_gen_noisy", "enocean", "FSK10", "homematic", "esaver", "two_participants"]

# What the original project returned in the parity tests, one digest per case (tests/golden/make_golden_parity.py)
REFERENCE_PARITY = os.path.join(GOLDEN, "reference_parity.json")


def _feed(h, x):
    if isinstance(x, dict):
        h.update(b"{%d" % len(x))
        for k in sorted(x, key=repr):
            _feed(h, k)
            _feed(h, x[k])
        return
    if isinstance(x, type):
        x = np.dtype(x) if issubclass(x, np.generic) else x.__name__   # np.float32 == np.dtype("float32")
    if x is None or isinstance(x, (str, bytes, np.dtype)):
        s = x if isinstance(x, bytes) else repr(str(x) if isinstance(x, np.dtype) else x).encode()
        h.update(b"s%d:" % len(s) + s)
        return
    scalar = (int, float, bool, np.number, np.bool_)
    if isinstance(x, (list, tuple)) and not all(isinstance(v, scalar) for v in x):
        h.update(b"[%d" % len(x))
        for v in x:
            _feed(h, v)
        return
    a = np.asarray(x)
    if a.dtype == object or a.ndim > 1:
        _feed(h, list(a))
        return
    if a.dtype.kind == "c":
        h.update(b"c")
        _feed(h, a.real)
        a = a.imag
    h.update(b"n" if a.ndim == 0 else b"v%d" % a.size)
    if a.dtype.kind == "f":
        a = a.astype(np.float64) + 0.0                              # -0.0 == 0.0
        if np.all(np.isfinite(a)) and np.all(a == np.round(a)) and np.all(np.abs(a) < 2.0 ** 62):
            a = a.astype(np.int64)                                  # 3.0 == 3
    if a.dtype.kind == "f":
        h.update(b"f" + np.where(np.isnan(a), np.nan, a).tobytes())
    else:
        h.update(b"i" + a.astype(np.int64).tobytes())


def fingerprint(obj) -> str:
    """Digest of a value as `==` / np.array_equal compare it: numbers by value (1 == 1.0 == np.int64(1)), lists, tuples and
    arrays element by element, dicts by sorted items; strings, bytes and dtypes exactly.  To compare bit patterns and dtypes,
    pass (a.dtype, a.shape, a.tobytes())."""
    h = hashlib.sha256()
    _feed(h, obj)
    return h.hexdigest()[:16]


def assert_matches_reference(key, observations):
    """observations[i] (any value fingerprint() takes) equals what the original project gave for case i"""
    with open(REFERENCE_PARITY) as f:
        want = json.load(f)[key]
    got = [fingerprint(o) for o in observations]
    assert len(got) == len(want), (key, len(got), len(want))
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, "%s: cases %s differ from the original project" % (key, bad[:20])


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as o

    o.build()
    return o


@pytest.fixture(scope="session")
def ctx():
    from urh_b200 import _lib

    return _lib.default_context()


def bits_equal(a: np.ndarray, b: np.ndarray) -> int:
    """number of differing 32-bit words between two float32 arrays (NaN-safe, sign-of-zero aware)"""
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    assert a.shape == b.shape, (a.shape, b.shape)
    return int((a.view(np.uint32) != b.view(np.uint32)).sum())


def synth_fsk(n, sps=100, seed=0, noise_sigma=0.01, gap_every=None, dtype=np.float32):
    """Seeded phase-continuous 2-FSK capture with AWGN and noise-only gaps (SURVEY §8d recipe, small)."""
    rng = np.random.default_rng(seed)
    nsym = n // sps + 1
    bits = rng.integers(0, 2, nsym)
    f = np.repeat(np.where(bits > 0, 0.01, -0.01), sps)[:n]
    phase = 2 * np.pi * np.cumsum(f)
    amp = np.ones(n)
    if gap_every:
        for s in range(gap_every, n, 2 * gap_every):
            amp[s: s + gap_every // 2] = 0.0
    x = amp * np.exp(1j * phase) + noise_sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    iq = np.empty((n, 2), dtype=np.float32)
    iq[:, 0] = x.real
    iq[:, 1] = x.imag
    if dtype == np.float32:
        return iq
    if dtype == np.int8:
        return np.clip(iq * 100, -128, 127).astype(np.int8)
    if dtype == np.uint8:
        return np.clip(iq * 100 + 128, 0, 255).astype(np.uint8)
    if dtype == np.int16:
        return np.clip(iq * 20000, -32768, 32767).astype(np.int16)
    if dtype == np.uint16:
        return np.clip(iq * 20000 + 32768, 0, 65535).astype(np.uint16)
    raise ValueError(dtype)
