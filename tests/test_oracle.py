"""CPU suite: pin the C/numpy oracle against the golden vectors generated from the unmodified reference
(tests/golden/make_golden.py) and against what the reference's compiled kernels returned on randomised cases
(tests/golden/make_golden_parity.py)."""
import numpy as np
import pytest

from conftest import CAPTURES, assert_matches_reference, bits_equal, load_golden


@pytest.mark.parametrize("name", CAPTURES)
def test_afp_demod_matches_golden(oracle, name):
    g = load_golden("capture_" + name)
    noise = float(g["noise"])
    for mod in ("ASK", "FSK", "PSK"):
        q = oracle.afp_demod(g["iq"], noise, mod, 2)
        assert bits_equal(q, g["qad_" + mod]) == 0, (name, mod)
    assert bits_equal(oracle.afp_demod(g["iq"], noise, "PSK", 4), g["qad_PSK4"]) == 0


@pytest.mark.parametrize("name", CAPTURES)
def test_grab_pulse_lens_matches_golden(oracle, name):
    g = load_golden("capture_" + name)
    m = g["meta"]
    qad = g["qad_" + m["mod"]]
    for key in [k for k in g if k.startswith("pulses_tol")]:
        tol = int(key[len("pulses_tol"):])
        r = oracle.grab_pulse_lens(qad, m["center"], tol, m["mod"], m["sps"], m["bps"], m["spacing"])
        assert np.array_equal(r, g[key]), (name, key)
    r = oracle.grab_pulse_lens(qad, m["center"], m["tol"], m["mod"], m["sps"], 2, 0.1)
    assert np.array_equal(r, g["pulses_bps2"])


@pytest.mark.parametrize("name", CAPTURES)
def test_magnitudes_noise_segments_center(oracle, name):
    g = load_golden("capture_" + name)
    m = g["meta"]
    mags = oracle.get_magnitudes(g["iq"])
    assert np.array_equal(mags[:64], g["mag_head"])
    assert mags.sum() == float(g["mag_sum"])
    assert oracle.detect_noise_level(mags) == float(g["auto_noise"])
    seg = oracle.segment_messages_from_magnitudes(mags, float(g["noise"]))
    assert np.array_equal(np.array(seg, dtype=np.int64).reshape(-1, 2), g["segments"])
    c = oracle.detect_center(g["qad_" + m["mod"]])
    gc = float(g["detect_center"])
    assert (c is None and np.isnan(gc)) or c == gc


def test_modulator_matches_golden(oracle):
    g = load_golden("modulator")
    bits = g["bits"]
    cases = {
        "ask": ("ASK", [0, 100], 1, np.float32), "ask_i8": ("ASK", [0, 100], 1, np.int8),
        "fsk": ("FSK", [-10e3, 10e3], 1, np.float32), "fsk4": ("FSK", [-20e3, -10e3, 10e3, 20e3], 2, np.float32),
        "fsk_i16": ("FSK", [-10e3, 10e3], 1, np.int16),
        "psk": ("PSK", [-90, 90], 1, np.float32), "psk4": ("PSK", [-135, -45, 45, 135], 2, np.float32),
        "oqpsk": ("OQPSK", [-135, -45, 45, 135], 2, np.float32),
        "gfsk": ("GFSK", [-10e3, 10e3], 1, np.float32), "gfsk_i8": ("GFSK", [-10e3, 10e3], 1, np.int8),
    }
    import math
    for name, (mt, params, bps, dt) in cases.items():
        a = 1 * (1 if dt == np.float32 else np.iinfo(dt).max)
        p = params
        if mt == "ASK":
            p = [a * x / 100 for x in params]
        elif mt in ("PSK", "OQPSK") and mt == "PSK":
            p = [x * (math.pi / 180) for x in params]
        for suffix, b, pause, start in (("", bits, 77, 0), ("_start5", bits[:32], 3, 5)):
            r = oracle.modulate_c(b, 50, mt, np.array(p, dtype=np.float32), bps, a, 40e3, 30 * (np.pi / 180), 1e6, pause, start, dt)
            ref = g["mod_" + name + suffix]
            assert r.dtype == ref.dtype and r.shape == ref.shape
            if np.issubdtype(ref.dtype, np.integer):
                assert np.array_equal(r, ref), name + suffix
            else:
                assert bits_equal(r, ref) == 0, name + suffix


def test_filters_match_golden(oracle):
    g = load_golden("filters")
    assert bits_equal(oracle.fir_filter(g["x"], g["taps"]).view(np.float32), g["fir"].view(np.float32)) == 0
    assert bits_equal(oracle.fir_filter(g["x"], np.array([0.1] * 10, np.complex64)).view(np.float32), g["fir_ma10"].view(np.float32)) == 0
    assert np.array_equal(oracle.fir_filter(g["kat_in"], np.array([0.25] * 4, np.complex64)), g["kat_out"])
    assert np.array_equal(g["kat_out"], np.array([0.25, 0.75, 1.5, 2.5, 3.5, 4.5, 5.5, 6.5, 7.5, 16.5], dtype=np.complex64))
    assert np.array_equal(oracle.design_windowed_sinc_bandpass(0.03, 0.07, 0.04), g["bandpass_taps"])
    assert np.array_equal(oracle.apply_bandpass_filter(g["x"][:300], 0.03, 0.07, 0.2), g["bandpass_direct"])
    assert np.array_equal(oracle.apply_bandpass_filter(g["x"], 0.03, 0.07, 0.04), g["bandpass_fft"])
    assert bits_equal(oracle.spectrogram_db(g["x"]), g["spec_db"]) == 0
    assert bits_equal(oracle.spectrogram_db(g["x"][:300]), g["short_db"]) == 0


def observe_random_kernel_cases(impl):
    """Randomised digitizer / demod / magnitude cases on an implementation of the three kernels"""
    rng = np.random.default_rng(7)
    out = []
    for trial in range(60):
        n = int(rng.integers(1, 3000))
        mod = ["ASK", "FSK", "PSK"][trial % 3]
        noise_v = 0.0 if mod == "ASK" else -4.0
        base = np.repeat(rng.standard_normal(n // 7 + 1), 7)[:n] * 0.5
        x = (base + 0.2 * rng.standard_normal(n)).astype(np.float32)
        x[rng.random(n) < 0.1] = noise_v
        s = int(rng.integers(0, n))
        x[s: s + int(rng.integers(0, 40))] = noise_v
        tol = int(rng.integers(0, 8))
        bps = int(rng.integers(1, 3))
        out.append(np.asarray(impl.grab_pulse_lens(x, 0.05, tol, mod, 20, bps, 0.3)))
    for dt in (np.int8, np.uint8, np.int16, np.uint16, np.float32):
        iq = (rng.standard_normal((777, 2)) * (0.5 if dt == np.float32 else 60)).astype(dt)
        iq[100:120] = 0
        for mod in ("ASK", "FSK", "PSK"):
            q = np.asarray(impl.afp_demod(iq, 0.1 if dt == np.float32 else 12.0, mod, 2), dtype=np.float32)
            q = q[1:] if mod == "PSK" else q      # PSK: the first sample is not defined
            out.append((q.dtype, q.shape, q.tobytes()))
        out.append(np.asarray(impl.get_magnitudes(iq)))
    return out


def test_oracle_vs_compiled_reference_random(oracle):
    """The oracle on randomised cases against what the original project's own compiled kernels returned for them"""
    assert_matches_reference("oracle_random_kernel_cases", observe_random_kernel_cases(oracle))
