"""CPU: the parameter setters of urh_b200.signalprocessing.Signal (one descriptor table) behave like the original project's
hand-written properties (Signal.py:215-400): same values, same events in the same order with the same arguments, same
invalidation of the cached demodulation.  The observe_* functions run the cases on a Signal class; the tests compare this
project's results with the digests tests/golden/make_golden_parity.py stored from the original's Signal."""
import numpy as np

from conftest import assert_matches_reference

EVENTS = ("samples_per_symbol_changed", "tolerance_changed", "noise_threshold_changed", "center_changed",
          "center_spacing_changed", "name_changed", "sample_rate_changed", "modulation_type_changed",
          "bits_per_symbol_changed", "protocol_needs_update")


class Recorder(object):
    def __init__(self, log, name):
        self.log, self.name = log, name

    def emit(self, *args):
        self.log.append((self.name, tuple(args)))

    def connect(self, *a, **k):
        pass


def instrument(sig):
    log = []
    for e in EVENTS:
        setattr(sig, e, Recorder(log, e))
    return log


SCRIPT = [
    ("tolerance", 5), ("tolerance", 7), ("tolerance", 7.9), ("tolerance", "9"),
    ("samples_per_symbol", 100), ("samples_per_symbol", 250), ("samples_per_symbol", 250),
    ("modulation_type", "FSK"), ("modulation_type", "ASK"), ("modulation_type", "PSK"), ("modulation_type", "PSK"),
    ("bits_per_symbol", 1), ("bits_per_symbol", 2), ("bits_per_symbol", 2.0), ("bits_per_symbol", 3),
    ("center", 0), ("center", 0.25), ("center", 0.25), ("center", -1e-3),
    ("center_spacing", 1), ("center_spacing", 0.5),
    ("pause_threshold", 8), ("pause_threshold", 0), ("pause_threshold", 0),
    ("message_length_divisor", 1), ("message_length_divisor", 4),
    ("costas_loop_bandwidth", 0.1), ("costas_loop_bandwidth", 0.05),
    ("name", "x"), ("name", "renamed"), ("name", "renamed"),
    ("sample_rate", 1e6), ("sample_rate", 2e6),
    ("block_protocol_update", True), ("tolerance", 3), ("modulation_type", "FSK"), ("center", 0.5), ("block_protocol_update", False),
    ("samples_per_symbol", 40), ("timestamp", 12.5),
]


def observe_parameter_setters(Signal):
    sig = Signal("", "x", sample_rate=1e6)
    log = instrument(sig)
    out = []
    for attr, value in SCRIPT:
        sig._qad = np.zeros(3, np.float32)   # a cached demodulation that the setter may have to drop
        setattr(sig, attr, value)
        rec = [sig._qad is None]
        if attr != "block_protocol_update":
            v = getattr(sig, attr)
            rec += [v, type(v).__name__]
        out.append(rec)
    out.append(log)
    out.append(sig.modulation_order)
    return out


def observe_construction_defaults(Signal):
    out = []
    for kw in (dict(), dict(modulation="ASK", sample_rate=250e3, timestamp=3.0)):
        sig = Signal("", "n", **kw)
        out.append([getattr(sig, attr) for attr in ("name", "tolerance", "samples_per_symbol", "pause_threshold", "message_length_divisor",
                                                    "costas_loop_bandwidth", "center", "sample_rate", "bits_per_symbol", "center_spacing",
                                                    "modulation_type", "timestamp", "noise_threshold", "already_demodulated",
                                                    "modulation_order")])
        out.append(sig.parameter_cache)
    return out


def observe_edit_operations(Signal):
    """insert / delete / mute / crop (Signal.py:613-651) on host data: samples, cached demodulation, flags"""
    rng = np.random.default_rng(8)
    out = []
    for trial in range(20):
        n = int(rng.integers(20, 200))
        iq = rng.integers(-100, 100, (n, 2)).astype(np.int16) if trial % 2 else rng.standard_normal((n, 2)).astype(np.float32)
        s = Signal.from_samples(iq.copy(), "e", 1e6)
        s._qad = rng.standard_normal(n).astype(np.float32)
        s.parameter_cache["FSK"]["center"] = 0.5
        a, b = sorted(int(v) for v in rng.integers(0, n, 2))
        op = trial % 4
        if op == 0:
            s.mute_range(a, b)
        elif op == 1:
            s.delete_range(a, b)
        elif op == 2:
            s.crop_to_range(a, max(b, a + 1))
        else:
            s.insert_data(a, iq[:5].copy())
        out.append([s.iq_array.data, s._qad is None, s._qad, s.changed, s.num_samples, s.parameter_cache])
    return out


def test_parameter_setters_match_reference():
    from urh_b200.signalprocessing.Signal import Signal

    obs = observe_parameter_setters(Signal)
    assert obs[-1] == 8
    assert_matches_reference("signal_parameter_setters", obs)


def test_construction_defaults_match_reference():
    from urh_b200.signalprocessing.Signal import Signal

    assert_matches_reference("signal_construction_defaults", observe_construction_defaults(Signal))


def test_edit_operations_match_reference():
    from urh_b200.signalprocessing.Signal import Signal

    assert_matches_reference("signal_edit_operations", observe_edit_operations(Signal))
