"""CPU: the host-side logic of the drop-in layer against the original project's own functions on randomized inputs.  These
functions never touch the GPU: pulses -> bits, plateau / bit-length bookkeeping of estimate(), modulator parameter preparation,
filter design, bit utilities.

Every observe_* function runs one test's seeded cases on an implementation namespace and returns what the test compares, one
entry per case.  The tests run them on this project and compare with the digests that tests/golden/make_golden_parity.py
stored from the same functions run on the original project (reference_namespace() there)."""
import importlib
import types

import numpy as np
import pytest

from conftest import assert_matches_reference


def ours_namespace():
    from oracle import oracle
    from urh_b200.ainterpretation import AutoInterpretation
    from urh_b200.cythonext import auto_interpretation, signal_functions, util
    from urh_b200.signalprocessing.Filter import Filter
    from urh_b200.signalprocessing.IQArray import IQArray
    from urh_b200.signalprocessing.Spectrogram import Spectrogram
    from urh_b200.util.RingBuffer import RingBuffer

    def noise_level(mags):
        # the device only delivers (sum, max) of the 100 end-aligned chunks; here they come from numpy, the decision logic is ours
        n = len(mags)
        chunksize, nchunks = AutoInterpretation._chunking(n)
        tail = mags[n - nchunks * chunksize:].reshape(nchunks, chunksize)   # chunks are taken from the end backwards
        sums = tail.astype(np.float64).sum(axis=1)
        maxs = tail.max(axis=1).astype(np.float64)
        return AutoInterpretation._noise_from_chunk_stats(n, chunksize, sums, maxs, mags.dtype)

    Modulator = importlib.import_module("urh_b200.signalprocessing.Modulator")
    return types.SimpleNamespace(
        # the sequential CPU restatement of ProtocolAnalyzer._ppseq_to_bits lives in the test oracle, not in the product
        ppseq_to_bits=oracle.ppseq_to_bits, AI=AutoInterpretation, cai=auto_interpretation, sf=signal_functions, util=util,
        Filter=Filter, Modulator=Modulator.Modulator, modulator_module=Modulator, IQArray=IQArray, RingBuffer=RingBuffer,
        Spectrogram=Spectrogram, num_frames=lambda spec, x: spec._num_frames(len(x)), noise_level=noise_level,
        convert_to=oracle.convert_iq)


@pytest.fixture(scope="module")
def ours():
    return ours_namespace()


def observe_ppseq_to_bits(impl):
    rng = np.random.default_rng(5)
    out = []
    for trial in range(300):
        bps = int(rng.choice([1, 2]))
        pt = int(rng.choice([8, 0, 2]))
        sps = int(rng.choice([1, 3, 10, 100]))
        k = int(rng.integers(1, 80))
        kinds = rng.integers(-1, 1 << bps, k)
        ns = np.where(rng.random(k) < 0.15, rng.integers(9, 30, k) * sps, rng.integers(0, 5 * sps + 1, k))
        rows = np.stack([kinds, ns], axis=1).astype(np.int64)
        wp = bool(trial % 2)
        r = impl.ppseq_to_bits(rows, sps, bps, write_bit_sample_pos=wp, pause_threshold=pt)
        out.append(([list(x) for x in r[0]], list(r[1]), [list(x) for x in r[2]]))
    return out


def observe_plateau_bookkeeping(impl):
    AI = impl.AI
    rng = np.random.default_rng(9)
    out = []
    for trial in range(300):
        n = int(rng.integers(2, 60))
        base = int(rng.choice([8, 40, 100, 300]))
        pl = (rng.integers(1, 6, n) * base + rng.integers(-base // 8 - 1, base // 8 + 2, n)).clip(1)
        if trial % 3 == 0:
            pl[rng.integers(0, n, max(1, n // 6))] = rng.integers(1, 4, max(1, n // 6))   # tiny glitches
        pl = pl.astype(np.uint64)
        rec = {"tolerance": AI.estimate_tolerance_from_plateau_lengths(pl)}
        for tol in (None, 0, 1, 3):
            rec["merge_%s" % tol] = list(AI.merge_plateau_lengths(pl, tolerance=tol))
        merged = AI.merge_plateau_lengths(pl)
        if len(merged) >= 2:
            rec["bit_length"] = AI.get_bit_length_from_plateau_lengths(merged)
        a = [int(v) for v in pl]
        AI.round_plateau_lengths(a)       # in place
        rec["rounded"] = a
        rec["gcd"] = AI.get_tolerant_greatest_common_divisor(list(pl))
        vals = [int(v) for v in rng.integers(0, 6, n)]
        rec["most_frequent"] = AI.get_most_frequent_value(vals)
        data = rng.standard_normal(n + 3) * 10 + 50
        rec["max"], rec["min"] = AI.max_without_outliers(data), AI.min_without_outliers(data)
        out.append(rec)
    return out


def observe_cython_host_helpers(impl):
    rng = np.random.default_rng(2)
    out = []
    for trial in range(200):
        n = int(rng.integers(1, 80))
        pl = rng.integers(1, 400, n).astype(np.uint64)
        tol, mc = int(rng.integers(0, 12)), int(rng.integers(1, 40))
        rec = {"merge": list(np.asarray(impl.cai.merge_plateaus(pl, tol, mc))),
               "hist": list(np.asarray(impl.cai.get_threshold_divisor_histogram(pl)))}
        if trial % 10 == 0:   # long tables with repeated values and zeros (a message of thousands of rounded plateaus)
            big = (rng.integers(0, 7, 3000) * int(rng.choice([10, 100, 300])) + (rng.integers(0, 3, 3000) if trial % 20 else 0)).astype(np.uint64)
            if big.max() == 0:
                big[0] = 5
            rec["hist_big"] = np.asarray(impl.cai.get_threshold_divisor_histogram(big))
        bits = rng.integers(0, 2, int(rng.integers(0, 40))).astype(np.uint8)
        rec["oqpsk"] = list(np.asarray(impl.sf.get_oqpsk_bits(bits)))
        if len(bits):
            a, b = sorted(rng.integers(0, len(bits) + 1, 2))
            rec["number"] = impl.util.bit_array_to_number(bits, int(b), int(a))
        out.append(rec)
    return out


def observe_modulator_and_filter_host_logic(impl):
    F = impl.Filter
    out = []
    for bw in (0.001, 0.04, 0.08, 0.42):
        N = F.get_filter_length_from_bandwidth(bw)
        rec = {"length": N, "bandwidth": F.get_bandwidth_from_filter_length(N)}
        if N < 2000:
            rec["lpf"] = F.design_windowed_sinc_lpf(0.1, bw)
            rec["bandpass"] = F.design_windowed_sinc_bandpass(-0.1, 0.2, bw)
        out.append(rec)
    for mod in ("ASK", "FSK", "PSK", "GFSK", "OQPSK"):
        for bps in ((1, 2, 3) if mod != "OQPSK" else (2,)):
            m = impl.Modulator("m")
            m.modulation_type = mod
            m.bits_per_symbol = bps
            m.sample_rate = 2e6
            out.append((list(m.get_default_parameters()), m.modulation_order, m.is_binary_modulation,
                        m.is_amplitude_based, m.is_frequency_based, m.is_phase_based))
    return out


def observe_iq_array_host_logic(impl):
    IQ = impl.IQArray
    rng = np.random.default_rng(4)
    out = [IQ.min_max_for_dtype(dt) for dt in (np.int8, np.uint8, np.int16, np.uint16, np.float32)]
    c = (rng.standard_normal(10) + 1j * rng.standard_normal(10)).astype(np.complex64)
    for arr in (c, c.astype(np.complex128), rng.standard_normal(20).astype(np.float32), rng.integers(-100, 100, (10, 2)).astype(np.int16),
                rng.integers(0, 255, 20).astype(np.uint8)):
        a = IQ(arr)
        out.append((IQ.convert_array_to_iq(arr), a.num_samples, a.dtype, a.minimum, a.maximum, a.real, a.imag))
    return out


def observe_ring_buffer(impl):
    """util/RingBuffer.py: push / pop / wrap-around / clear on randomized traffic"""
    rng = np.random.default_rng(6)
    out = []
    for dtype in (np.float32, np.int8):
        ring = impl.RingBuffer(size=64, dtype=dtype)
        for step in range(300):
            rec = []
            if rng.random() < 0.55:
                k = int(rng.integers(1, 40))
                vals = (rng.standard_normal((k, 2)) * 50).astype(dtype)
                rec.append(ring.will_fit(k))
                if ring.will_fit(k):
                    ring.push(impl.IQArray(vals.copy()))
            else:
                k = int(rng.integers(1, 50))
                rec.append(np.asarray(ring.pop(k, ensure_even_length=bool(step % 2))))
            rec += [ring.left_index, ring.right_index, ring.space_left, ring.is_empty, len(ring), np.asarray(ring.view_data)]
            out.append(rec)
            if step % 97 == 0:
                ring.clear()
    return out


def observe_modulator_kernel_calls(impl, monkeypatch):
    """Modulator.modulate: the arguments handed to modulate_c (the kernel is replaced by a recorder, so no GPU and no Cython code
    runs), and the shape and dtype of what modulate returns"""
    calls = []

    def fake(bits, sps, mod_type, parameters, bps, a, f, phi, sr, pause, start, dtype=np.float32, gauss_bt=0.5, filter_width=1.0):
        calls.append((list(bits), sps, mod_type, [float(p) for p in parameters], bps, float(a), float(f), float(phi), float(sr),
                      pause, start, np.dtype(dtype), float(gauss_bt), float(filter_width)))
        total = (len(bits) // bps) * sps + pause
        return np.zeros((total, 2), dtype=dtype)

    monkeypatch.setattr(impl.modulator_module.signal_functions, "modulate_c", fake)
    rng = np.random.default_rng(12)
    out = []
    for mod in ("ASK", "FSK", "PSK", "GFSK"):
        for trial in range(6):
            m = impl.modulator_module.Modulator("t")
            bps = int(rng.choice([1, 2]))
            cfg = dict(modulation_type=mod, bits_per_symbol=bps, samples_per_symbol=int(rng.choice([8, 100])), sample_rate=float(rng.choice([1e6, 2e6])),
                       carrier_freq_hz=float(rng.choice([0.0, 20e3])), carrier_amplitude=float(rng.choice([1.0, 0.5])),
                       carrier_phase_deg=float(rng.choice([0.0, 45.0])), gauss_bt=0.5, gauss_filter_width=1.0)
            for k_, v in cfg.items():
                setattr(m, k_, v)
            m.parameters = m.get_default_parameters()
            nbits = int(rng.integers(0, 12)) * bps
            data = [int(b) for b in rng.integers(0, 2, nbits)]
            payload = "".join(map(str, data)) if trial % 2 else list(data)
            pause, start = int(rng.integers(0, 50)), int(rng.integers(0, 1000))
            dtype = [None, np.int8, np.int16, np.float32][trial % 4]
            n_calls = len(calls)
            a = m.modulate(payload, pause=pause, start=start, dtype=dtype)
            out.append((a.data.shape, a.dtype, calls[n_calls:]))
    return out


def observe_spectrogram_geometry(impl):
    """Spectrogram.py: hop size, bin counts and the number of STFT frames (the original's frame count is the shape of its strided
    view; ours is computed up front to size the device buffers)"""
    rng = np.random.default_rng(1)
    out = []
    for trial in range(40):
        n = int(rng.integers(1, 5000))
        w = int(rng.choice([16, 64, 256, 1024]))
        ov = float(rng.choice([0.5, 0.0, 0.75, 0.3]))
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        a = impl.Spectrogram(x, window_size=w, overlap_factor=ov)
        out.append((a.hop_size, a.time_bins, a.freq_bins, impl.num_frames(a, x)))
    return out


def observe_merge_message_segments_for_ook(impl):
    rng = np.random.default_rng(21)
    out = [impl.AI.merge_message_segments_for_ook([])]
    for trial in range(300):
        k = int(rng.integers(1, 25))
        pos = 0
        segs = []
        pulse = int(rng.choice([20, 100, 400]))
        for _ in range(k):
            pos += int(rng.choice([pulse // 2, pulse, 3 * pulse, 9 * pulse, 40 * pulse])) + int(rng.integers(0, 5))
            length = int(rng.integers(1, 4)) * pulse + int(rng.integers(0, 7))
            segs.append((pos, pos + length))
            pos += length
        out.append(impl.AI.merge_message_segments_for_ook(list(segs)))
    return out


def observe_noise_level(impl):
    """detect_noise_level (AutoInterpretation.py) on bursts, signal everywhere and silence"""
    rng = np.random.default_rng(14)
    out = []
    for trial in range(200):
        n = int(rng.integers(4, 40000))
        dtype = np.float64 if trial % 2 else np.float32
        mags = np.abs(rng.standard_normal(n) * 0.01)
        kind = trial % 5
        if kind < 3:
            a = int(rng.integers(0, n))
            mags[a: a + n // 3] += rng.uniform(0.3, 1.0)          # a burst
        elif kind == 3:
            mags += 0.5                                            # signal everywhere: chunk means nearly equal -> 0
        else:
            mags[:] = 0.0
        out.append(impl.noise_level(mags.astype(dtype)))
    return out


def observe_convert_iq(impl):
    rng = np.random.default_rng(5)
    types_ = [np.int8, np.uint8, np.int16, np.uint16, np.float32]
    out = []
    for src in types_:
        if src == np.float32:
            x = np.concatenate([rng.uniform(-1, 1, 4000), [-1.0, 1.0, 0.0, -0.0, 0.999999, -0.999999]]).astype(np.float32)
        else:
            info = np.iinfo(src)
            x = np.concatenate([rng.integers(info.min, info.max + 1, 4000), [info.min, info.max, 0, 1]]).astype(src)
        x = np.ascontiguousarray(x.reshape(-1, 2))
        for dst in types_:
            a = impl.convert_to(x, dst)
            out.append((a.dtype, a.shape, a.tobytes()))
    return out


def test_ppseq_to_bits_port(ours):
    assert_matches_reference("ppseq_to_bits", observe_ppseq_to_bits(ours))


def test_plateau_bookkeeping(ours):
    assert_matches_reference("plateau_bookkeeping", observe_plateau_bookkeeping(ours))


def test_cython_host_helpers(ours):
    assert_matches_reference("cython_host_helpers", observe_cython_host_helpers(ours))


def test_modulator_and_filter_host_logic(ours):
    assert_matches_reference("modulator_and_filter_host_logic", observe_modulator_and_filter_host_logic(ours))


def test_iq_array_host_logic(ours):
    assert_matches_reference("iq_array_host_logic", observe_iq_array_host_logic(ours))
    for name in ("x.complex", "x.cs8", "x.complex16u", "x.cu16", "x.complex32s", "x.wav"):
        exp = {"x.complex": np.float32, "x.cs8": np.int8, "x.complex16u": np.uint8, "x.cu16": np.uint16, "x.complex32s": np.int16, "x.wav": np.float32}[name]
        assert ours.IQArray._dtype_for_filename(name) == exp


def test_ring_buffer(ours):
    assert_matches_reference("ring_buffer", observe_ring_buffer(ours))


def test_modulator_prepares_the_same_kernel_call(ours, monkeypatch):
    obs = observe_modulator_kernel_calls(ours, monkeypatch)
    assert sum(len(calls) for _, _, calls in obs) > 0
    assert_matches_reference("modulator_kernel_calls", obs)


def test_spectrogram_geometry(ours):
    assert_matches_reference("spectrogram_geometry", observe_spectrogram_geometry(ours))


def test_merge_message_segments_for_ook(ours):
    assert_matches_reference("merge_message_segments_for_ook", observe_merge_message_segments_for_ook(ours))


def test_noise_level_decision_from_chunk_statistics(ours):
    assert_matches_reference("noise_level", observe_noise_level(ours))


def test_oracle_convert_iq_is_the_references_convert_to(ours, oracle):
    """closes the chain for the format conversions: the original's IQArray.convert_to == oracle.convert_iq (here) == convert.cu
    (tests/test_gpu_objects.py::test_convert_to_all_pairs)"""
    assert_matches_reference("convert_iq", observe_convert_iq(ours))
