#!/usr/bin/env python
"""Record what the UNMODIFIED reference returns in the parity tests -> tests/golden/reference_parity.json.

The parity tests (test_host_vs_reference.py, test_signal_params.py, test_signal_files.py and
test_oracle.py::test_oracle_vs_compiled_reference_random) run their seeded cases through observe_* functions on an
implementation namespace.  This script runs the same functions on the reference's own Python layer and compiled Cython kernels
(oracle/ref_loader.py; set URH_REFERENCE to the reference checkout) and stores one digest per case (conftest.fingerprint), so
the tests compare against the reference without needing it.

    python tests/golden/make_golden_parity.py
"""
import importlib
import json
import os
import sys
import tempfile
import types
from pathlib import Path

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from conftest import REFERENCE_PARITY, fingerprint  # noqa: E402
from oracle import ref_loader  # noqa: E402


def reference_namespace():
    ns = ref_loader.load_python_layer()
    sf, ut, ai = ref_loader.load_kernels()
    return types.SimpleNamespace(
        ppseq_to_bits=ns.ProtocolAnalyzer(None)._ppseq_to_bits, AI=ns.AutoInterpretation, cai=ai, sf=sf, util=ut,
        Filter=ns.Filter, Modulator=ns.Modulator, modulator_module=importlib.import_module("urh.signalprocessing.Modulator"),
        IQArray=ns.IQArray, RingBuffer=importlib.import_module("urh.util.RingBuffer").RingBuffer, Spectrogram=ns.Spectrogram,
        num_frames=lambda spec, x: spec.stft(x).shape[0], noise_level=ns.AutoInterpretation.detect_noise_level,
        convert_to=lambda x, dst: ns.IQArray(x).convert_to(dst),
        grab_pulse_lens=sf.grab_pulse_lens, afp_demod=sf.afp_demod, get_magnitudes=ut.get_magnitudes), ns


def main():
    import test_host_vs_reference as hv
    import test_oracle
    import test_signal_files as files
    import test_signal_params as params

    ref, ns = reference_namespace()
    obs = {
        "ppseq_to_bits": hv.observe_ppseq_to_bits(ref),
        "plateau_bookkeeping": hv.observe_plateau_bookkeeping(ref),
        "cython_host_helpers": hv.observe_cython_host_helpers(ref),
        "modulator_and_filter_host_logic": hv.observe_modulator_and_filter_host_logic(ref),
        "iq_array_host_logic": hv.observe_iq_array_host_logic(ref),
        "ring_buffer": hv.observe_ring_buffer(ref),
        "spectrogram_geometry": hv.observe_spectrogram_geometry(ref),
        "merge_message_segments_for_ook": hv.observe_merge_message_segments_for_ook(ref),
        "noise_level": hv.observe_noise_level(ref),
        "convert_iq": hv.observe_convert_iq(ref),
        "signal_parameter_setters": params.observe_parameter_setters(ns.Signal),
        "signal_construction_defaults": params.observe_construction_defaults(ns.Signal),
        "signal_edit_operations": params.observe_edit_operations(ns.Signal),
        "oracle_random_kernel_cases": test_oracle.observe_random_kernel_cases(ref),
    }
    with pytest.MonkeyPatch.context() as mp:
        obs["modulator_kernel_calls"] = hv.observe_modulator_kernel_calls(ref, mp)
    with tempfile.TemporaryDirectory() as d:
        for key, path in files.parity_files(Path(d)).items():
            obs[key] = [files.observe(ns.Signal(str(path), "t"))]
    out = {k: [fingerprint(o) for o in v] for k, v in sorted(obs.items())}
    with open(REFERENCE_PARITY, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    for k, v in out.items():
        print("%-40s %d cases" % (k, len(v)))


if __name__ == "__main__":
    main()
