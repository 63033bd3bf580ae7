"""CPU: capture files into ``Signal`` (reference: src/urh/signalprocessing/Signal.py:114-213, IQArray.py:206-227) - wav (8 / 16 / 24 /
32 bit, one and two channels), Flipper ``.sub`` run lengths, ``.coco`` archives and the raw sample formats by file extension -
loaded by urh_b200.signalprocessing.Signal: the same samples, dtype, sample rate and already-demodulated flag as the original
project's class gave for the same files (digests stored by tests/golden/make_golden_parity.py).  The noise threshold is fixed
through the settings so that no GPU is needed (with "automatic" the constructor runs detect_noise_level on the device)."""
import tarfile
import wave

import numpy as np
import pytest

from conftest import assert_matches_reference

RAW = [(".complex", np.float32), (".cs8", np.int8), (".complex16s", np.int8), (".cs16", np.int16), (".complex32s", np.int16)]


def make_wav(directory, width, channels):
    rng = np.random.default_rng(10 * width + channels)
    frames, rate = 1234, 48000 if channels == 1 else 250000
    raw = rng.integers(0, 256, frames * channels * width, dtype=np.uint8).tobytes()
    path = directory / ("c%d_w%d.wav" % (channels, width))
    with wave.open(str(path), "w") as f:
        f.setnchannels(channels)
        f.setsampwidth(width)
        f.setframerate(rate)
        f.writeframes(raw)
    return path, rate


def make_flipper_sub(directory):
    path = directory / "remote.sub"
    path.write_text("Filetype: Flipper SubGhz RAW File\nVersion: 1\nFrequency: 433920000\nProtocol: RAW\n"
                    "RAW_Data: 300 -900 300 -300 900 -9000\nRAW_Data: 450 -450 1350 -100\nsomething else: 5\n")
    return path


def make_raw_and_coco(directory, ext, dtype):
    """the raw capture, and the same file inside a .coco archive (Signal.py:190-205)"""
    rng = np.random.default_rng(len(ext))
    n = 777
    if dtype == np.float32:
        data = rng.standard_normal((n, 2)).astype(np.float32)
    else:
        info = np.iinfo(dtype)
        data = rng.integers(info.min, info.max + 1, (n, 2)).astype(dtype)
    path = directory / ("capture" + ext)
    data.tofile(str(path))
    coco = directory / ("capture" + ext.replace(".", "_") + ".coco")
    with tarfile.open(str(coco), "w:bz2") as tar:
        tar.add(str(path), arcname="capture" + ext)
    return path, coco, data


def parity_files(directory):
    """every capture file the tests load, by its key in reference_parity.json"""
    files = {}
    for width in (1, 2, 3, 4):
        for channels in (1, 2):
            files["signal_file_c%d_w%d.wav" % (channels, width)] = make_wav(directory, width, channels)[0]
    files["signal_file_remote.sub"] = make_flipper_sub(directory)
    for ext, dtype in RAW:
        path, coco, _ = make_raw_and_coco(directory, ext, dtype)
        files["signal_file_capture" + ext] = path
        files["signal_file_capture" + ext + ".coco"] = coco
    return files


def observe(sig):
    a = np.asarray(sig.iq_array.data)
    return [(a.dtype, a.shape, a.tobytes()), sig.sample_rate, sig.already_demodulated, sig.wav_mode, sig.num_samples]   # bit-identical samples


@pytest.fixture(scope="module")
def load():
    from urh_b200 import settings
    from urh_b200.signalprocessing.Signal import Signal

    settings.write("default_noise_threshold", "3")

    def run(key, path):
        sig = Signal(str(path), "t")
        assert_matches_reference(key, [observe(sig)])
        return sig
    yield run
    settings.write("default_noise_threshold", "automatic")


@pytest.mark.parametrize("width", [1, 2, 3, 4])
@pytest.mark.parametrize("channels", [1, 2])
def test_wav(load, tmp_path, width, channels):
    path, rate = make_wav(tmp_path, width, channels)
    mine = load("signal_file_" + path.name, path)
    assert mine.sample_rate == rate
    assert mine.already_demodulated == (channels == 1)


def test_flipper_sub(load, tmp_path):
    path = make_flipper_sub(tmp_path)
    mine = load("signal_file_" + path.name, path)
    assert mine.already_demodulated and mine.num_samples == 300 + 900 + 300 + 300 + 900 + 9000 + 450 + 450 + 1350 + 100


@pytest.mark.parametrize("ext,dtype", RAW)
def test_raw_formats_and_coco(load, tmp_path, ext, dtype):
    path, coco, data = make_raw_and_coco(tmp_path, ext, dtype)
    mine = load("signal_file_capture" + ext, path)
    assert mine.iq_array.data.dtype == dtype and np.array_equal(mine.iq_array.data, data)
    mine2 = load("signal_file_capture" + ext + ".coco", coco)
    assert np.array_equal(mine2.iq_array.data, data)


@pytest.mark.gpu
@pytest.mark.parametrize("ext,dtype", [(".cu8", np.uint8), (".complex16u", np.uint8), (".cu16", np.uint16), (".complex32u", np.uint16)])
def test_unsigned_formats_become_signed(tmp_path, ext, dtype):
    """unsigned captures are handled as signed (IQArray.py:214-218): the conversion runs on the device (convert.cu)"""
    from urh_b200 import settings
    from urh_b200.signalprocessing.Signal import Signal

    info = np.iinfo(dtype)
    data = np.random.default_rng(len(ext)).integers(info.min, info.max + 1, (999, 2)).astype(dtype)
    data[0], data[1] = info.min, info.max
    path = tmp_path / ("capture" + ext)
    data.tofile(str(path))
    settings.write("default_noise_threshold", "3")
    try:
        sig = Signal(str(path), "t")
    finally:
        settings.write("default_noise_threshold", "automatic")
    signed = np.int8 if dtype == np.uint8 else np.int16
    half = 128 if dtype == np.uint8 else 32768
    assert sig.iq_array.data.dtype == signed
    assert np.array_equal(sig.iq_array.data, (data.astype(np.int64) - half).astype(signed))
