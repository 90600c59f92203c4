"""Training-side data path (SURVEY §8f row N4): the native wav reader + aligned random crop against the reference's
`dataset/waveform_dataset.py:56-67` / `util/utils.py:101-113`. CPU only. The wav files are written here with scipy / the
stdlib. What the UNCHANGED reference Dataset class returned for them (its `librosa.load` stubbed with a scipy reader that
converts like soundfile does), with the same numpy seed, is stored in tests/golden/dataset_items.json."""
import hashlib
import json
import os
import wave

import torch

import numpy as np
import pytest
import scipy.io.wavfile as wavfile

from wave_u_net_for_speech_enhancement_b200 import _lib
from wave_u_net_for_speech_enhancement_b200 import dataset as ds


def soundfile_like(path):
    """What librosa.load(path, sr=None) returns for a wav file: float32, integer PCM scaled by 2^-(bits-1), channel mean."""
    sr, a = wavfile.read(path)
    if a.dtype == np.int16:
        f = a.astype(np.float32) / 32768.0
    elif a.dtype == np.int32:
        f = (a.astype(np.float64) / 2147483648.0).astype(np.float32)
    elif a.dtype == np.uint8:
        f = (a.astype(np.float32) - 128.0) / 128.0
    else:
        f = a.astype(np.float32)
    if f.ndim == 2:
        f = f.mean(axis=1, dtype=np.float32) if f.dtype == np.float32 else f.mean(axis=1).astype(np.float32)
    return f, sr


def write_pcm24(path, samples, rate=16000):
    """24-bit PCM through the stdlib (scipy cannot write it): samples = int32 values in [-2^23, 2^23)."""
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(3)
        w.setframerate(rate)
        b = bytearray()
        for v in samples.tolist():
            b += int(v & 0xFFFFFF).to_bytes(3, "little")
        w.writeframes(bytes(b))


@pytest.fixture()
def wavs(tmp_path):
    rng = np.random.default_rng(11)
    n = 40000
    out = {}
    a16 = rng.integers(-32768, 32767, n, dtype=np.int16)
    out["pcm16"] = str(tmp_path / "a16.wav"); wavfile.write(out["pcm16"], 16000, a16)
    a32 = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int32)
    out["pcm32"] = str(tmp_path / "a32.wav"); wavfile.write(out["pcm32"], 22050, a32)
    af = (0.3 * rng.standard_normal(n)).astype(np.float32)
    out["f32"] = str(tmp_path / "af.wav"); wavfile.write(out["f32"], 16000, af)
    a8 = rng.integers(0, 255, n, dtype=np.uint8)
    out["u8"] = str(tmp_path / "a8.wav"); wavfile.write(out["u8"], 8000, a8)
    st = rng.integers(-32768, 32767, (n, 2), dtype=np.int16)
    out["stereo16"] = str(tmp_path / "st.wav"); wavfile.write(out["stereo16"], 16000, st)
    a24 = rng.integers(-2**23, 2**23 - 1, 5000, dtype=np.int32)
    out["pcm24"] = str(tmp_path / "a24.wav"); write_pcm24(out["pcm24"], a24)
    out["_a24"] = a24
    return out


@pytest.mark.parametrize("kind", ["pcm16", "pcm32", "f32", "u8", "stereo16"])
def test_wav_reader_matches_soundfile_conversion(wavs, kind):
    want, sr = soundfile_like(wavs[kind])
    got, sr2 = ds.load_wav(wavs[kind])
    assert sr2 == sr and got.dtype == np.float32 and got.shape == want.shape
    assert np.array_equal(got, want)
    info = ds.wav_info(wavs[kind])
    assert info["frames"] == len(want) and info["channels"] == (2 if kind == "stereo16" else 1)
    # a window of the file = the same samples
    win, _ = ds.load_wav(wavs[kind], 1234, 777)
    assert np.array_equal(win, want[1234:1234 + 777])


def test_wav_reader_pcm24_and_errors(wavs, tmp_path):
    got, sr = ds.load_wav(wavs["pcm24"])
    assert sr == 16000 and np.array_equal(got, (wavs["_a24"].astype(np.float64) / 8388608.0).astype(np.float32))
    with pytest.raises(_lib.WunetError):
        ds.load_wav(str(tmp_path / "missing.wav"))
    bad = tmp_path / "bad.wav"
    bad.write_bytes(b"not a wav file at all")
    with pytest.raises(_lib.WunetError):
        ds.wav_info(str(bad))
    with pytest.raises(_lib.WunetError):
        ds.load_wav(wavs["pcm16"], 39000, 2000)          # window past the end


def _pair_files(tmp_path, n_items=5, base_len=20000):
    rng = np.random.default_rng(3)
    lines = []
    for i in range(n_items):
        n = base_len + 137 * i
        clean = rng.integers(-20000, 20000, n, dtype=np.int16)
        noisy = np.clip(clean.astype(np.int32) + rng.integers(-3000, 3000, n), -32768, 32767).astype(np.int16)
        pc, pn = str(tmp_path / f"clean_{i}.wav"), str(tmp_path / f"noisy_{i}.wav")
        wavfile.write(pc, 16000, clean)
        wavfile.write(pn, 16000, noisy)
        lines.append(f"{pn} {pc}")
    lst = tmp_path / "train.txt"
    lst.write_text("\n".join(lines) + "\n")
    return str(lst), lines


def test_dataset_items_and_crops(tmp_path):
    lst, lines = _pair_files(tmp_path)
    d = ds.Dataset(lst, sample_length=16384, mode="train")
    assert len(d) == 5
    np.random.seed(42)
    items = [d[i] for i in range(5)]
    np.random.seed(42)
    for i, (mix, clean, name) in enumerate(items):
        pn, pc = lines[i].split(" ")
        fm, _ = soundfile_like(pn)
        fc, _ = soundfile_like(pc)
        start = np.random.randint(len(fm) - 16384 + 1)            # util/utils.py:109
        assert mix.shape == (1, 16384) and clean.shape == (1, 16384) and name == f"noisy_{i}"
        assert np.array_equal(mix[0], fm[start:start + 16384]) and np.array_equal(clean[0], fc[start:start + 16384])
    v = ds.Dataset(lst, limit=2, offset=1, mode="validation")
    mix, clean, name = v[0]
    assert len(v) == 2 and name == "noisy_1" and mix.shape == (1, 20137) and np.array_equal(mix[0], soundfile_like(lines[1].split(" ")[0])[0])
    with pytest.raises(AssertionError):
        ds.Dataset(lst, sample_length=30000)[0]                   # clip shorter than sample_length: the reference asserts too


def test_dataset_matches_unchanged_reference_class(tmp_path, golden_dir):
    lst, _lines = _pair_files(tmp_path)
    want = json.load(open(os.path.join(golden_dir, "dataset_items.json")))
    for mode in ("train", "validation"):
        o = ds.Dataset(lst, sample_length=want["sample_length"], mode=mode)
        np.random.seed(want["seed"])
        got = [o[i] for i in range(len(o))]
        assert len(got) == len(want[mode])
        for w, (gm, gc, gn) in zip(want[mode], got):
            assert gn == w["name"] and list(gm.shape) == w["shape"] and list(gc.shape) == w["shape"]
            assert str(gm.dtype) == str(gc.dtype) == w["dtype"]
            assert hashlib.sha256(np.ascontiguousarray(gm).tobytes()).hexdigest() == w["mixture_sha256"], (mode, gn)
            assert hashlib.sha256(np.ascontiguousarray(gc).tobytes()).hexdigest() == w["clean_sha256"], (mode, gn)


@pytest.mark.parametrize("pcm", [False, True])
def test_cached_pairs_batches(tmp_path, pcm):
    rng = np.random.default_rng(9)
    pairs = []
    for i in range(6):
        n = 17000 + 501 * i
        if pcm:
            a = rng.integers(-32768, 32767, n, dtype=np.int16); b = rng.integers(-32768, 32767, n, dtype=np.int16)
        else:
            a = rng.standard_normal(n).astype(np.float32); b = rng.standard_normal(n).astype(np.float32)
        pairs.append((a, b))
    cp = ds.CachedPairs(pairs, sample_length=16384, pin=False)
    idx = [5, 0, 3, 3, 1]
    np.random.seed(1)
    mix, clean = cp.batch(idx)
    np.random.seed(1)
    assert mix.shape == (5, 1, 16384) and clean.shape == (5, 1, 16384)
    for row, i in enumerate(idx):
        s = np.random.randint(len(pairs[i][0]) - 16384 + 1)
        wa, wb = pairs[i][0][s:s + 16384], pairs[i][1][s:s + 16384]
        if pcm:
            wa, wb = wa.astype(np.float32) / 32768.0, wb.astype(np.float32) / 32768.0
        assert np.array_equal(mix[row, 0].numpy(), wa) and np.array_equal(clean[row, 0].numpy(), wb)
    with pytest.raises(_lib.WunetError):
        cp.batch([0], starts=[len(pairs[0][0]) - 16383])           # window past the end of the clip
    with pytest.raises(AssertionError):
        ds.CachedPairs([(np.zeros(100, np.float32), np.zeros(100, np.float32))])


def test_cached_pairs_from_files(tmp_path):
    lst, lines = _pair_files(tmp_path, n_items=3)
    cp = ds.CachedPairs([tuple(l.split(" ")) for l in lines], pin=False)
    mix, clean = cp.batch([2, 1], starts=[5, 0])
    assert np.array_equal(mix[0, 0].numpy(), soundfile_like(lines[2].split(" ")[0])[0][5:5 + 16384])
    assert np.array_equal(clean[1, 0].numpy(), soundfile_like(lines[1].split(" ")[1])[0][:16384])


def test_batch_stream_prefetches_in_order_and_keeps_buffers_valid():
    rng = np.random.default_rng(4)
    pairs = [(rng.standard_normal(17000 + 33 * i).astype(np.float32), rng.standard_normal(17000 + 33 * i).astype(np.float32))
             for i in range(7)]
    cp = ds.CachedPairs(pairs, sample_length=16384, pin=False)
    batches = [[0, 1, 2], [3, 4], [5, 6, 0], [1, 1, 1], [2]]
    stream = ds.BatchStream(cp, batches, depth=3, rng=np.random.default_rng(123))
    ref_rng = np.random.default_rng(123)
    got = []
    for k, (mix, clean) in enumerate(stream):
        starts = [int(ref_rng.integers(len(pairs[i][0]) - 16384 + 1)) for i in batches[k]]
        assert stream.last_starts == starts and mix.shape == (len(batches[k]), 1, 16384)
        for row, (i, s) in enumerate(zip(batches[k], starts)):
            assert np.array_equal(mix[row, 0].numpy(), pairs[i][0][s:s + 16384])
            assert np.array_equal(clean[row, 0].numpy(), pairs[i][1][s:s + 16384])
        got.append((mix, mix.clone()))
        if len(got) >= 2:                              # the previous batch's buffers are still intact (depth 3: two stay valid)
            assert torch.equal(got[-2][0], got[-2][1])
    assert len(got) == len(batches)
    # errors of the producer thread surface in the consumer
    bad = ds.BatchStream(cp, [[0], [99]], depth=2)
    with pytest.raises(IndexError):
        for _ in bad:
            pass


def test_wav_reader_skips_other_chunks_and_reads_extensible_headers(tmp_path):
    """A LIST chunk (odd size, padded) before "data", and a WAVE_FORMAT_EXTENSIBLE header whose sub-format says PCM: what
    ffmpeg / soundfile write for multi-channel or 24-bit files."""
    import struct
    rng = np.random.default_rng(1)
    pcm = rng.integers(-32768, 32767, 3001, dtype=np.int16)
    data = pcm.tobytes()
    fmt_ext = struct.pack("<HHIIHHHHIH14s", 0xFFFE, 1, 16000, 32000, 2, 16, 22, 16, 4, 1, b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71")
    lst = b"INFOISFT\x05\x00\x00\x00Lavf\x00"                      # odd-sized sub-chunk inside, total length odd
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt_ext)) + fmt_ext
    body += b"LIST" + struct.pack("<I", len(lst)) + lst + (b"\x00" if len(lst) & 1 else b"")
    body += b"data" + struct.pack("<I", len(data)) + data
    p = tmp_path / "ext.wav"
    p.write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)
    info = ds.wav_info(str(p))
    assert info == {"sample_rate": 16000, "channels": 1, "frames": 3001, "bits": 16, "is_float": False}
    got, _ = ds.load_wav(str(p))
    assert np.array_equal(got, pcm.astype(np.float32) / 32768.0)
    # a streamed file with a zero data size: the rest of the file is the data
    body0 = b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 1, 1, 8000, 16000, 2, 16) + b"data" + struct.pack("<I", 0) + data
    q = tmp_path / "stream.wav"
    q.write_bytes(b"RIFF" + struct.pack("<I", 0xFFFFFFFF) + body0)
    assert ds.wav_info(str(q))["frames"] == 3001 and np.array_equal(ds.load_wav(str(q))[0], got)
    # ADPCM (format tag 2) is refused loudly
    bad = b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 2, 1, 8000, 4000, 256, 4) + b"data" + struct.pack("<I", 8) + b"\x00" * 8
    r = tmp_path / "adpcm.wav"
    r.write_bytes(b"RIFF" + struct.pack("<I", len(bad)) + bad)
    with pytest.raises(_lib.WunetError, match="unsupported"):
        ds.wav_info(str(r))
