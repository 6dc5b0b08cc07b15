"""Host-side callers of the hot path (SURVEY.md §8f rows 1-2): text normalisation, text2tokens, lexicon,
duration fix-ups and the PCM-16 WAV writer, against vectors produced by the reference's own functions
(tests/golden/make_text_golden.py)."""
import json
import struct

import numpy as np
import pytest

from viettts_b200 import config, synthesizer
from viettts_b200.nat import text2mel as t2m


@pytest.fixture(scope="module")
def golden(golden_dir):
    return json.loads((golden_dir / "text_frontend.json").read_text())


def test_alphabet_matches_reference(golden):
    assert config.PHONEMES == golden["phonemes"]
    assert config.SIL_INDEX == golden["sil_index"] and config.WORD_END_INDEX == golden["word_end_index"]
    assert len(config.PHONEMES) == config.ALPHABET_SIZE == 93


def test_normalize_text(golden):
    for c in golden["cases"]:
        assert synthesizer.nat_normalize_text(c["text"]) == c["normalized"], c["text"]


def test_text2tokens(golden, golden_dir):
    lex = golden_dir / "lexicon_small.txt"
    for c in golden["cases"]:
        if "error" in c:   # lexicon phoneme outside the alphabet: the reference raises ValueError (text2mel.py:49)
            with pytest.raises(ValueError):
                t2m.text2tokens(c["normalized"], lex)
        else:
            assert t2m.text2tokens(c["normalized"], lex) == c["tokens"], c["text"]


def test_load_lexicon(golden_dir):
    lex = t2m.load_lexicon(golden_dir / "lexicon_small.txt")
    assert lex["xin"].split() == ["x", "i", "n"]
    assert all(k == k.lower() for k in lex)


def test_adjust_durations_and_trim():
    from oracle import nat_oracle as no
    tokens = [0, 10, 3, 12, 0]
    d = np.array([[0.02, 0.1, 0.07, 0.2, 0.31]], np.float32)
    for sd in (-1.0, 0.05, 0.5):
        got = t2m.adjust_durations(tokens, d, sd)
        ref = no.adjust_durations(tokens, d, sd)
        np.testing.assert_array_equal(got, ref)
        assert got[0, 2] == 0.0 and got[0, 0] == max(0.02, sd) and got[0, 1] == np.float32(0.1)
    mel = np.zeros((1, 40, 80), np.float32)
    assert no.trim_end_silence(tokens, d, mel).shape[1] == 40 - int(float(d[0, -1]) * 62.5)
    assert no.trim_end_silence([0, 5, 7], d[:, :3], mel).shape[1] == 40   # no trailing silence token


def test_pcm16_conversion_is_libsndfile_style():
    x = np.array([0.0, 1.0, -1.0, 0.5, -0.5, 0.25, 0.75, 2.0, -2.0], np.float32)
    pcm = synthesizer.float_to_pcm16(x)
    assert pcm.dtype == np.dtype("<i2")
    assert pcm.tolist()[:3] == [0, 32767, -32767]
    assert pcm[3] == 16384 and pcm[4] == -16384  # 16383.5 -> even neighbour (lrintf rounds half to even)
    assert pcm[5] == 8192 and pcm[6] == 24575    # 8191.75 -> 8192, 24575.25 -> 24575
    assert pcm[7] == 32767 and pcm[8] == -32768  # clipped, never wrapped


def test_wav_roundtrip(tmp_path):
    rng = np.random.default_rng(0)
    w = np.tanh(rng.standard_normal(4000)).astype(np.float32) * 0.9
    fn = tmp_path / "a.wav"
    synthesizer.write_wav(fn, w, 16000)
    raw = fn.read_bytes()
    assert len(raw) == 44 + 2 * w.size
    assert raw[:4] == b"RIFF" and struct.unpack("<I", raw[4:8])[0] == len(raw) - 8
    assert struct.unpack("<HHIIHH", raw[20:36]) == (1, 1, 16000, 32000, 2, 16)
    back, sr = synthesizer.read_wav(fn)
    assert sr == 16000 and np.abs(back - w).max() <= 0.5 / 32767 + 1e-7
    import wave
    with wave.open(str(fn)) as f:   # an independent parser agrees on the header
        assert (f.getnchannels(), f.getsampwidth(), f.getframerate(), f.getnframes()) == (1, 2, 16000, w.size)


def test_pinned_buffers_are_released_with_the_array(monkeypatch):
    """Engine.pinned_empty keeps the owning tensor alive only as long as the numpy array (or a view of it) lives."""
    import gc
    import torch
    from viettts_b200.engine import Engine
    real = torch.empty
    monkeypatch.setattr(torch, "empty", lambda *a, pin_memory=False, **k: real(*a, **k))   # no CUDA here: unpinned stand-in
    n0 = len(Engine._pinned_keepalive)
    a = Engine.pinned_empty((4, 8))
    view = a[1:]
    assert a.shape == (4, 8) and a.dtype == np.float32 and len(Engine._pinned_keepalive) == n0 + 1
    del a
    gc.collect()
    assert len(Engine._pinned_keepalive) == n0 + 1      # the view still references the buffer
    view[:] = 1.0
    del view
    gc.collect()
    assert len(Engine._pinned_keepalive) == n0
