"""GPU parity: NAT acoustic model (CUDA, through the C ABI) vs the CPU restatement.

The oracle for this stage is pinned to the reference's own source (tests/test_reference_goldens.py); the direct
comparison of the CUDA path with reference-produced vectors is tests/test_gpu_reference_goldens.py.
Tolerance (fp32, shared dropout masks): mel L-inf <= 1e-3 (log-mel units) after the
full autoregressive scan; encoder/upsample taps <= 1e-4."""
import numpy as np
import pytest
import torch

from oracle import nat_oracle as no
from viettts_b200 import synthetic

pytestmark = pytest.mark.gpu
MEL_LINF = 1e-3


@pytest.fixture(scope="module", params=["fp32", "bf16x3"])
def eng(acoustic_ckpt, request):
    """Both arithmetic paths of the dense contractions (convs + hoisted LSTM input GEMMs) must meet
    the same tolerance; the recurrent part is fp32 in both."""
    from viettts_b200.engine import Engine
    e = Engine(0)
    e.load_acoustic(acoustic_ckpt)
    e.set_precision(request.param)
    yield e
    e.close()


def _utt(seed, L, seconds):
    tokens, dur = synthetic.utterance(seed, L, seconds)
    d, n = no.seconds_to_frames(dur)
    return np.asarray(tokens, np.int32), d[0], n


def test_small_utterance_all_taps(eng, acoustic_ckpt):
    tk, d, n = _utt(0, 20, 0.5)
    masks = synthetic.dropout_masks(42, 1, n)
    mel = eng.predict_mel(tk[None], d[None], n_frames=[n], masks=masks)
    taps = {}
    ref = no.inference(acoustic_ckpt, tk[None], d[None], n, masks, taps=taps).numpy()
    enc = eng.debug_read("enc", (1, 20, 512))
    cond = eng.debug_read("cond", (1, n, 512))
    pre = eng.debug_read("mel_pre", (1, n, 80))
    e_enc = np.abs(enc - taps["enc"].numpy()).max()
    e_cond = np.abs(cond - taps["cond"].numpy()).max()
    e_pre = np.abs(pre - taps["pre"].numpy()).max()
    e_mel = np.abs(mel - ref).max()
    print(f"enc {e_enc:.3e} cond {e_cond:.3e} pre {e_pre:.3e} mel {e_mel:.3e}")
    assert e_enc < 1e-4 and e_cond < 1e-4
    assert e_pre < MEL_LINF and e_mel < MEL_LINF


def test_c1_100_phonemes_5s(eng, acoustic_ckpt):
    """BASELINE config 1 shape: 100 phonemes, 312 frames, shared masks."""
    tk, d, n = _utt(0, 100, 5.0)
    assert n == 312
    masks = synthetic.dropout_masks(42, 1, n)
    mel = eng.predict_mel(tk[None], d[None], n_frames=[n], masks=masks)
    ref = no.inference(acoustic_ckpt, tk[None], d[None], n, masks).numpy()
    ref64 = no.inference(acoustic_ckpt, tk[None], d[None], n, masks, dtype=torch.float64).numpy()
    print(f"C1: gpu-vs-f32 {np.abs(mel-ref).max():.3e}  gpu-vs-f64 {np.abs(mel-ref64).max():.3e}  f32-vs-f64 {np.abs(ref-ref64).max():.3e}")
    assert np.abs(mel - ref64).max() < MEL_LINF


def test_dropout_off_mode(eng, acoustic_ckpt):
    tk, d, n = _utt(3, 30, 1.0)
    mel = eng.predict_mel(tk[None], d[None], n_frames=[n])
    ref = no.inference(acoustic_ckpt, tk[None], d[None], n, None).numpy()
    assert np.abs(mel - ref).max() < MEL_LINF


def _threefry2x32(k0, k1, c0, c1):
    """numpy restatement of the device generator (csrc/nat.cu) for the SEED mode check."""
    M = np.uint32
    k0, k1, c0, c1 = (np.asarray(v, dtype=np.uint32) for v in (k0, k1, c0, c1))
    ks = [k0, k1, M(0x1BD11BDA) ^ k0 ^ k1]
    x0, x1 = c0 + k0, c1 + k1
    R = [[13, 15, 26, 6], [17, 29, 16, 24]]
    with np.errstate(over="ignore"):
        for blk in range(5):
            for r in R[blk & 1]:
                x0 = x0 + x1
                x1 = (x1 << M(r)) | (x1 >> M(32 - r))
                x1 = x1 ^ x0
            x0 = x0 + ks[(blk + 1) % 3]
            x1 = x1 + ks[(blk + 2) % 3] + M(blk + 1)
    return x0, x1


def test_seed_mode_matches_documented_stream(eng, acoustic_ckpt):
    tk, d, n = _utt(4, 25, 0.8)
    seed = (7 << 32) | 12345
    mel = eng.predict_mel(tk[None], d[None], n_frames=[n], seed=seed)
    t = np.arange(n, dtype=np.uint32)[:, None, None]
    lu = (np.arange(2, dtype=np.uint32)[None, :, None] * 256 + np.arange(256, dtype=np.uint32)[None, None, :])
    o0, _ = _threefry2x32(np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32), t + 0 * lu, lu + 0 * t)
    masks = (o0 < np.uint32(0x80000000)).astype(np.uint8)[None]
    assert 0.4 < masks.mean() < 0.6
    ref = no.inference(acoustic_ckpt, tk[None], d[None], n, masks).numpy()
    assert np.abs(mel - ref).max() < MEL_LINF
    again = eng.predict_mel(tk[None], d[None], n_frames=[n], seed=seed)
    assert np.array_equal(mel, again)


def test_ragged_batch_equals_single_rows(eng, acoustic_ckpt):
    """Batched semantics (SURVEY H4): row b == reference run on row b alone."""
    utts = [_utt(10, 12, 0.3), _utt(11, 31, 1.1), _utt(12, 20, 0.7), _utt(13, 5, 0.2)]
    B = len(utts)
    Lmax = max(len(u[0]) for u in utts)
    tokens = np.zeros((B, Lmax), np.int32)
    dur = np.zeros((B, Lmax), np.float32)
    lens = np.array([len(u[0]) for u in utts], np.int32)
    nfs = np.array([u[2] for u in utts], np.int32)
    for b, (tk, d, n) in enumerate(utts):
        tokens[b, : len(tk)] = tk
        dur[b, : len(tk)] = d
    N = int(nfs.max())
    masks = synthetic.dropout_masks(5, B, N)
    mel = eng.predict_mel(tokens, dur, lengths=lens, n_frames=nfs, masks=masks)
    refs = no.inference_ragged(acoustic_ckpt, [u[0] for u in utts], [u[1] for u in utts], [masks[b] for b in range(B)])
    for b in range(B):
        e = np.abs(mel[b, : nfs[b]] - refs[b]).max()
        print(f"row {b}: L={lens[b]} N={nfs[b]} err {e:.3e}")
        assert e < MEL_LINF
        assert np.all(mel[b, nfs[b] :] == 0.0)


def test_batch32_rows_independent(eng, acoustic_ckpt):
    """Config-3 size (B=32, L=100, N=312): every row must equal that row run alone (bit exact:
    same kernels, same reduction order), and one row is checked against the oracle."""
    B = 32
    utts = [_utt(100 + b, 100, 5.0) for b in range(B)]
    tokens = np.stack([u[0] for u in utts])
    dur = np.stack([u[1] for u in utts])
    nfs = np.array([u[2] for u in utts], np.int32)
    assert (nfs == 312).all()
    masks = synthetic.dropout_masks(9, B, 312)
    mel = eng.predict_mel(tokens, dur, n_frames=nfs, masks=masks)
    assert np.isfinite(mel).all()
    for b in (0, 13, 31):
        alone = eng.predict_mel(tokens[b : b + 1], dur[b : b + 1], n_frames=nfs[b : b + 1], masks=masks[b : b + 1])
        assert np.abs(alone[0] - mel[b]).max() < 1e-5
    ref = no.inference(acoustic_ckpt, tokens[7:8], dur[7:8], 312, masks[7:8]).numpy()
    assert np.abs(mel[7] - ref[0]).max() < MEL_LINF


def test_synthesize_equals_two_stage(eng, acoustic_ckpt, hifigan_params):
    eng.load_hifigan(hifigan_params)
    tk, d, n = _utt(0, 16, 0.4)
    masks = synthetic.dropout_masks(1, 1, n)
    wav, mel = eng.synthesize(tk[None], d[None], n_frames=[n], masks=masks, return_mel=True)
    mel2 = eng.predict_mel(tk[None], d[None], n_frames=[n], masks=masks)
    assert np.array_equal(mel, mel2)
    assert np.array_equal(wav, eng.mel2wave(mel2))


def test_mixed_length_bucketed_synthesis(eng, hifigan_params):
    """configs[4]-style mixed lengths: bucketed ragged batches must return, per utterance, what a
    single-utterance call returns (dropout off so that rows do not depend on their batch position)."""
    eng.load_hifigan(hifigan_params)
    rng = np.random.default_rng(3)
    utts = []
    for i in range(10):
        L = int(rng.integers(8, 40))
        tk, d, n = _utt(200 + i, L, None)
        utts.append((tk, d))
    wavs = eng.synthesize_many(utts, max_rows=4)
    assert len(wavs) == len(utts)
    for i in (0, 3, 7, 9):
        tk, d = utts[i]
        n = int(np.sum(d, dtype=np.float32))
        alone = eng.synthesize(tk[None], d[None], n_frames=[n])
        assert wavs[i].shape == (n * 256,)
        assert np.abs(wavs[i] - alone[0]).max() < 1e-5


def test_pinned_output_buffer_path(eng, hifigan_params):
    """`out=` with page-locked memory takes the direct D2H path and must give the same samples."""
    from viettts_b200.engine import Engine
    eng.load_hifigan(hifigan_params)
    tk, d, n = _utt(5, 14, 0.4)
    ref = eng.synthesize(tk[None], d[None], n_frames=[n], seed=3)
    buf = Engine.pinned_empty((1, n * 256))
    got = eng.synthesize(tk[None], d[None], n_frames=[n], seed=3, out=buf)
    assert got is buf and np.array_equal(got, ref)
    buf2 = np.empty((1, n * 256), np.float32)           # pageable out= goes through the staging copy
    assert np.array_equal(eng.synthesize(tk[None], d[None], n_frames=[n], seed=3, out=buf2), ref)


def test_batch_spanning_two_decoder_launches(eng, acoustic_ckpt):
    """40 rows = one scan launch with two 32-row groups (up to 128 rows share a launch): rows must not depend on their
    row group."""
    B = 40
    utts = [_utt(300 + b, 24, 0.6) for b in range(B)]
    L = 24
    tokens = np.stack([u[0] for u in utts])
    dur = np.stack([u[1] for u in utts])
    nfs = np.array([u[2] for u in utts], np.int32)
    masks = synthetic.dropout_masks(17, B, int(nfs.max()))
    mel = eng.predict_mel(tokens, dur, n_frames=nfs, masks=masks)
    for b in (0, 31, 32, 39):
        ref = no.inference(acoustic_ckpt, tokens[b : b + 1], dur[b : b + 1], int(nfs[b]), masks[b : b + 1, : nfs[b]]).numpy()
        assert np.abs(mel[b, : nfs[b]] - ref[0]).max() < MEL_LINF
        assert np.all(mel[b, nfs[b] :] == 0.0)


def test_long_utterance_300_phonemes(eng, acoustic_ckpt):
    """Upper end of BASELINE configs[4]: 300 phonemes, 937 frames (upsampling shared memory, long scan)."""
    tk, d, n = _utt(77, 300, 15.0)
    assert n >= 930
    masks = synthetic.dropout_masks(4, 1, n)
    mel = eng.predict_mel(tk[None], d[None], n_frames=[n], masks=masks)
    ref = no.inference(acoustic_ckpt, tk[None], d[None], n, masks, dtype=torch.float64).numpy()
    err = np.abs(mel - ref).max()
    print(f"L=300 N={n}: err {err:.3e}")
    assert err < MEL_LINF
