"""Engine: one libviettts_b200 context per GPU + the host-side plumbing around it.

Host buffers are numpy arrays (the reference's seams take/return numpy / jax
arrays on the host); device buffers are torch tensors used purely as memory
containers (`tensor.data_ptr()` is what crosses the C ABI)."""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib, config, weights

DROPOUT_OFF, DROPOUT_MASK, DROPOUT_SEED = 0, 1, 2


def _chunk_seed(seed: int, chunk: int) -> int:
    """Key of the on-device dropout stream for the chunk-th slice of an over-long batch (a distinct 64-bit key per
    chunk: `seed + offset` would alias the next seed's first chunk)."""
    return (int(seed) ^ (chunk * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF
PRECISION_FP32, PRECISION_BF16X3 = 0, 1
MAX_ACOUSTIC_ROWS = 128   # rows per vtts_acoustic_forward call (csrc/nat.cu MAX_ROWS)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _np(a, dtype, shape=None, what="array"):
    a = np.ascontiguousarray(np.asarray(a), dtype=dtype)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError(f"{what}: expected shape {tuple(shape)}, got {tuple(a.shape)}")
    return a


class Engine:
    """A context on one B200.  Not thread-safe (like the C context)."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        self.device = int(device)
        h = _lib.c_ctx()
        rc = self.lib.vtts_create(self.device, C.byref(h))
        if rc != 0:
            msg = self.lib.vtts_last_error(None)
            raise _lib.VttsError(rc, msg.decode() if msg else "?")
        self.h = h
        self._hifigan_key = None
        self._acoustic_key = None
        self._duration_key = None
        self._mel_loaded = False

    def close(self):
        if getattr(self, "h", None):
            self.lib.vtts_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _lib.check(self.h, rc)

    # ---- info ----
    def device_info(self) -> dict:
        sm, ma, mi, hb = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        self._ck(self.lib.vtts_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(hb)))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), hbm_bytes=hb.value)

    def launch_count(self) -> int:
        return int(self.lib.vtts_launch_count(self.h))

    def last_stage_ms(self, stage: int) -> float:
        ms = C.c_float()
        self._ck(self.lib.vtts_last_stage_ms(self.h, stage, C.byref(ms)))
        return float(ms.value)

    def set_precision(self, mode) -> None:
        """'fp32' (strict, FMA pipe) or 'bf16x3' (tcgen05 tensor cores, split-bf16, fp32 accumulate)."""
        m = {"fp32": PRECISION_FP32, "bf16x3": PRECISION_BF16X3}.get(mode, mode)
        self._ck(self.lib.vtts_set_precision(self.h, int(m)))

    def debug_conv1d(self, precision, x_t, w_t, bias_t, k, dil, pre_slope=1.0, resid_t=None, len_t=None):
        """Test hook: one conv layer (SAME padding, leaky_relu(pre_slope) on the input unless pre_slope == 1, optional
        residual) on torch CUDA tensors through either arithmetic path; x [B,T,Cin], w [k,Cin,Cout] -> [B,T,Cout]."""
        import torch
        B, T, Cin = x_t.shape
        out = torch.empty((B, T, w_t.shape[2]), dtype=torch.float32, device=x_t.device)
        self.debug_conv(precision, [dict(x0=x_t, w=w_t, bias=bias_t, resid=resid_t, out=out, k=k, dil=dil, in_off=-((k - 1) * dil // 2))],
                        B=B, T_rows=T, rows_out=T, Cin=Cin, Cout=w_t.shape[2], len_t=len_t,
                        pre_mode=0 if pre_slope == 1.0 else 1, pre_slope=pre_slope)
        return out

    _CONV_PTRS = ("x0", "x1", "x2", "w", "bias", "resid", "bn_mean", "bn_inv", "bn_off", "out")

    def debug_conv(self, precision, problems, *, B, T_rows, rows_out, Cin, Cout, len_t=None, len_mul=1, pre_mode=0, pre_slope=1.0,
                   post_act=0):
        """Test hook vtts_debug_conv: one conv launch of up to 8 problems through the models' own dispatch.  `problems`
        is a list of dicts with torch CUDA tensors under x0, x1, x2, w, bias, resid, bn_mean, bn_inv, bn_off, out (absent =
        NULL) and the ints k, dil, in_off, out_stride (default 1), out_off (default 0).  Writes the `out` tensors."""
        m = {"fp32": PRECISION_FP32, "bf16x3": PRECISION_BF16X3}.get(precision, precision)
        geom = _lib.ConvGeometry(B, T_rows, rows_out, Cin, Cout, _ptr(len_t), len_mul, pre_mode, pre_slope, post_act)
        probs = (_lib.ConvProblem * max(1, len(problems)))()
        for p, d in zip(probs, problems):
            for name in self._CONV_PTRS:
                setattr(p, name, _ptr(d.get(name)))
            p.k, p.dil, p.in_off = int(d["k"]), int(d["dil"]), int(d["in_off"])
            p.out_stride, p.out_off = int(d.get("out_stride", 1)), int(d.get("out_off", 0))
        self._ck(self.lib.vtts_debug_conv(self.h, int(m), C.byref(geom), probs, len(problems)))

    def debug_conv_transpose(self, precision, x0_t, w_t, bias_t, out_t, u, x1_t=None, x2_t=None, len_t=None, len_mul=1):
        """Test hook vtts_debug_conv_transpose: one generator up-sampling stage, lrelu(0.1) of x0 (or of (x0+x1+x2)/3)
        -> ConvTranspose(stride u); x [B,T,C], w Haiku [K,C/2,C] -> out_t [B,T*u,C/2] (rows past len*len_mul*u untouched)."""
        m = {"fp32": PRECISION_FP32, "bf16x3": PRECISION_BF16X3}.get(precision, precision)
        B, T, Cc = x0_t.shape
        self._ck(self.lib.vtts_debug_conv_transpose(self.h, int(m), _ptr(x0_t), _ptr(x1_t), _ptr(x2_t), _ptr(w_t), _ptr(bias_t),
                                                    _ptr(len_t), int(len_mul), B, T, Cc, int(u), int(w_t.shape[0]), _ptr(out_t)))

    def debug_pair(self, x_t, w1_t, b1_t, w2_t, b2_t, k, dil, slope=0.1, len_t=None):
        """Test hook: one fused ResBlock pair on torch CUDA tensors (tensor-core path)."""
        import torch
        B, T, Cc = x_t.shape
        out = torch.empty_like(x_t)
        self._ck(self.lib.vtts_debug_pair(self.h, _ptr(x_t), _ptr(w1_t), _ptr(b1_t), _ptr(w2_t), _ptr(b2_t), _ptr(len_t),
                                          B, T, Cc, int(k), int(dil), float(slope), _ptr(out)))
        return out

    PAIR_KERNELS = {"smem": 0, "tmem": 1, "smem2": 2, "smem2c": 3}

    def set_fused_pairs(self, on: bool, ts=None, kind: str | None = None):
        """Run the C <= 64 ResBlock pairs in a fused pair kernel (off: two tensor-core conv launches per pair).
        kind: "smem2" tc_pair2.cu (two decoupled pipelines, A operand in shared memory; the default), "smem2c" the same kernel
        in the CTA-pair form (cta_group::2 over clusters of two SMs, half of the weight operand per SM), "tmem"
        tc_pair_ts.cu (A operand in tensor memory), "smem" tc_pair.cu (first generation).  `ts` is the old spelling
        (True = "tmem", False = "smem")."""
        if kind is None:
            kind = "smem2" if ts is None else ("tmem" if ts else "smem")
        self._ck(self.lib.vtts_debug_tc_stats(self.h, 0x200 | ((1 if on else 0) << 10) | 0x800 | (self.PAIR_KERNELS[kind] << 12), None))

    def tc_stats(self, enable=True, variant=None):
        """Per-CTA stall counters of the last tensor-core conv launch (see vtts_debug_tc_stats);
        `variant` optionally selects the conv form for later launches: 3 = CTA pairs (cta_group::2) for C >= 128 (default),
        1 = single-CTA form, 0 / 2 = older tile-shape experiments."""
        out = np.zeros((256, 16), np.int64)
        flags = (1 if enable else 0) | (0 if variant is None else (0x100 | (int(variant) << 4)))
        self._ck(self.lib.vtts_debug_tc_stats(self.h, flags, _ptr(out)))
        return out

    SUBSTAGES = {1: "acoustic.encoder", 2: "acoustic.upsample", 3: "acoustic.cond_gemm", 4: "acoustic.decoder_scan",
                 5: "acoustic.projection", 6: "acoustic.postnet", 9: "hifigan.conv_pre", 10: "hifigan.stage0", 11: "hifigan.stage1",
                 12: "hifigan.stage2", 13: "hifigan.stage3", 14: "hifigan.conv_post", 17: "teacher.encoder_upsample",
                 18: "teacher.prenet_hoisted_gemm", 19: "teacher.zoneout_scan", 20: "teacher.projection_postnet"}

    def substages(self, enable=True) -> dict:
        """Per-kernel-group device times (ms) of the forward calls since the previous call (vtts_debug_substages);
        `enable` switches the event recording on/off for the following calls."""
        out = np.zeros(24, np.float32)
        self._ck(self.lib.vtts_debug_substages(self.h, 1 if enable else 0, _ptr(out)))
        return {name: float(out[i]) for i, name in self.SUBSTAGES.items() if out[i] > 0}

    # ---- weights ----
    def load_hifigan(self, params, key=None):
        """params: Haiku-layout dict, a packed float32 numpy blob, or a torch CUDA
        tensor holding the blob (e.g. received through an NCCL broadcast)."""
        blob = weights.pack_hifigan(params) if isinstance(params, dict) else params
        n = int(blob.size if isinstance(blob, np.ndarray) else blob.numel())
        if isinstance(blob, np.ndarray):
            blob = _np(blob, np.float32)
        self._ck(self.lib.vtts_load_hifigan(self.h, _ptr(blob), n))
        self._hifigan_key = key if key is not None else object()

    def load_acoustic(self, ckpt, key=None):
        blob = weights.pack_acoustic(ckpt) if isinstance(ckpt, dict) else ckpt
        n = int(blob.size if isinstance(blob, np.ndarray) else blob.numel())
        if isinstance(blob, np.ndarray):
            blob = _np(blob, np.float32)
        self._ck(self.lib.vtts_load_acoustic(self.h, _ptr(blob), n))
        self._acoustic_key = key if key is not None else object()

    def load_duration(self, ckpt, key=None):
        """ckpt: the duration checkpoint dict (params/aux), a packed numpy blob, or a torch CUDA tensor."""
        blob = weights.pack_duration(ckpt) if isinstance(ckpt, dict) else ckpt
        n = int(blob.size if isinstance(blob, np.ndarray) else blob.numel())
        if isinstance(blob, np.ndarray):
            blob = _np(blob, np.float32)
        self._ck(self.lib.vtts_load_duration(self.h, _ptr(blob), n))
        self._duration_key = key if key is not None else object()

    def broadcast_weights(self, nccl_comm, root: int, is_root: bool, stream=None):
        """vtts_broadcast_weights: the root's loaded models reach every rank's context by one grouped ncclBroadcast.
        `nccl_comm`: an ncclComm_t as ctypes.c_void_p / int (e.g. parallel.NcclComm(...).handle)."""
        self._ck(self.lib.vtts_broadcast_weights(self.h, nccl_comm, int(root), 1 if is_root else 0, stream))
        if not is_root:
            self._hifigan_key = self._acoustic_key = self._duration_key = object()

    def load_mel_filterbank(self, fb=None):
        fb = _np(weights.mel_filterbank() if fb is None else fb, np.float32, (config.MEL_DIM, config.N_FFT // 2 + 1), "filterbank")
        self._ck(self.lib.vtts_load_mel_filterbank(self.h, _ptr(fb), fb.shape[0], fb.shape[1]))
        self._mel_loaded = True

    # ---- host-buffer calls -----------------------------------------------------------
    def mel2wave(self, mel, n_frames=None, out=None) -> np.ndarray:
        """mel f32 [B,T,80] -> wav f32 [B,256T] (Generator.__call__, hifigan/model.py:109-125)."""
        mel = _np(mel, np.float32)
        if mel.ndim != 3 or mel.shape[2] != config.MEL_DIM:
            raise ValueError(f"mel must be [B,T,{config.MEL_DIM}], got {mel.shape}")
        B, T, _ = mel.shape
        nf = None if n_frames is None else _np(n_frames, np.int32, (B,), "n_frames")
        if out is not None and (out.shape != (B, T * config.HOP) or out.dtype != np.float32 or not out.flags.c_contiguous):
            raise ValueError(f"out must be C-contiguous float32 {(B, T * config.HOP)}")
        wav = out if out is not None else np.empty((B, T * config.HOP), np.float32)
        self._ck(self.lib.vtts_mel2wave_host(self.h, _ptr(mel), _ptr(nf), B, T, _ptr(wav)))
        return wav

    # receptive field of the generator in mel frames, one side: conv_pre 3 + ups_0 1 + stage-0 ResBlocks 60/8 +
    # stage 1 60/64 + stage 2 60/128 + stage 3 60/256 + ups/conv_post crumbs = 13.3 (hifigan/model.py:44-51,109-125)
    STREAM_HALO = 16

    def mel2wave_stream(self, mel, chunk_frames: int = 32, halo: int | None = None):
        """Chunked vocoding of ONE utterance for low first-audio latency (SURVEY.md §8f row 4): yields the waveform
        in pieces of `chunk_frames` mel frames.  Each piece is computed from its frames plus `halo` frames of
        context on both sides (recomputed, not carried), so the concatenation equals `mel2wave(mel)` exactly:
        every output sample sees its full receptive field, and samples inside the halo are discarded."""
        mel = _np(mel, np.float32)
        if mel.ndim == 3:
            if mel.shape[0] != 1:
                raise ValueError("mel2wave_stream takes one utterance ([T,80] or [1,T,80])")
            mel = mel[0]
        if mel.ndim != 2 or mel.shape[1] != config.MEL_DIM:
            raise ValueError(f"mel must be [T,{config.MEL_DIM}], got {mel.shape}")
        halo = self.STREAM_HALO if halo is None else int(halo)
        if chunk_frames < 1 or halo < 0:
            raise ValueError("chunk_frames >= 1 and halo >= 0 required")
        T = mel.shape[0]
        for t0 in range(0, T, chunk_frames):
            t1 = min(T, t0 + chunk_frames)
            a, b = max(0, t0 - halo), min(T, t1 + halo)
            wav = self.mel2wave(mel[None, a:b])[0]
            yield wav[(t0 - a) * config.HOP: (t1 - a) * config.HOP]

    def _acoustic_args(self, tokens, dur_frames, lengths, n_frames, masks, seed):
        tokens = _np(tokens, np.int32)
        if tokens.ndim != 2:
            raise ValueError("tokens must be [B,L]")
        B, L = tokens.shape
        dur = _np(dur_frames, np.float32, (B, L), "durations")
        lens = None if lengths is None else _np(lengths, np.int32, (B,), "lengths")
        if n_frames is None:
            nf = np.array([int(np.sum(dur[b, : (L if lens is None else lens[b])], dtype=np.float32)) for b in range(B)], np.int32)
        else:
            nf = _np(n_frames, np.int32, (B,), "n_frames")
        N = int(nf.max())
        if N < 1:
            raise ValueError("durations sum to less than one frame")
        if masks is not None:
            mode = DROPOUT_MASK
            masks = _np(masks, np.uint8)
            if masks.shape[0] != B or masks.shape[1] < N or masks.shape[2:] != (2, config.PRENET_DIM):
                raise ValueError(f"masks must be uint8 [B,>=N,2,256], got {masks.shape}")
            masks = np.ascontiguousarray(masks[:, :N])
        elif seed is not None:
            mode = DROPOUT_SEED
        else:
            mode = DROPOUT_OFF
        return tokens, dur, lens, nf, N, masks, mode, int(seed or 0)

    def predict_mel(self, tokens, dur_frames, lengths=None, n_frames=None, masks=None, seed=None) -> np.ndarray:
        """AcousticModel.inference for a (ragged) batch: tokens int [B,L], durations in FRAMES
        [B,L] -> mel f32 [B,N,80] with N = max_b n_frames[b] (rows past n_frames[b] are 0).
        Dropout (live at inference in the reference): `masks` uint8 [B,N,2,256] keep-masks,
        else `seed` for the on-device threefry stream, else off."""
        tokens, dur, lens, nf, N, masks, mode, seed = self._acoustic_args(tokens, dur_frames, lengths, n_frames, masks, seed)
        B, L = tokens.shape
        mel = np.empty((B, N, config.MEL_DIM), np.float32)
        for b0 in range(0, B, MAX_ACOUSTIC_ROWS):
            b1 = min(B, b0 + MAX_ACOUSTIC_ROWS)
            sl = slice(b0, b1)
            out = np.empty((b1 - b0, N, config.MEL_DIM), np.float32)
            self._ck(self.lib.vtts_predict_mel_host(
                self.h, _ptr(tokens[sl]), _ptr(None if lens is None else lens[sl]), _ptr(dur[sl]), _ptr(nf[sl]),
                _ptr(None if masks is None else np.ascontiguousarray(masks[sl])), mode, _chunk_seed(seed, b0 // MAX_ACOUSTIC_ROWS),
                b1 - b0, L, N, _ptr(out)))
            mel[sl] = out
        return mel

    def predict_duration(self, tokens, lengths=None) -> np.ndarray:
        """DurationModel.__call__ (nat/model.py:64-70) for a (ragged) batch: tokens int [B,L] -> predicted
        durations in SECONDS f32 [B,L] (0 past lengths[b]); row b equals the reference run on row b alone."""
        tokens = _np(tokens, np.int32)
        if tokens.ndim != 2:
            raise ValueError("tokens must be [B,L]")
        B, L = tokens.shape
        lens = None if lengths is None else _np(lengths, np.int32, (B,), "lengths")
        out = np.empty((B, L), np.float32)
        for b0 in range(0, B, MAX_ACOUSTIC_ROWS):
            b1 = min(B, b0 + MAX_ACOUSTIC_ROWS)
            o = np.empty((b1 - b0, L), np.float32)
            self._ck(self.lib.vtts_predict_duration_host(
                self.h, _ptr(np.ascontiguousarray(tokens[b0:b1])), _ptr(None if lens is None else np.ascontiguousarray(lens[b0:b1])),
                b1 - b0, L, _ptr(o)))
            out[b0:b1] = o
        return out

    @staticmethod
    def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
        """numpy array backed by page-locked host memory.  Passed as `out=` to synthesize / mel2wave the
        library copies D2H straight into it (no staging copy, no page faults of a fresh array).
        The pinned allocation lives exactly as long as the array (or any view of it)."""
        import weakref
        import torch
        t = torch.empty(tuple(shape), dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
        a = t.numpy()
        key = a.ctypes.data
        Engine._pinned_keepalive[key] = t            # the tensor owns the memory ...
        weakref.finalize(a, Engine._pinned_keepalive.pop, key, None)   # ... and is dropped with the array
        return a

    _pinned_keepalive: dict = {}

    def synthesize(self, tokens, dur_frames, lengths=None, n_frames=None, masks=None, seed=None, return_mel=False, out=None):
        """predict_mel -> mel2wave with the mel staying on the device.  Returns wav [B,256N]
        (and mel [B,N,80] if return_mel).  `out`: optional preallocated float32 [B,256N] result array
        (ideally from `pinned_empty`); it is validated and written in every path (rows land directly in it).
        In SEED mode row r of a call draws the device stream keyed by (seed, r, frame): an utterance's masks depend on
        its row index, not on the padded frame count of the batch; MASK / OFF modes are position independent."""
        tokens, dur, lens, nf, N, masks, mode, seed = self._acoustic_args(tokens, dur_frames, lengths, n_frames, masks, seed)
        B, L = tokens.shape
        if out is not None and (out.shape != (B, N * config.HOP) or out.dtype != np.float32 or not out.flags.c_contiguous):
            raise ValueError(f"out must be C-contiguous float32 {(B, N * config.HOP)}")
        wav = out if out is not None else np.empty((B, N * config.HOP), np.float32)
        mel = np.empty((B, N, config.MEL_DIM), np.float32) if return_mel else None
        for b0 in range(0, B, MAX_ACOUSTIC_ROWS):
            b1 = min(B, b0 + MAX_ACOUSTIC_ROWS)
            sl = slice(b0, b1)
            # row slices of C-contiguous arrays are contiguous: the library writes straight into the result
            self._ck(self.lib.vtts_synthesize_host(
                self.h, _ptr(tokens[sl]), _ptr(None if lens is None else lens[sl]), _ptr(dur[sl]), _ptr(nf[sl]),
                _ptr(None if masks is None else np.ascontiguousarray(masks[sl])), mode, _chunk_seed(seed, b0 // MAX_ACOUSTIC_ROWS),
                b1 - b0, L, N, _ptr(None if mel is None else mel[sl]), _ptr(wav[sl])))
        return (wav, mel) if return_mel else wav

    def tts(self, tokens, lengths=None, silence_duration=-1.0, seed=None, max_frames=None):
        """Token rows -> waveforms in ONE library call (vtts_tts_host): duration model, the duration fix-ups of
        text2mel.py:88-97, acoustic model, trailing-silence trim (:99-102) and generator, the mel never leaving
        the device.  tokens int [B,L] (rows padded to L), lengths int [B].  Returns (list of f32 waveforms,
        durations_sec f32 [B,L])."""
        tokens = _np(tokens, np.int32)
        if tokens.ndim != 2:
            raise ValueError("tokens must be [B,L]")
        B, L = tokens.shape
        if B > MAX_ACOUSTIC_ROWS:
            raise ValueError(f"tts: at most {MAX_ACOUSTIC_ROWS} rows per call")
        lens = None if lengths is None else _np(lengths, np.int32, (B,), "lengths")
        dur = np.empty((B, L), np.float32)
        nf = np.zeros(B, np.int32)
        nmax = C.c_int32(0)
        cap = int(max_frames) if max_frames else max(16, int(L * 0.12 * config.SAMPLE_RATE / config.HOP))
        mode = DROPOUT_SEED if seed is not None else DROPOUT_OFF
        for _ in range(2):
            wav = np.empty(B * cap * config.HOP, np.float32)
            rc = self.lib.vtts_tts_host(self.h, _ptr(tokens), _ptr(lens), B, L, float(silence_duration), mode, int(seed or 0),
                                        cap, _ptr(dur), _ptr(nf), C.byref(nmax), _ptr(wav))
            if rc == 0 or not (0 < cap < nmax.value):
                break
            cap = int(nmax.value)       # buffer too small: the call reported the size it needs
        self._ck(rc)
        n = int(nmax.value)
        wav = wav[: B * n * config.HOP].reshape(B, n * config.HOP)
        return [wav[b, : int(nf[b]) * config.HOP].copy() for b in range(B)], dur

    def synthesize_many(self, utterances, seed=None, masks=None, max_pad_frac=0.08, max_rows=32):
        """Mixed-length workload (BASELINE configs[4]): `utterances` is a list of (tokens list[int],
        durations_in_frames f32[L]).  They are bucketed by frame count so that padding stays below
        `max_pad_frac`, each bucket runs as one ragged batch, and the waveforms come back in input order
        (list of np.float32 [256*n_frames_i]).  Row i of any bucket equals utterance i run alone."""
        from .parallel import bucket_by_length
        nfs = [int(np.sum(np.asarray(d, np.float32), dtype=np.float32)) for _, d in utterances]
        out = [None] * len(utterances)
        for bucket in bucket_by_length(nfs, max_pad_frac, max_rows):
            Lmax = max(len(utterances[i][0]) for i in bucket)
            tok = np.zeros((len(bucket), Lmax), np.int32)
            dur = np.zeros((len(bucket), Lmax), np.float32)
            lens = np.zeros(len(bucket), np.int32)
            for r, i in enumerate(bucket):
                t, d = utterances[i]
                tok[r, : len(t)] = t
                dur[r, : len(t)] = d
                lens[r] = len(t)
            nf = np.asarray([nfs[i] for i in bucket], np.int32)
            m = None if masks is None else np.stack([np.asarray(masks[i])[: nf.max()] if np.asarray(masks[i]).shape[0] >= nf.max()
                                                     else np.pad(np.asarray(masks[i]), ((0, nf.max() - np.asarray(masks[i]).shape[0]), (0, 0), (0, 0)))
                                                     for i in bucket])
            wav = self.synthesize(tok, dur, lengths=lens, n_frames=nf, masks=m, seed=seed)
            for r, i in enumerate(bucket):
                out[i] = wav[r, : nfs[i] * config.HOP].copy()
        return out

    def _tf_masks(self, B, N, keep_masks, zone_masks, seed):
        if keep_masks is not None or zone_masks is not None:
            if keep_masks is None or zone_masks is None:
                raise ValueError("keep_masks and zone_masks must be given together")
            km = _np(keep_masks, np.uint8, (B, N, 2, config.PRENET_DIM), "keep_masks")
            zm = _np(zone_masks, np.uint8, (B, N, 4, config.ACOUSTIC_DECODER_DIM), "zone_masks")
            return km, zm, DROPOUT_MASK
        return None, None, (DROPOUT_SEED if seed is not None else DROPOUT_OFF)

    def teacher_forced(self, tokens, dur_frames, mels_in, lengths=None, n_frames=None, keep_masks=None, zone_masks=None, seed=None):
        """AcousticModel.__call__ (nat/model.py:146-169, is_training=False): tokens int [B,L], durations in frames
        [B,L], mels_in f32 [B,N,80] (ground truth shifted by one frame) -> (mel1, mel2) f32 [B,N,80].
        keep_masks uint8 [B,N,2,256] / zone_masks uint8 [B,N,4,512] (1 = keep previous state), else `seed` for the
        on-device stream, else both off.  Host buffers; the device work is vtts_acoustic_teacher_forward."""
        import torch
        tokens = _np(tokens, np.int32)
        B, L = tokens.shape
        mels_in = _np(mels_in, np.float32)
        N = mels_in.shape[1]
        if mels_in.shape != (B, N, config.MEL_DIM):
            raise ValueError(f"mels_in must be [B,N,{config.MEL_DIM}]")
        if B > MAX_ACOUSTIC_ROWS:
            raise ValueError(f"teacher_forced: at most {MAX_ACOUSTIC_ROWS} rows per call")
        km, zm, mode = self._tf_masks(B, N, keep_masks, zone_masks, seed)
        dev = torch.device("cuda", self.device)
        up = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)   # noqa: E731
        t_tok, t_dur, t_in = up(tokens), up(_np(dur_frames, np.float32, (B, L), "durations")), up(mels_in)
        t_len = up(None if lengths is None else _np(lengths, np.int32, (B,), "lengths"))
        t_nf = up(None if n_frames is None else _np(n_frames, np.int32, (B,), "n_frames"))
        t_km, t_zm = up(km), up(zm)
        m1 = torch.empty((B, N, config.MEL_DIM), dtype=torch.float32, device=dev)
        m2 = torch.empty_like(m1)
        st = torch.cuda.current_stream(dev).cuda_stream
        self._ck(self.lib.vtts_acoustic_teacher_forward(self.h, _ptr(t_tok), _ptr(t_len), _ptr(t_dur), _ptr(t_nf), _ptr(t_in), _ptr(t_km),
                                                        _ptr(t_zm), mode, int(seed or 0), B, L, N, _ptr(m1), _ptr(m2), st))
        torch.cuda.synchronize(dev)
        return m1.cpu().numpy(), m2.cpu().numpy()

    def gta(self, wav_i16, tokens, dur_sec, lengths=None, wav_lengths=None, keep_masks=None, zone_masks=None, seed=None, return_gt=False):
        """forward_fn of nat/gta.py:28-44 in one library call: int16 wavs [B,S] + aligned phonemes -> mel2_hat
        f32 [B,S/256,80] (rows past wav_lengths[b]//256 are 0)."""
        if not self._mel_loaded:
            self.load_mel_filterbank()
        wav = np.ascontiguousarray(np.asarray(wav_i16))
        if wav.dtype != np.int16 or wav.ndim != 2:
            raise ValueError("wav_i16 must be int16 [B,S]")
        B, S = wav.shape
        tokens = _np(tokens, np.int32)
        if tokens.ndim != 2 or tokens.shape[0] != B:
            raise ValueError("tokens must be [B,L]")
        L = tokens.shape[1]
        if B > MAX_ACOUSTIC_ROWS:
            raise ValueError(f"gta: at most {MAX_ACOUSTIC_ROWS} rows per call")
        N = S // config.HOP
        km, zm, mode = self._tf_masks(B, N, keep_masks, zone_masks, seed)
        lens = None if lengths is None else _np(lengths, np.int32, (B,), "lengths")
        wl = None if wav_lengths is None else _np(wav_lengths, np.int32, (B,), "wav_lengths")
        gt = np.empty((B, N, config.MEL_DIM), np.float32) if return_gt else None
        out = np.empty((B, N, config.MEL_DIM), np.float32)
        self._ck(self.lib.vtts_gta_host(self.h, _ptr(wav), _ptr(wl), _ptr(tokens), _ptr(lens), _ptr(_np(dur_sec, np.float32, (B, L), "durations")),
                                        _ptr(km), _ptr(zm), mode, int(seed or 0), B, L, S, _ptr(gt), _ptr(out)))
        return (out, gt) if return_gt else out

    def melspec(self, wav) -> np.ndarray:
        """MelFilter.__call__ (nat/dsp.py:115-128): wav f32 [B,S] -> log-mel [B,S/256,80]."""
        if not self._mel_loaded:
            self.load_mel_filterbank()
        wav = _np(wav, np.float32)
        assert wav.ndim == 2, "MelFilter expects [B,S] (dsp.py:118)"
        B, S = wav.shape
        mel = np.empty((B, S // config.HOP, config.MEL_DIM), np.float32)
        self._ck(self.lib.vtts_melspec_host(self.h, _ptr(wav), B, S, _ptr(mel)))
        return mel

    def debug_read(self, name: str, shape) -> np.ndarray:
        out = np.empty(shape, np.float32)
        self._ck(self.lib.vtts_debug_read(self.h, name.encode(), _ptr(out), out.size))
        return out

    # ---- device-pointer calls (torch tensors as memory containers) --------------------
    def hifigan_forward(self, mel_t, n_frames_t=None, out=None, stream=None):
        import torch
        assert mel_t.is_cuda and mel_t.dtype == torch.float32 and mel_t.is_contiguous()
        B, T, _ = mel_t.shape
        if out is None:
            out = torch.empty((B, T * config.HOP), dtype=torch.float32, device=mel_t.device)
        st = torch.cuda.current_stream(mel_t.device).cuda_stream if stream is None else stream
        self._ck(self.lib.vtts_hifigan_forward(self.h, _ptr(mel_t), _ptr(n_frames_t), B, T, _ptr(out), st))
        return out

    def acoustic_forward(self, tokens_t, dur_t, N, lengths_t=None, n_frames_t=None, masks_t=None, seed=None, out=None, stream=None):
        import torch
        assert tokens_t.is_cuda and tokens_t.dtype == torch.int32 and dur_t.dtype == torch.float32
        B, L = tokens_t.shape
        if out is None:
            out = torch.empty((B, N, config.MEL_DIM), dtype=torch.float32, device=tokens_t.device)
        mode = DROPOUT_MASK if masks_t is not None else (DROPOUT_SEED if seed is not None else DROPOUT_OFF)
        st = torch.cuda.current_stream(tokens_t.device).cuda_stream if stream is None else stream
        self._ck(self.lib.vtts_acoustic_forward(self.h, _ptr(tokens_t), _ptr(lengths_t), _ptr(dur_t), _ptr(n_frames_t),
                                                _ptr(masks_t), mode, int(seed or 0), B, L, int(N), _ptr(out), st))
        return out

    def duration_forward(self, tokens_t, lengths_t=None, out=None, stream=None):
        import torch
        assert tokens_t.is_cuda and tokens_t.dtype == torch.int32 and tokens_t.is_contiguous()
        B, L = tokens_t.shape
        if out is None:
            out = torch.empty((B, L), dtype=torch.float32, device=tokens_t.device)
        st = torch.cuda.current_stream(tokens_t.device).cuda_stream if stream is None else stream
        self._ck(self.lib.vtts_duration_forward(self.h, _ptr(tokens_t), _ptr(lengths_t), B, L, _ptr(out), st))
        return out

    def melspec_forward(self, wav_t, out=None, stream=None):
        import torch
        if not self._mel_loaded:
            self.load_mel_filterbank()
        B, S = wav_t.shape
        if out is None:
            out = torch.empty((B, S // config.HOP, config.MEL_DIM), dtype=torch.float32, device=wav_t.device)
        st = torch.cuda.current_stream(wav_t.device).cuda_stream if stream is None else stream
        self._ck(self.lib.vtts_melspec(self.h, _ptr(wav_t), B, S, _ptr(out), st))
        return out


_engines: dict = {}
_lock = threading.Lock()


def get_engine(device: int | None = None) -> Engine:
    """Process-wide engine per device (LOCAL_RANK by default under torchrun)."""
    import os
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    with _lock:
        if device not in _engines:
            _engines[device] = Engine(device)
        return _engines[device]
