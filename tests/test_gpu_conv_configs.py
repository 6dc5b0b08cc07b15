"""Every conv configuration the models launch, one layer at a time, against float64.

The models reach the dense conv engines (tc_conv.cu on the tensor cores, conv1d.cu in strict fp32) through the conv
dispatcher and the generator's up-sampling stage.  vtts_debug_conv and vtts_debug_conv_transpose run exactly those code
paths on the real shapes: partial N tiles (80 output channels), BatchNorm with tanh / relu, several N tiles, inputs of
80 channels, launches of several problems with different k, multi-phase ConvTranspose tiles (the 4-phase CTA-pair form
at C = 256) over the 3-way mean, and the flattened B = 1 GEMM form.

Each case checks, in both precisions:
  * every valid output row within L-inf <= tol * max(1, |ref|_inf) of a float64 torch reference written out here
    (bf16x3 2e-4, fp32 2e-5);
  * output rows of tau >= len[b]*len_mul (ConvTranspose: their u output rows) and a guard region after each output
    buffer still hold the sentinel they were filled with;
  * bf16x3: the float64 result of the same operands rounded to bf16 (no lo terms) misses the reference by at least 5x
    the tolerance, so a tile that drops a correction term fails.
Geometry: row counts that are not a multiple of any tile, more tiles than SMs (the persistent loop wraps), and ragged
rows -- one ending in the second CTA's half of a pair tile, one of 2 rows (shorter than the halo), one on a tile
boundary, one full."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import hifigan_oracle as ho

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
TOL = {"bf16x3": 2e-4, "fp32": 2e-5}
NOLO_MARGIN = 5.0
SENT = 0x7FC0DEAD          # a NaN bit pattern no kernel produces
GUARD = 4096               # sentinel floats after every output buffer
MIN_TILES = 160            # > 148 SMs and > 74 CTA pairs
SLOPE = 0.1


@pytest.fixture(scope="module")
def eng():
    from viettts_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


# The two helpers below restate tc_conv.cu's tile choice (vtts_tc_tile_n, and MT / CTA pairs in launch_ne for the default
# tc_variant 3) so that the geometry below lands on tile edges.  launch_ne points back here: change them together, or
# the ragged-row and wrap-around cases stop hitting the edges they are meant to (the correctness checks still pass).
def _tile_n(cout):
    return 32 if cout <= 32 else 64 if cout <= 64 else 128 if cout <= 128 else 256


def _tile_rows(n, nph=1):
    """Rows of one tile of tc_conv.cu in its default form: 128 * MT, twice that for the CTA pairs (N >= 128)."""
    mt = {(256, 1): 1, (128, 1): 2, (128, 4): 1, (64, 1): 4, (64, 2): 2, (32, 1): 4, (32, 2): 4}[(n, nph)]
    return 128 * mt * (2 if n >= 128 else 1)


def _ragged(tile, units, B=4):
    """(T, lens) with B rows and at least MIN_TILES tiles over `units` tile problems: T is no multiple of the tile;
    the lengths are full, ending in the second half of a tile, 2 rows, and on a tile boundary."""
    tpr = max(4, math.ceil(MIN_TILES / (units * B)))
    T = tpr * tile + 77
    return T, np.array([T, (tpr // 2) * tile + tile // 2 + 3, 2, 3 * tile], np.int32)[:B]


def _sentinel(shape):
    n = int(np.prod(shape))
    buf = torch.full((n + GUARD,), SENT, dtype=torch.int32, device=DEV)
    return buf, buf[:n].view(torch.float32).view(shape)


def _g(rng, *shape, scale=1.0):
    return torch.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32)).to(DEV)


def _bf16(t):
    return t.to(torch.bfloat16).double()


def _check(tag, prec, errs, ref_max, untouched_ok, guard_ok, nolo_err=None):
    """errs: one L-inf per (problem, batch row); a NaN entry (a valid row left at the sentinel, or a NaN the kernel
    computed) fails wherever it is in the list -- Python's max() would skip it unless it came first."""
    tol = TOL[prec] * max(1.0, ref_max)
    err = max(errs, key=lambda e: math.inf if math.isnan(e) else e)
    msg = f"[{tag} {prec}] Linf={err:.3e} tol={tol:.2e} |ref|={ref_max:.2f}"
    if nolo_err is not None:
        msg += f" bf16-only Linf={nolo_err:.3e} ({nolo_err / tol:.1f}x tol)"
    print(msg)
    assert all(e <= tol for e in errs), msg
    assert untouched_ok, f"{tag} {prec}: rows past the valid length were written"
    assert guard_ok, f"{tag} {prec}: the guard region after the output was written"
    if nolo_err is not None:
        assert nolo_err >= NOLO_MARGIN * tol, f"{tag}: the tolerance would not notice a missing correction term ({msg})"


# ---------------------------------------------------------------------------------------------------------------------
# conv dispatcher: the production matrix
# ---------------------------------------------------------------------------------------------------------------------
# name, Cin, Cout, problems [(k, dil)], residual, BatchNorm, post_act (1 tanh, 2 relu), pre_mode (1 = lrelu 0.1), flat
CONFIGS = [
    # acoustic model (nat.cu)
    ("encoder_conv_bn_relu", 256, 256, [(3, 1)], False, True, 2, 0, False),
    ("postnet0_80_bn_tanh", 80, 512, [(5, 1)], False, True, 1, 0, False),
    ("postnet_512_bn_tanh", 512, 512, [(5, 1)], False, True, 1, 0, False),
    ("postnet4_512_to_80_resid", 512, 80, [(5, 1)], True, False, 0, 0, False),
    ("projection_1024_to_80", 1024, 80, [(1, 1)], False, False, 0, 0, False),
    ("gemm_encoder_lstm_256x1024x2", 256, 1024, [(1, 1), (1, 1)], False, False, 0, 0, True),
    ("gemm_decoder_512x2048x2", 512, 2048, [(1, 1), (1, 1)], False, False, 0, 0, True),
    ("gemm_teacher_768x2048x2", 768, 2048, [(1, 1), (1, 1)], False, False, 0, 0, True),
    ("gemm_prenet_80x256", 80, 256, [(1, 1)], False, False, 0, 0, True),
    ("gemm_duration_fc1_512x256", 512, 256, [(1, 1)], False, False, 0, 0, True),
    # generator (hifigan.cu)
    ("conv_pre_80_to_512", 80, 512, [(7, 1)], False, False, 0, 0, False),
] + [
    (f"resblock{c}_conv1_d{d}", c, c, [(3, d), (7, d), (11, d)], False, False, 0, 1, False) for c in (256, 128, 64, 32) for d in (1, 5)
] + [
    (f"resblock{c}_conv2_resid", c, c, [(3, 1), (7, 1), (11, 1)], True, False, 0, 1, False) for c in (256, 128, 64, 32)
]


def _ref_conv(x, w, b, k, dil, pre_mode, bn, act, resid):
    """float64 hk.Conv1D (SAME: zero padding (k-1)*dil/2 at both ends) of one row x [n, Cin] as one matrix product per
    tap -> bias -> BatchNorm -> activation -> + residual."""
    if pre_mode == 1:
        x = F.leaky_relu(x, SLOPE)
    n, pad = x.shape[0], (k - 1) * dil // 2
    xp = F.pad(x, (0, 0, pad, pad))
    y = sum(xp[j * dil : j * dil + n] @ w[j] for j in range(k)) + b
    if bn is not None:
        mean, inv, off = bn
        y = (y - mean) * inv + off
    if act == 1:
        y = torch.tanh(y)
    elif act == 2:
        y = torch.relu(y)
    return y if resid is None else y + resid


def _make_conv_case(name, seed):
    name, Cin, Cout, kd, has_res, has_bn, act, pre, flat = next(c for c in CONFIGS if c[0] == name)
    rng = np.random.default_rng(seed)
    tile = _tile_rows(_tile_n(Cout))
    units = len(kd) * math.ceil(Cout / _tile_n(Cout))
    if flat:
        B, lens = 1, None
        T = max(4, math.ceil(MIN_TILES / units)) * tile + 77
    else:
        B = 4
        T, lens = _ragged(tile, units, B)
    x = _g(rng, B, T, Cin)
    probs = []
    for k, dil in kd:
        p = dict(x0=x, w=_g(rng, k, Cin, Cout, scale=1 / np.sqrt(k * Cin)), bias=_g(rng, Cout, scale=0.1), k=k, dil=dil,
                 in_off=-((k - 1) * dil // 2))
        if has_res:
            p["resid"] = _g(rng, B, T, Cout)
        if has_bn:
            scale = rng.uniform(0.8, 1.25, Cout)
            var = rng.uniform(0.6, 1.6, Cout)
            p["bn_mean"] = _g(rng, Cout, scale=0.5)
            p["bn_inv"] = torch.from_numpy((scale / np.sqrt(var + 1e-5)).astype(np.float32)).to(DEV)
            p["bn_off"] = _g(rng, Cout, scale=0.3)
        probs.append(p)
    geom = dict(B=B, T_rows=T, rows_out=T, Cin=Cin, Cout=Cout, pre_mode=pre, pre_slope=SLOPE if pre else 1.0, post_act=act,
                len_t=None if lens is None else torch.from_numpy(lens).to(DEV))
    return geom, probs, lens, act


def _run_conv(eng, prec, geom, probs):
    bufs = []
    for p in probs:
        buf, p["out"] = _sentinel((geom["B"], geom["rows_out"], geom["Cout"]))
        bufs.append(buf)
    eng.debug_conv(prec, probs, **geom)
    return bufs


@pytest.mark.parametrize("prec", ["bf16x3", "fp32"])
@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
def test_conv_config_vs_float64(eng, name, prec):
    geom, probs, lens, act = _make_conv_case(name, sum(map(ord, name)))
    bufs = _run_conv(eng, prec, geom, probs)
    B, T, Cout = geom["B"], geom["T_rows"], geom["Cout"]
    errs, ref_max, untouched, nolo = [], 0.0, True, None
    for pi, (p, buf) in enumerate(zip(probs, bufs)):
        d = lambda key: None if p.get(key) is None else p[key].double()  # noqa: E731
        bn = (d("bn_mean"), d("bn_inv"), d("bn_off")) if "bn_mean" in p else None
        out = p["out"].double()
        words = buf[: B * T * Cout].view(B, T, Cout)
        for b in range(B):
            n = T if lens is None else int(lens[b])
            res = None if p.get("resid") is None else d("resid")[b, :n]
            ref = _ref_conv(p["x0"][b, :n].double(), d("w"), d("bias"), p["k"], p["dil"], geom["pre_mode"], bn, act, res)
            errs.append(float((out[b, :n] - ref).abs().max()))
            ref_max = max(ref_max, float(ref.abs().max()))
            untouched &= bool((words[b, n:] == SENT).all())
            if prec == "bf16x3" and pi == 0 and b == 0:
                # the same operands rounded to bf16, no lo terms, in float64 on the host: a window of 1024 rows
                k, dil = p["k"], p["dil"]
                W = min(n, 1024)
                xw = p["x0"][0, : W + (k - 1) * dil // 2].double().cpu()
                if geom["pre_mode"] == 1:
                    xw = F.leaky_relu(xw, SLOPE)
                bnc = None if bn is None else tuple(t.cpu() for t in bn)
                rw = None if res is None else res[: W + (k - 1) * dil // 2].cpu()
                y = _ref_conv(_bf16(xw), _bf16(d("w").cpu()), d("bias").cpu(), k, dil, 0, bnc, act, rw)[:W]
                nolo = float((y - ref[:W].cpu()).abs().max())
    guard = all(bool((buf[B * T * Cout :] == SENT).all()) for buf in bufs)
    _check(name, prec, errs, ref_max, untouched, guard, nolo)


def test_check_fails_on_a_nan_in_any_row():
    """A valid row that still holds the NaN sentinel fails the check in every position, not only the first."""
    for pos in range(4):
        errs = [1e-6] * 4
        errs[pos] = math.nan
        with pytest.raises(AssertionError):
            _check("nan", "fp32", errs, 1.0, True, True)


def test_conv_hook_rejects_malformed_descriptors(eng):
    from viettts_b200 import _lib
    x = torch.zeros((1, 64, 32), device=DEV)
    w = torch.zeros((3, 32, 32), device=DEV)
    b = torch.zeros(32, device=DEV)
    out = torch.zeros((1, 64, 32), device=DEV)
    ok = dict(x0=x, w=w, bias=b, out=out, k=3, dil=1, in_off=-1)
    geom = dict(B=1, T_rows=64, rows_out=64, Cin=32, Cout=32)
    eng.debug_conv("bf16x3", [ok], **geom)
    bad = [
        ([], geom),
        ([ok] * 9, geom),
        ([ok], dict(geom, Cin=24)),
        ([ok], dict(geom, Cout=30)),
        ([dict(ok, bn_mean=b, bn_inv=b)], geom),
        ([dict(ok, bn_off=b)], geom),
        ([ok], dict(geom, pre_mode=2)),
        ([dict(ok, x1=x)], dict(geom, pre_mode=2)),
        ([dict(ok, x1=x)], geom),
        ([dict(ok, x1=x, x2=x)], geom),
        ([dict(ok, out_stride=2)], geom),
    ]
    for prec in ("bf16x3", "fp32"):
        for probs, g in bad:
            with pytest.raises(_lib.VttsError) as e:
                eng.debug_conv(prec, probs, **g)
            assert e.value.code == -1, (prec, len(probs), g)
    with pytest.raises(_lib.VttsError) as e:
        eng.debug_conv_transpose("bf16x3", torch.zeros((1, 8, 256), device=DEV), torch.zeros((4, 128, 256), device=DEV),
                                 torch.zeros(128, device=DEV), torch.zeros((1, 16, 128), device=DEV), 2)
    assert e.value.code == -1


# ---------------------------------------------------------------------------------------------------------------------
# ConvTranspose: the generator's four up-sampling stages
# ---------------------------------------------------------------------------------------------------------------------
STAGES = [(512, 8, 16), (256, 8, 16), (128, 2, 4), (64, 2, 4)]   # (C, u, K); stage 0 reads lrelu(x0), 1-3 the 3-way mean


def _make_ups_case(stage, len_mul, seed):
    C, u, K = STAGES[stage]
    Co = C // 2
    nph = 1 if Co == 256 else (4 if Co == 128 else 2)
    tile = _tile_rows(Co, nph)
    units = u // nph
    rng = np.random.default_rng(seed)
    B = 4
    T, lens = _ragged(tile, units, B)
    if len_mul > 1:
        Tm = math.ceil(T / len_mul)
        T = Tm * len_mul
        l2 = Tm // 2
        while (l2 * len_mul) % tile <= tile // 2:    # ends in the second half of a tile
            l2 += 1
        lens = np.array([Tm, l2, 1, Tm - 1], np.int32)
    xs = [_g(rng, B, T, C) for _ in range(1 if stage == 0 else 3)]
    w = _g(rng, K, Co, C, scale=1 / np.sqrt(2 * C))     # two taps reach every output row
    bias = _g(rng, Co, scale=0.1)
    return C, u, K, T, B, lens, xs, w, bias


def _ref_ups(xs, w, bias, u, b, n, device, round_bf16=False):
    """float64 lrelu(0.1) of x0 or of the 3-way mean, row b cut to its n valid rows -> oracle ConvTranspose(stride u);
    round_bf16: both operands rounded to bf16 after the activation."""
    x = xs[0][b, :n].double() if len(xs) == 1 else sum(t[b, :n].double() for t in xs) / 3
    x, w = F.leaky_relu(x.to(device), SLOPE), w.double().to(device)
    if round_bf16:
        x, w = _bf16(x), _bf16(w)
    return ho.conv1d_transpose_nwc(x[None], w, bias.double().to(device), u)[0]


_UPS_REFS = {}     # (stage, len_mul) -> float64 references of the valid rows, shared by both precisions


@pytest.mark.parametrize("prec", ["bf16x3", "fp32"])
@pytest.mark.parametrize("len_mul", [1, 64])
@pytest.mark.parametrize("stage", [0, 1, 2, 3])
def test_conv_transpose_stage_vs_float64(eng, stage, len_mul, prec):
    C, u, K, T, B, lens, xs, w, bias = _make_ups_case(stage, len_mul, 100 * stage + len_mul)
    Co = C // 2
    buf, out = _sentinel((B, T * u, Co))
    eng.debug_conv_transpose(prec, xs[0], w, bias, out, u, x1_t=xs[1] if stage else None, x2_t=xs[2] if stage else None,
                             len_t=torch.from_numpy(lens).to(DEV), len_mul=len_mul)
    words = buf[: B * T * u * Co].view(B, T * u, Co)
    valid = [min(int(lens[b]) * len_mul, T) for b in range(B)]
    if (stage, len_mul) not in _UPS_REFS:
        _UPS_REFS[(stage, len_mul)] = [_ref_ups(xs, w, bias, u, b, valid[b], DEV) for b in range(B)]
    errs, ref_max, untouched, nolo = [], 0.0, True, None
    for b in range(B):
        n = valid[b]
        ref = _UPS_REFS[(stage, len_mul)][b]
        errs.append(float((out[b, : n * u].double() - ref).abs().max()))
        ref_max = max(ref_max, float(ref.abs().max()))
        untouched &= bool((words[b, n * u :] == SENT).all())
        if prec == "bf16x3" and b == 0:
            # bf16-rounded operands, no lo terms, float64 on the host: output rows < W*u need input rows <= W
            W = min(n - 2, 256)
            y = _ref_ups(xs, w, bias, u, b, W + 2, "cpu", round_bf16=True)
            nolo = float((y[: W * u] - ref[: W * u].cpu()).abs().max())
    guard = bool((buf[B * T * u * Co :] == SENT).all())
    _check(f"conv_transpose_stage{stage}_len_mul{len_mul}", prec, errs, ref_max, untouched, guard, nolo)


# ---------------------------------------------------------------------------------------------------------------------
# the CTA-pair (tc_variant 3, default) and single-CTA (tc_variant 1) forms of tc_conv.cu compute the same products in
# the same order: bit-identical results, sentinels included
# ---------------------------------------------------------------------------------------------------------------------
def _pair_generic_case():
    """Partial N tile (80 of 128 columns) with BatchNorm, tanh and a residual: the generic epilogue of both forms."""
    rng = np.random.default_rng(7)
    Cin, Cout, k = 512, 80, 5
    T, lens = _ragged(_tile_rows(128), 1)
    x = _g(rng, 4, T, Cin)
    p = dict(x0=x, w=_g(rng, k, Cin, Cout, scale=1 / np.sqrt(k * Cin)), bias=_g(rng, Cout, scale=0.1), resid=_g(rng, 4, T, Cout),
             bn_mean=_g(rng, Cout, scale=0.5), bn_inv=_g(rng, Cout, scale=0.2) + 1.0, bn_off=_g(rng, Cout, scale=0.3), k=k, dil=1, in_off=-2)
    geom = dict(B=4, T_rows=T, rows_out=T, Cin=Cin, Cout=Cout, post_act=1, len_t=torch.from_numpy(lens).to(DEV))
    return geom, [p]


@pytest.mark.parametrize("case", ["generic_partial_bn", "gemm_decoder_512x2048x2", "resblock128_conv1_d5", "conv_transpose_stage1"])
def test_cta_pair_and_single_cta_forms_bit_identical(eng, case):
    outs = {}
    try:
        for variant in (1, 3):
            eng.tc_stats(False, variant=variant)
            if case == "conv_transpose_stage1":
                C, u, K, T, B, lens, xs, w, bias = _make_ups_case(1, 1, 11)
                buf, out = _sentinel((B, T * u, C // 2))
                eng.debug_conv_transpose("bf16x3", xs[0], w, bias, out, u, x1_t=xs[1], x2_t=xs[2], len_t=torch.from_numpy(lens).to(DEV))
                outs[variant] = [buf.cpu().numpy()]
            else:
                geom, probs = _pair_generic_case() if case == "generic_partial_bn" else _make_conv_case(case, 5)[:2]
                outs[variant] = [b.cpu().numpy() for b in _run_conv(eng, "bf16x3", geom, probs)]
    finally:
        eng.tc_stats(False, variant=3)
    for a, b in zip(outs[1], outs[3]):
        assert np.array_equal(a, b), case
