"""GPU tests of the differentiable reconstruction (reconstruct_differentiable / reconstruct_spec_differentiable, avse_inverse_backward)
on the filterbanks and contexts the inverse serves, against finite differences of the shipped forward, and through the autograd
plumbing test_gpu_inverse_backward.py does not reach.

  * every bank of test_gpu_filterbanks.BANKS plus two specialised 22.05 kHz banks (F4 and band gather at cond ~5e4): a ragged batch
    with NaN past each row's length, an all-zero row with lengths 0 (no frame has a mixture), n slices <, = and > the mixture's
    frames, against the float64 VJP of tests/inverse_vjp.py built with the bank's filterbank (1e-4 of the peak), the forward
    bit-identical to reconstruct / reconstruct_spec;
  * the gradient is the derivative of what reconstruct computes: <g, y(m + hV) - y(m - hV)> / 2h of the float32 kernel output
    against <grad_mel, V>, for directions that isolate the first and last frames, the slice and chunk boundaries, single bands and
    the frames past T_use (the reference bank on a golden int16-scale mixture with ragged lengths, a band-gather bank, a refused
    bank on the generic kernels, an odd-n_fft generic geometry);
  * float16 / bfloat16 and non-contiguous leaves, a non-contiguous grad_out, stride-padded and B = 1 grad_pcm rows through the C ABI,
    an engine on a device that is not the current one."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import FRAME_RATES, GOLDEN_CASES, SR, FPS, oracle_pair
from tests.test_gpu_filterbanks import BANKS
from tests.test_gpu_inverse_backward import _want_spec, _abi_args

pytestmark = pytest.mark.gpu

TOL = 1e-4
H_DB = 0.05           # finite-difference step in dB: truncation ~ (ln10 / 20 h)^2 / 6 ~ 5e-6 relative

# (sample rate, video fps, slice ms, fmin, fmax, specialised): the nine banks of test_gpu_filterbanks and two specialised 22.05 kHz
# banks built as SpectralEngine(sr, sr / 640, 146, fmin, fmax, n_fft=640) (3 219 samples per slice: 20 frames per slice)
BANKS_BW = [b[:6] for b in BANKS] + [
    (22050, 22050 / 640, 146, 180.0, 7980.0, True),      # F4 + fused scan + I8
    (22050, 22050 / 640, 146, 1480.0, 7280.0, True),     # F2 band gather + I8, cond(F F^T) ~ 5e4
]
IDS = ["%d_%g_%g" % (b[0], b[3], b[4]) for b in BANKS_BW]


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


_ENGINES = {}


def _engine(mod, b):
    if b not in _ENGINES:
        kw = {"n_fft": 640} if b[0] == 22050 else {}
        _ENGINES[b] = mod.SpectralEngine(b[0], b[1], b[2], fmin=b[3], fmax=b[4], device="cuda:0", **kw)
    return _ENGINES[b]


@pytest.fixture(params=BANKS_BW, ids=IDS)
def bank(request, mod):
    b = request.param
    e = _engine(mod, b)
    assert e.specialised == b[5]
    assert (e.n_fft, e.hop, e.n_mels, e.spss) == (640, 160, 80, 20)
    return e, b


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _to_slices(spec, spss):
    """SPEC [..., 80, n spss] -> SLICES [..., n, 80, spss]."""
    *lead, m, t = spec.shape
    return np.ascontiguousarray(np.moveaxis(spec.reshape(*lead, m, t // spss, spss), -2, -3))


def _to_spec(sl):
    """SLICES [..., n, 80, spss] -> SPEC [..., 80, n spss]."""
    *lead, n, m, s = sl.shape
    return np.ascontiguousarray(np.moveaxis(sl, -3, -2).reshape(*lead, m, n * s))


def _err(got, want):
    assert got.shape == want.shape and np.isfinite(got).all()
    peak = np.max(np.abs(want))
    assert peak > 0
    return float(np.max(np.abs(got - want)) / peak)


def _signal(n, sr, seed):
    return (O.synth_speech(n, sr, seed) + 0.3 * O.synth_noise(n, seed + 1)).astype(np.float32)


def _backward(eng, pcm, mel, g, lengths, spec):
    """(grad_mel, y) through the differentiable entry point of the layout; pcm / mel / g numpy or CUDA tensors."""
    t = lambda x: x if torch.is_tensor(x) else _dev(x)
    m = t(mel).detach().clone().requires_grad_(True)
    fn = eng.reconstruct_spec_differentiable if spec else eng.reconstruct_differentiable
    y = fn(t(pcm), m, lengths=lengths)
    y.backward(t(g))
    return m.grad, y.detach()


def _forward(eng, pcm, mel, lengths, spec):
    fn = eng.reconstruct_spec if spec else eng.reconstruct
    return fn(_dev(pcm), _dev(mel), lengths=lengths)


# ---------------------------------------------------------------------------------------------------------------------------------
# B. the banks
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("frames", ["fewer", "equal", "more"])
@pytest.mark.parametrize("spec", [False, True], ids=["slices", "spec"])
def test_ragged_batch_against_the_vjp(bank, spec, frames):
    """Three rows, lengths L, L - 3001 and L / 2 + 11 with NaN past each (never read); 5 slices = 100 mel frames against a mixture of
    106, 100 or 91 frames."""
    eng, b = bank
    sr = b[0]
    L = {"fewer": 160 * 105, "equal": 160 * 99 + 50, "more": 160 * 90}[frames]
    T = eng.n_frames(L)
    assert T == {"fewer": 106, "equal": 100, "more": 91}[frames]
    rng = np.random.RandomState(int(b[3] + b[4]) + L)
    lens = np.array([L, L - 3001, L // 2 + 11], np.int32)
    B = len(lens)
    pcm = np.full((B, L), np.nan, np.float32)
    for i, n in enumerate(lens):
        pcm[i, :n] = _signal(n, sr, 90 + i)
    mel = (-40.0 + 12.0 * rng.randn(B, 80, 100)).astype(np.float32)
    T_use = min(100, T)
    g = rng.randn(B, 160 * (T_use - 1)).astype(np.float32)
    x = mel if spec else _to_slices(mel, 20)
    d_lens = _dev(lens)
    grad, y = _backward(eng, pcm, x, g, d_lens, spec)
    grad, y = grad.cpu().numpy(), y.cpu().numpy()
    assert np.array_equal(y, _forward(eng, pcm, x, d_lens, spec).cpu().numpy())
    assert np.isfinite(y).all()
    if not spec:
        grad = _to_spec(grad)
    assert np.all(grad[:, :, T_use:] == 0.0)
    worst = 0.0
    for i in range(B):
        want = _want_spec(mel[i], pcm[i], g[i], sr=sr, valid=int(lens[i]), fmin=b[3], fmax=b[4])
        worst = max(worst, _err(grad[i], want))
    print("WORST %s %s_%s %.3g" % ("%d_%g_%g" % (b[0], b[3], b[4]), "spec" if spec else "slices", frames, worst))
    assert worst <= TOL, worst


def test_empty_row_has_no_mixture_frame(bank):
    """Row 1 has lengths 0 and NaN everywhere: an all-zero mixture, phase 1 + 0j in every frame (no frame has a mixture)."""
    eng, b = bank
    L = 12000
    rng = np.random.RandomState(int(b[3]) + 7)
    pcm = np.full((2, L), np.nan, np.float32)
    pcm[0] = _signal(L, b[0], 5)
    lens = _dev(np.array([L, 0], np.int32))
    sl = (-40.0 + 12.0 * rng.randn(2, 3, 80, 20)).astype(np.float32)      # 60 frames of the mixture's 76
    g = rng.randn(2, 160 * 59).astype(np.float32)
    grad, y = _backward(eng, pcm, sl, g, lens, False)
    grad, y = _to_spec(grad.cpu().numpy()), y.cpu().numpy()
    assert np.array_equal(y, _forward(eng, pcm, sl, lens, False).cpu().numpy())
    mel = _to_spec(sl)
    errs = [_err(grad[i], _want_spec(mel[i], np.nan_to_num(pcm[i]) * (i == 0), g[i], sr=b[0], fmin=b[3], fmax=b[4])) for i in range(2)]
    print("WORST %s empty_row %.3g" % ("%d_%g_%g" % (b[0], b[3], b[4]), max(errs)))
    assert max(errs) <= TOL, errs


# ---------------------------------------------------------------------------------------------------------------------------------
# C. finite differences of the shipped inverse
# ---------------------------------------------------------------------------------------------------------------------------------
def _fd_context(mod, name, slices="mixed"):
    """(engine, pcm [B, L], mel in the layout, lengths or None, spec flag).  The golden context reconstructs from the mixture's own
    slices: in the speech slices bands 0 and 79 sit at the top_db floor, 80 dB under the loudest band, and a 0.05 dB step there
    moves y by less than its float32 resolution."""
    if name == "reference_golden_int16":
        eng = _engine(mod, BANKS[0][:6])
        o = oracle_pair(GOLDEN_CASES[2])                     # int16-scale, zero-padded speech
        pcm = np.stack([o["mixed_pcm"], o["mixed_pcm"]]).astype(np.float32)
        L = pcm.shape[1]
        pcm[1, 9001:] = np.nan
        sl = o[slices].astype(np.float32)
        sl = np.concatenate([sl, sl])[:6]                    # 120 frames against the mixture's 101
        sl = np.stack([sl, sl[::-1]])
        return eng, pcm, sl, _dev(np.array([L, 9001], np.int32)), False
    rng = np.random.RandomState(len(name))
    if name == "frame_rate_22k05_29.97":
        geo = next(g for g in FRAME_RATES if g["name"] == "22k05_29.97")
        eng = mod.SpectralEngine(geo["sr"], geo["fps"], 200, device="cuda:0", n_fft=geo["n_fft"])
        assert not eng.specialised and (eng.n_fft, eng.hop) == (735, 183)
        L = 183 * 70
    else:
        fmin, fmax, specialised = {"16000_1000_8000": (1000.0, 8000.0, True), "16000_550_4600": (550.0, 4600.0, False)}[name]
        eng = _engine(mod, (16000, 25.0, 200, fmin, fmax, specialised))
        L = 16000
    T = eng.n_frames(L)
    pcm = _signal(L, eng.sample_rate, 17)[None]
    mel = (-40.0 + 12.0 * rng.randn(1, 80, T + 9)).astype(np.float32)
    return eng, pcm, mel, None, True


FD_CONTEXTS = ["reference_golden_int16", "16000_1000_8000", "16000_550_4600", "frame_rate_22k05_29.97"]


def _directions(eng, shape_spec, T_use, seed):
    """name -> direction V in SPEC shape [B, 80, t_mel]."""
    B, _, t_mel = shape_spec
    rng = np.random.RandomState(seed)
    out = {"gaussian": rng.randn(*shape_spec)}
    for t in sorted({0, eng.spss - 1, eng.spss, 31, 32, T_use - 1}):
        v = np.zeros(shape_spec)
        v[:, :, t] = rng.randn(B, 80)
        out["frame_%d" % t] = v
    fb = eng.filterbank()
    widest = int(np.argmax((fb > 0).sum(axis=1)))
    for m in sorted({0, 79, widest}):
        v = np.zeros(shape_spec)
        v[:, m, :] = rng.randn(B, t_mel)
        out["band_%d%s" % (m, "_widest" if m == widest else "")] = v
    v = np.zeros(shape_spec)
    v[:, :, T_use:] = rng.randn(B, 80, t_mel - T_use)
    out["past_T_use"] = v
    return out


def _fd_residuals(eng, pcm, mel, lengths, spec, h=H_DB, min_band=0.0):
    """direction -> |D_fd - D_bw| / sum |grad_mel V| (see the test below).  A band direction whose band carries less than `min_band`
    of the peak |grad_mel| is left out (returned in the second dict with that fraction)."""
    B, L = pcm.shape
    spec_mel = mel if spec else _to_spec(mel)
    T_use = min(spec_mel.shape[2], eng.n_frames(L))
    g = np.random.RandomState(3).randn(B, eng.hop * (T_use - 1)).astype(np.float32)
    grad, y0 = _backward(eng, pcm, mel, g, lengths, spec)
    grad = grad.cpu().numpy().astype(np.float64)
    y0 = y0.cpu().numpy()
    assert np.isfinite(y0).all() and np.isfinite(grad).all()
    g64 = g.astype(np.float64)
    resid, unresolved = {}, {}
    peak = np.max(np.abs(grad))
    for dname, V in _directions(eng, spec_mel.shape, T_use, 11).items():
        if dname.startswith("band_"):
            share = np.max(np.abs(_to_spec(grad) if not spec else grad)[:, int(dname.split("_")[1]), :]) / peak
            if share < min_band:
                unresolved[dname] = share
                continue
        Vl = V if spec else _to_slices(V, eng.spss)
        mp = (mel + h * Vl).astype(np.float32)
        mm = (mel - h * Vl).astype(np.float32)
        yp = _forward(eng, pcm, mp, lengths, spec).cpu().numpy()
        ym = _forward(eng, pcm, mm, lengths, spec).cpu().numpy()
        Vr = (mp.astype(np.float64) - mm.astype(np.float64)) / (2 * h)
        terms = grad * Vr
        if dname == "past_T_use":
            assert np.array_equal(yp, y0) and np.array_equal(ym, y0)
            assert np.all(terms == 0.0) and np.all(grad[Vr != 0.0] == 0.0)
            resid[dname] = 0.0
            continue
        d_fd = float(np.sum(g64 * (yp.astype(np.float64) - ym.astype(np.float64)))) / (2 * h)
        d_bw = float(np.sum(terms))
        scale = float(np.sum(np.abs(terms)))
        assert scale > 0, dname
        resid[dname] = abs(d_fd - d_bw) / scale
    return resid, unresolved


# cond(F F^T) ~ 2e15: pinv(F) amplifies float32 rounding, and the float32 forward resolves y to ~3.5e-7 of its peak.  A 0.05 dB step
# in one frame then moves y by little more than that (measured residual 1.2e-5 ... 2.6e-4 at h = 0.02 ... 0.1 dB, not falling with h:
# rounding, not truncation), and a band carrying 1e-5 ... 1e-7 of the peak gradient (bands 0, 77, 79) moves it by less: for those
# the kernel's gradient is checked band by band against the float64 VJP instead, where it agrees to 1e-7 of the band's own peak.
FD_TOL = {"16000_550_4600": 1e-3}
FD_MIN_BAND = {"16000_550_4600": 1e-3}
FD_BANK_EDGES = {"16000_550_4600": (550.0, 4600.0)}


@pytest.mark.parametrize("name", FD_CONTEXTS)
def test_gradient_matches_finite_differences_of_reconstruct(mod, name):
    """|<g, y(m + hV) - y(m - hV)> / 2h - <grad_mel, V>| <= 1e-4 sum |grad_mel V|, y the float32 output of reconstruct /
    reconstruct_spec, h = 0.05 dB and the sums in float64.  V is the direction the float32 inputs m +- hV realise, (m_+ - m_-) / 2h.
    Along a direction confined to the frames past T_use, y does not change by a bit and the gradient there is exactly 0."""
    ctx = _fd_context(mod, name)
    resid, unresolved = _fd_residuals(*ctx, min_band=FD_MIN_BAND.get(name, 0.0))
    print("WORST fd %s %.3g (%s)" % (name, max(resid.values()), ", ".join("%s %.2g" % kv for kv in resid.items())))
    assert max(resid.values()) <= FD_TOL.get(name, TOL), resid
    if unresolved:
        eng, pcm, mel, lengths, spec = ctx
        assert spec and lengths is None and pcm.shape[0] == 1
        T_use = min(mel.shape[2], eng.n_frames(pcm.shape[1]))
        g = np.random.RandomState(3).randn(1, eng.hop * (T_use - 1)).astype(np.float32)
        grad = _backward(eng, pcm, mel, g, None, True)[0].cpu().numpy()[0]
        fmin, fmax = FD_BANK_EDGES[name]
        want = _want_spec(mel[0], pcm[0], g[0], fmin=fmin, fmax=fmax)
        for dname in unresolved:
            b = int(dname.split("_")[1])
            err = np.max(np.abs(grad[b] - want[b])) / np.max(np.abs(want[b]))
            print("band-relative %s %s %.3g (band share of the peak gradient %.2g)" % (name, dname, err, unresolved[dname]))
            assert err <= TOL, (dname, err)


# ---------------------------------------------------------------------------------------------------------------------------------
# E. autograd plumbing
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng(mod):
    return _engine(mod, BANKS[0][:6])


def _plumbing_case(seed=61, B=2, L=16000, T_mel=101):
    rng = np.random.RandomState(seed)
    pcm = np.stack([_signal(L, SR, seed + i) for i in range(B)])
    mel = (-40.0 + 12.0 * rng.randn(B, 80, T_mel)).astype(np.float32)
    g = rng.randn(B, 160 * (min(T_mel, 1 + L // 160) - 1)).astype(np.float32)
    return pcm, mel, g


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_precision_leaves(eng, dtype):
    """A float16 / bfloat16 leaf gets the float32 gradient of its float32 values, cast to its dtype."""
    pcm, mel, g = _plumbing_case()
    m = _dev(mel).to(dtype).requires_grad_(True)
    y = eng.reconstruct_spec_differentiable(_dev(pcm), m)
    y.backward(_dev(g))
    assert m.grad.dtype == dtype
    ref, y32 = _backward(eng, pcm, m.detach().float(), g, None, True)
    assert torch.equal(y, y32)
    assert torch.equal(m.grad, ref.to(dtype))


def test_non_contiguous_leaf_and_grad_out(eng):
    """SPEC built as x.transpose(1, 2) from a [B, T, 80] leaf, and a loss on y.t() (autograd hands over a transposed grad_out)."""
    pcm, mel, g = _plumbing_case(62)
    ref, y_ref = _backward(eng, pcm, mel, g, None, True)
    x = _dev(np.ascontiguousarray(mel.transpose(0, 2, 1))).requires_grad_(True)
    y = eng.reconstruct_spec_differentiable(_dev(pcm), x.transpose(1, 2))
    assert torch.equal(y, y_ref)
    (y.t() * _dev(np.ascontiguousarray(g.T))).sum().backward()
    assert torch.equal(x.grad, ref.transpose(1, 2))


def test_grad_pcm_rows_through_the_c_abi(mod, eng):
    """grad_pcm rows with a NaN gap between them (never read), and B = 1 with grad_pcm_stride < out_len (allowed: one row)."""
    pcm, mel, g = _plumbing_case(63, B=3)
    d_pcm, d_mel = _dev(pcm), _dev(mel)
    ref, _ = _backward(eng, pcm, mel, g, None, True)
    out_len = g.shape[1]
    padded = torch.full((3, out_len + 37), float("nan"), device="cuda")
    padded[:, :out_len] = _dev(g)
    a = _abi_args(mod, d_mel, d_pcm, 1, n_frames=101, ld_t=101)
    stream = torch.cuda.current_stream().cuda_stream
    got = torch.full_like(d_mel, float("nan"))
    assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a), padded.data_ptr(), padded.stride(0), got.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(got, ref)
    a1 = _abi_args(mod, d_mel[:1], d_pcm[:1], 1, n_frames=101, ld_t=101)
    got1 = torch.full_like(d_mel[:1], float("nan"))
    for stride in (0, out_len // 2):
        got1.fill_(float("nan"))
        assert eng._lib.avse_inverse_backward(eng._ctx, ctypes.byref(a1), padded.data_ptr(), stride, got1.data_ptr(), stream) == 0
        torch.cuda.synchronize()
        assert torch.equal(got1[0], ref[0])


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_engine_on_a_device_that_is_not_current(mod, eng):
    """An engine on cuda:1 driven while cuda:0 is current: forward and gradient bit-identical to the cuda:0 engine's."""
    pcm, mel, g = _plumbing_case(64)
    ref, y_ref = _backward(eng, pcm, mel, g, None, True)
    e1 = mod.SpectralEngine(SR, FPS, 200, device="cuda:1")
    with torch.cuda.device(0):
        m = torch.from_numpy(mel).to("cuda:1").requires_grad_(True)
        y = e1.reconstruct_spec_differentiable(torch.from_numpy(pcm).to("cuda:1"), m)
        y.backward(torch.from_numpy(g).to("cuda:1"))
        assert torch.cuda.current_device() == 0
    assert y.device == torch.device("cuda:1") and m.grad.device == torch.device("cuda:1")
    assert torch.equal(y.cpu(), y_ref.cpu()) and torch.equal(m.grad.cpu(), ref.cpu())
