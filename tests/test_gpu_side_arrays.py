"""Per-row side arrays (lengths, noise lengths, SNRs) in whatever form a caller holds them: every SpectralEngine entry point that
forwards them to a kernel converts them to the contiguous int32 / float32 [B] device tensor the kernels read.  Without that, an int64
`lengths` such as torch.tensor([16000, 9001], device="cuda") was read as int32 pairs (row 1 saw the high word of 16000, 0, and was
processed as an empty utterance) and a float64 SNR of 10 dB as 0 dB in row 0.  Each form must give outputs bit-identical to the
int32 / float32 call; an array that does not hold one value per row raises ValueError."""
import importlib

import numpy as np
import pytest
import torch

from oracle import avse_oracle as O
from tests.cases import SR, FPS

pytestmark = pytest.mark.gpu

LENS = [16000, 9001, 4007]
NOISE_LENS = [16000, 5000, 1121]
SNR = [-5.0, 0.0, 7.5]
B, L, NVS = 3, 16000, 5


@pytest.fixture(scope="module")
def mod():
    return importlib.import_module("audio-visual-speech-enhancement_b200.engine")


@pytest.fixture(scope="module")
def eng(mod):
    return mod.SpectralEngine(SR, FPS, 200, device="cuda:0")


@pytest.fixture(scope="module")
def data():
    rng = np.random.RandomState(7)
    s = np.zeros((B, L), np.float32)
    z = np.zeros((B, L), np.float32)
    for i, n in enumerate(LENS):
        s[i, :n] = O.synth_speech(n, SR, 30 + i)
    for i, n in enumerate(NOISE_LENS):
        z[i, :n] = O.synth_noise(n, 40 + i)
    pcm = (s + 0.5 * z).astype(np.float32)
    sl = (-40.0 + 12.0 * rng.randn(B, NVS, 80, 20)).astype(np.float32)
    spec = (-40.0 + 12.0 * rng.randn(B, 80, 101)).astype(np.float32)
    g = rng.randn(B, 160 * 99).astype(np.float32)
    g_spec = rng.randn(B, 160 * 100).astype(np.float32)
    return {k: torch.from_numpy(v).cuda() for k, v in dict(s=s, z=z, pcm=pcm, sl=sl, spec=spec, g=g, g_spec=g_spec).items()}


def _int_forms(vals):
    """form -> the lengths in that form."""
    base = torch.tensor(vals, dtype=torch.int32, device="cuda")
    wide = torch.zeros(2 * len(vals), dtype=torch.int32, device="cuda")
    wide[::2] = base
    return {"wide_cuda": torch.tensor(vals, dtype=torch.int64, device="cuda"), "numpy_wide": np.array(vals, np.int64),
            "numpy_kernel_dtype": np.array(vals, np.int32), "list": list(vals), "strided_view": wide[::2],
            "cpu": torch.tensor(vals, dtype=torch.int32), "narrow_cuda": torch.tensor(vals, dtype=torch.int16, device="cuda")}


def _float_forms(vals):
    """form -> the SNRs in that form."""
    base = torch.tensor(vals, dtype=torch.float32, device="cuda")
    wide = torch.zeros(2 * len(vals), dtype=torch.float32, device="cuda")
    wide[1::2] = base
    return {"wide_cuda": torch.tensor(vals, dtype=torch.float64, device="cuda"), "numpy_wide": np.array(vals, np.float64),
            "numpy_kernel_dtype": np.array(vals, np.float32), "list": list(vals), "strided_view": wide[1::2],
            "cpu": torch.tensor(vals, dtype=torch.float32), "narrow_cuda": torch.tensor(vals, dtype=torch.float16, device="cuda")}


# wide: int64 / float64, narrow: int16 / float16 (the values here are exact in both), kernel dtype: int32 / float32
FORMS = ["wide_cuda", "numpy_wide", "numpy_kernel_dtype", "list", "strided_view", "cpu", "narrow_cuda"]


def _outs(x):
    """Flatten an entry point's result into a list of tensors."""
    if torch.is_tensor(x):
        return [x]
    if isinstance(x, dict):
        return [t for k in sorted(x) for t in _outs(x[k]) if k not in ("T", "ld_t", "n_slices", "layout")]
    if isinstance(x, (tuple, list)):
        return [t for v in x for t in _outs(v)]
    if hasattr(x, "buf"):                       # DbKeys
        return [x.buf] + ([x.equalizer] if x.equalizer is not None else [])
    return []


def _grad(fn, mel, g):
    m = mel.detach().clone().requires_grad_(True)
    y = fn(m)
    y.backward(g)
    return [y.detach(), m.grad]


def _calls(eng, d):
    """entry point -> fn(lengths, noise_lengths, snr_db) -> list of output tensors."""
    def forward_raw(ln, nl, snr):
        factor, keys = eng.snr_factor(d["s"], d["z"], lengths=_REF["lens"], snr_db=_REF["snr"], noise_lengths=_REF["nl"])
        return eng.forward_raw(d["s"], d["z"], L=L, len_speech=ln, len_noise=ln, factor=factor, n_slices=NVS, max_key=keys,
                               noise_lengths=nl)
    return {
        "snr_factor": lambda ln, nl, snr: eng.snr_factor(d["s"], d["z"], lengths=ln, snr_db=snr, noise_lengths=nl),
        "forward_raw": forward_raw,
        "preprocess_pairs": lambda ln, nl, snr: eng.preprocess_pairs(d["s"], d["z"], NVS, lengths=ln, snr_db=snr, noise_lengths=nl),
        "spectrogram": lambda ln, nl, snr: eng.spectrogram(d["pcm"], lengths=ln, stft=True),
        "preprocess_signals": lambda ln, nl, snr: eng.preprocess_signals(d["pcm"], NVS, lengths=ln),
        "reconstruct": lambda ln, nl, snr: eng.reconstruct(d["pcm"], d["sl"], lengths=ln),
        "reconstruct_spec": lambda ln, nl, snr: eng.reconstruct_spec(d["pcm"], d["spec"], lengths=ln),
        "reconstruct_differentiable": lambda ln, nl, snr: _grad(lambda m: eng.reconstruct_differentiable(d["pcm"], m, lengths=ln),
                                                                d["sl"], d["g"]),
        "reconstruct_spec_differentiable": lambda ln, nl, snr: _grad(
            lambda m: eng.reconstruct_spec_differentiable(d["pcm"], m, lengths=ln), d["spec"], d["g_spec"]),
    }


_REF = {}
ENTRIES = ["snr_factor", "forward_raw", "preprocess_pairs", "spectrogram", "preprocess_signals", "reconstruct", "reconstruct_spec",
           "reconstruct_differentiable", "reconstruct_spec_differentiable"]


@pytest.fixture(scope="module")
def ref(eng, data):
    _REF.update(lens=torch.tensor(LENS, dtype=torch.int32, device="cuda"), nl=torch.tensor(NOISE_LENS, dtype=torch.int32, device="cuda"),
                snr=torch.tensor(SNR, dtype=torch.float32, device="cuda"))
    calls = _calls(eng, data)
    out = {k: [t.clone() for t in _outs(fn(_REF["lens"], _REF["nl"], _REF["snr"]))] for k, fn in calls.items()}
    torch.cuda.synchronize()
    return calls, out


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("entry", ENTRIES)
def test_side_array_forms_are_bit_identical(ref, entry, form):
    calls, want = ref
    got = _outs(calls[entry](_int_forms(LENS)[form], _int_forms(NOISE_LENS)[form], _float_forms(SNR)[form]))
    assert len(got) == len(want[entry]) > 0
    for i, (a, b) in enumerate(zip(got, want[entry])):
        assert a.dtype == b.dtype and a.shape == b.shape and a.device == b.device, (entry, i)
        assert torch.equal(a, b) or (torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(), b.nan_to_num())), \
            (entry, form, i, float((a.double() - b.double()).abs().max()))


def test_the_reference_call_sees_every_row(ref):
    """The int32 reference itself: row 1 (9001 samples) is not an empty utterance."""
    _, want = ref
    y = want["reconstruct"][0]
    assert float(y[1].abs().max()) > 0 and bool(torch.isfinite(y).all())


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("n", [B - 1, B + 1])
def test_wrong_row_count_raises(ref, entry, n):
    calls, _ = ref
    bad_i, bad_f = list(range(1000, 1000 + n)), [0.0] * n
    ln, nl, snr = _REF["lens"], _REF["nl"], _REF["snr"]
    args = {"lengths": (bad_i, nl, snr), "noise_lengths": (ln, bad_i, snr), "snr_db": (ln, nl, bad_f)}
    for which, a in args.items():
        if which != "lengths" and entry not in ("snr_factor", "forward_raw", "preprocess_pairs"):
            continue
        if which == "snr_db" and entry == "forward_raw":
            continue
        with pytest.raises(ValueError):
            calls[entry](*a)
    with pytest.raises(ValueError):
        calls[entry](torch.tensor([LENS], dtype=torch.int32, device="cuda"), nl, snr)     # [1, B]: not one value per row
