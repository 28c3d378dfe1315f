"""LibrosaFbank drop-in (`B200LibrosaFbank`, SURVEY.md §8f-4) vs the reference's `LibrosaFbank`
(lhotse/features/librosa_fbank.py).  librosa itself is absent: see oracle/librosa_oracle.py for what pins parity (the
reference's own code run on a transformers-based stand-in + an independent restatement that agrees with it bit for bit on
11 of the 13 golden cases)."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import load_golden_reference_api
from lhotse_b200 import build_plan
from lhotse_b200.plan import PAD_CENTER, make_periodic_window, make_slaney_mel_bank
from oracle import librosa_oracle as LO

HERE = os.path.dirname(os.path.abspath(__file__))


def _classes():
    import lhotse_b200.extractors as ex

    return ex.B200LibrosaFbank, ex.B200LibrosaFbankConfig


def load_golden_librosa():
    g = np.load(os.path.join(HERE, "golden", "golden_librosa_v1.npz"))
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


GOLD = load_golden_librosa()
IDS = [f"{i}-{c['signal']}-{c['n']}-N{c['cfg']['fft_size']}" for i, c, _, _ in GOLD]


def librosa_gate(got, truth64, cfg):
    """Linear (mel-magnitude) domain: |ours - truth| <= 1e-4 * truth + 4e-6 * wsum[m] * (frame's peak line), where the
    peak line is estimated from the truth itself (mel[m] <= wsum[m] * max|X|).  north_star's 1e-4 relative, plus the
    amplitude floor every fp32 FFT has relative to the frame's largest line (the reference transforms in float64)."""
    fmin = 0.0 if cfg["fmin"] is None else cfg["fmin"]
    fmax = cfg["sampling_rate"] / 2 if cfg["fmax"] is None else cfg["fmax"]
    wsum = make_slaney_mel_bank(cfg["sampling_rate"], cfg["fft_size"], cfg["num_mel_bins"], fmin, fmax).astype(np.float64).sum(axis=0)
    lin_t, lin_g = 10.0 ** np.asarray(truth64, np.float64), 10.0 ** np.asarray(got, np.float64)
    peak = (lin_t / np.maximum(wsum, 1e-30)).max(axis=1, keepdims=True)
    tol = 1e-4 * lin_t + 4e-6 * wsum[None, :] * peak + 1e-14
    r = np.abs(lin_g - lin_t) / tol
    return bool(r.max() <= 1.0), f"max err/tol {r.max():.3f}, max|d log10| {np.abs(np.asarray(got, np.float64) - truth64).max():.3e}"


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("i,c,x,y", GOLD, ids=IDS)
def test_librosa_oracle_matches_golden(i, c, x, y):
    got = LO.extract(x, **c["cfg"])
    assert got.dtype == np.float32 and got.shape == y.shape == (LO.num_rows(c["n"], c["cfg"]["hop_size"]), c["cfg"]["num_mel_bins"])
    np.testing.assert_allclose(got, y, rtol=0, atol=2e-5)
    ok, msg = librosa_gate(y, LO.extract(x, float64=True, **c["cfg"]), c["cfg"])  # the gate accepts the reference itself
    assert ok, msg


def test_librosa_oracle_against_live_reference_on_the_standin():
    """Against the reference's `LibrosaFbank.extract` (run on the stand-in) on the same seeded inputs, stored by
    tests/golden/make_golden_reference_api.py."""
    from golden.make_golden_reference_api import librosa_inputs

    man, arr = load_golden_reference_api()
    cfgs = man["librosa_configs"]
    cases = list(librosa_inputs(cfgs))
    assert [(c["config"], c["n"]) for c in man["librosa"]] == [(k, n) for k, n, _ in cases] and len(cases) == 6
    for j, (k, n, x) in enumerate(cases):
        want = arr[f"librosa{j}"]
        got = LO.extract(x, **cfgs[k])
        assert got.shape == want.shape
        np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)


def test_librosa_tables_pinned():
    tf = pytest.importorskip("transformers.audio_utils")
    sig = pytest.importorskip("scipy.signal")
    for sr, N, M, fmin, fmax in ((22050, 1024, 80, 80.0, 7600.0), (16000, 512, 40, 0.0, 8000.0), (24000, 2048, 100, 50.0, 12000.0)):
        want = tf.mel_filter_bank(N // 2 + 1, M, fmin, fmax, sr, norm="slaney", mel_scale="slaney").astype(np.float32)
        assert np.array_equal(make_slaney_mel_bank(sr, N, M, fmin, fmax), want)          # product table
        assert np.array_equal(LO.slaney_mel_filters(sr, N, M, fmin, fmax).T, want)        # oracle table
    for name in ("hann", "hamming", "blackman", "boxcar"):
        for L in (400, 1024, 1200):  # librosa: scipy.signal.get_window(name, L, fftbins=True)
            want = sig.get_window(name, L, fftbins=True)
            np.testing.assert_allclose(make_periodic_window(name, L), want.astype(np.float32), rtol=0, atol=6e-8)
            np.testing.assert_allclose(LO.periodic_window(name, L), want, rtol=0, atol=1e-15)


def test_librosa_plan_and_config_contract():
    B200LibrosaFbank, B200LibrosaFbankConfig = _classes()
    ext = B200LibrosaFbank()
    p = ext.plan
    assert ext.name == "b200-librosa-fbank" and ext.frame_shift == 256 / 22050 and ext.feature_dim(22050) == 80
    assert (p.L, p.S, p.N, p.K, p.num_filters, p.pad_mode, p.use_fft_mag) == (1024, 256, 1024, 513, 80, PAD_CENTER, True)
    assert not p.remove_dc_offset and p.preemph_coeff == 0.0 and p.mel_floor == pytest.approx(1e-10)
    for n in (22050, 22050 + 127, 22050 + 128, 513):
        assert p.num_frames(n) == LO.num_rows(n, 256)
    d = ext.to_dict()
    assert d == {"sampling_rate": 22050, "fft_size": 1024, "hop_size": 256, "win_length": None, "window": "hann",
                 "num_mel_bins": 80, "fmin": 80, "fmax": 7600, "device": "cuda", "kernel": "auto", "feature_type": "b200-librosa-fbank"}
    assert type(ext).from_dict(dict(d)).config.to_dict() == ext.config.to_dict()
    q = build_plan("librosa-fbank", B200LibrosaFbankConfig(win_length=800))  # window centred in the frame (pad_center)
    assert np.all(q.window[:112] == 0) and np.all(q.window[912:] == 0) and q.window[112 + 400] == pytest.approx(1.0)
    # fmin / fmax = None mean 0 Hz / Nyquist (librosa_fbank.py:119-120), not "use the default"
    for i, c, _, _ in GOLD:
        cfg = c["cfg"]
        pl = build_plan("librosa-fbank", B200LibrosaFbankConfig(**cfg))
        fmin = 0.0 if cfg["fmin"] is None else cfg["fmin"]
        fmax = cfg["sampling_rate"] / 2 if cfg["fmax"] is None else cfg["fmax"]
        assert np.array_equal(pl.mel_bank, LO.slaney_mel_filters(cfg["sampling_rate"], cfg["fft_size"], cfg["num_mel_bins"], fmin, fmax).T)
    with pytest.raises(ValueError):
        B200LibrosaFbank(B200LibrosaFbankConfig(window="kaiser"))
    with pytest.raises(AssertionError):
        ext.extract(np.zeros(8000, dtype=np.float32), 16000)
    with pytest.raises(AssertionError):
        ext.extract(np.zeros((2, 8000), dtype=np.float32), 22050)  # librosa_fbank.py:101-105
    import lhotse_b200
    from lhotse_b200.base import _REGISTRY, get_extractor_type

    saved = dict(_REGISTRY)
    try:
        lhotse_b200.install_as_default()
        assert get_extractor_type("librosa-fbank").__name__ == "B200LibrosaFbank"
    finally:
        _REGISTRY.clear()
        _REGISTRY.update(saved)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("i,c,x,y", GOLD, ids=IDS)
def test_gpu_librosa_golden(i, c, x, y):
    B200LibrosaFbank, B200LibrosaFbankConfig = _classes()
    cfg = c["cfg"]
    truth = LO.extract(x, float64=True, **cfg)
    auto = B200LibrosaFbank(B200LibrosaFbankConfig(**cfg))
    assert auto.engine.kernel == ("fast" if cfg["fft_size"] in (256, 400, 512, 1024, 2048) else "generic")
    for k in dict.fromkeys((auto.engine.kernel, "generic")):
        got = B200LibrosaFbank(B200LibrosaFbankConfig(kernel=k, **cfg)).extract(x, cfg["sampling_rate"])
        assert got.dtype == np.float32 and got.shape == y.shape, (k, got.shape)  # row counts: bit-exact
        ok, msg = librosa_gate(got, truth, cfg)
        assert ok, f"kernel={k}: {msg}"
        if c["signal"] == "zeros":
            assert np.all(got == np.float32(-10.0))


@pytest.mark.gpu
def test_gpu_librosa_ragged_batch_and_padded():
    B200LibrosaFbank, _ = _classes()
    rs = np.random.RandomState(31)
    lens = [513, 4000, 22050, 22050 + 127, 22050 + 128, 66150, 1025]
    xs = [(0.1 * rs.randn(n)).astype(np.float32) for n in lens]
    ext = B200LibrosaFbank()
    batch = ext.extract_batch(xs, 22050)
    for x, got in zip(xs, batch):
        assert got.shape == (LO.num_rows(len(x), 256), 80)
        ok, msg = librosa_gate(got, LO.extract(x, float64=True), ext.config.to_dict())
        assert ok, msg
        assert np.array_equal(got, ext.extract(x, 22050))
    tb = ext.extract_batch([torch.from_numpy(x) for x in xs], 22050)
    assert all(t.is_cuda and np.array_equal(t.cpu().numpy(), b) for t, b in zip(tb, batch))
    padded, flens = ext.extract_batch_padded([torch.from_numpy(x) for x in xs], 22050, padding_value=-23.0)
    pc = padded.cpu().numpy()
    for i, got in enumerate(batch):
        assert int(flens[i]) == got.shape[0] and np.array_equal(pc[i, : got.shape[0]], got) and np.all(pc[i, got.shape[0]:] == -23.0)
    with pytest.raises(ValueError):
        ext.extract(np.zeros(512, dtype=np.float32), 22050)  # reflect padding needs more than fft_size / 2 samples
    # gain: magnitudes scale by a, so log10 features move by log10(a) everywhere above the floor
    y1, y3 = ext.extract(xs[2], 22050), ext.extract(3.0 * xs[2], 22050)
    assert np.abs(y3 - y1 - np.log10(3.0)).max() < 2e-5
