"""Whisper log-mel front end (SURVEY.md §8f-4): `B200WhisperFbank` vs the reference's `WhisperFbank`
(lhotse/features/whisper_fbank.py).  CPU tier: oracle pinned to the golden vectors / the live reference, mel table pinned to
transformers' restatement of librosa, host-side contract.  GPU tier (`-m gpu`): parity through the C ABI."""
import json
import os
import pickle

import numpy as np
import pytest
import torch

from helpers import load_golden_reference_api
from lhotse_b200 import LOG_EPSILON, build_plan
from lhotse_b200.plan import PAD_CENTER, make_slaney_mel_bank
from oracle import whisper_oracle as W

HERE = os.path.dirname(os.path.abspath(__file__))


def _classes():
    """Resolved at call time: test_host_logic / test_next_rows reload `lhotse_b200.extractors` once the reference tree is
    importable, which replaces the class objects."""
    import lhotse_b200.extractors as ex

    return ex.B200WhisperFbank, ex.B200WhisperFbankConfig


def load_golden_whisper():
    g = np.load(os.path.join(HERE, "golden", "golden_whisper_v1.npz"))
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


GOLD = load_golden_whisper()
IDS = [f"{i}-{c['signal']}-{c['n']}-m{c['num_filters']}" for i, c, _, _ in GOLD]

# Tolerance.  Features are (log10(mel) + 4) / 4, so north_star's 1e-4 relative on the mel energies is 1.1e-5 absolute
# here; the fp32 reference itself sits up to 1.2e-5 from its own float64 evaluation (speech / sine cases), so the gate is
#   max|ours - truth64| <= max(ATOL, NOISE_X * max|ref32 - truth64|)
ATOL, NOISE_X = 2e-5, 3.0


def whisper_gate(got, ref32, truth64):
    got, ref32, truth64 = (np.asarray(a, dtype=np.float64) for a in (got, ref32, truth64))
    assert np.all(np.isfinite(got))
    err, noise = np.abs(got - truth64).max(), np.abs(ref32 - truth64).max()
    limit = max(ATOL, NOISE_X * noise)
    return err <= limit, f"max|ours-truth|={err:.3e} max|ref32-truth|={noise:.3e} limit={limit:.3e} max|ours-ref32|={np.abs(got - ref32).max():.3e}"


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("i,c,x,y", GOLD, ids=IDS)
def test_whisper_oracle_matches_golden(i, c, x, y):
    got = W.extract(x, c["num_filters"])
    assert got.dtype == np.float32 and got.shape == y.shape == (W.num_rows(c["n"]), c["num_filters"])
    if np.array_equal(got, y):
        return
    # another CPU / BLAS path may move last bits (seen: 1 ulp on the single-frame case)
    np.testing.assert_allclose(got, y, rtol=0, atol=2e-6)


def test_whisper_oracle_bit_identical_to_live_reference():
    """Against the reference's `WhisperFbank.extract` on the same seeded inputs, stored by
    tests/golden/make_golden_reference_api.py."""
    from golden.make_golden_reference_api import whisper_inputs

    man, arr = load_golden_reference_api()
    cases = list(whisper_inputs())
    assert [(c["num_filters"], c["n"]) for c in man["whisper"]] == [(M, n) for M, n, _ in cases]
    for j, (M, n, x) in enumerate(cases):
        want = arr[f"whisper{j}"]
        got = W.extract(x, M)
        assert got.shape == want.shape
        assert np.array_equal(got, want), (M, n, np.abs(got - want).max())
        assert np.array_equal(W.extract(x[None, :], M), want)  # (1, n) input


def test_mel_table_pinned_to_transformers():
    """librosa is absent: both restatements of librosa.filters.mel (product and oracle) are pinned bit-for-bit to
    transformers' implementation, which upstream tests against librosa."""
    tf = pytest.importorskip("transformers.audio_utils")
    for M in (80, 128, 40):
        want = tf.mel_filter_bank(201, M, 0.0, 8000.0, 16000, norm="slaney", mel_scale="slaney").astype(np.float32)  # (K, M)
        assert np.array_equal(make_slaney_mel_bank(16000, 400, M), want)
        assert np.array_equal(W.slaney_mel_filters(M).T, want)


def test_mel_table_known_answers():
    """Values of OpenAI Whisper's published `mel_filters.npz` (= librosa.filters.mel(sr=16000, n_fft=400, n_mels=80))
    that are recoverable in closed form: below 1 kHz the Slaney scale is linear, so the first filters are triangles of
    width 2 * (200/3 Hz) * (mel step) with peak 2 / width."""
    fb = make_slaney_mel_bank(16000, 400, 80)  # (201, 80)
    assert fb.shape == (201, 80) and fb.dtype == np.float32
    assert np.all(fb >= 0) and np.all(fb[0] == 0)  # DC bin is in no filter
    assert np.all(fb[200] == 0)  # the Nyquist bin sits on the last filter's upper corner
    step = (15.0 + np.log(8.0) / (np.log(6.4) / 27.0)) / 81.0 * (200.0 / 3)  # corner spacing in Hz below 1 kHz
    # step = 37.24 Hz: bin 1 = 40 Hz lies on the falling edge of filter 0 (corners 0, step, 2 step) -> 0.024863
    np.testing.assert_allclose(fb[1, 0], ((2 * step - 40.0) / step) * (2.0 / (2 * step)), rtol=1e-6)
    np.testing.assert_allclose(fb[1, 1], ((40.0 - step) / step) * (2.0 / (2 * step)), rtol=1e-5)  # rising edge of filter 1
    assert abs(float(fb.sum(axis=0)[0]) * 40.0 - 1.0) < 0.2  # ~unit area (Hz) up to sampling of the triangle


def test_whisper_plan_and_config_contract():
    B200WhisperFbank, B200WhisperFbankConfig = _classes()
    ext = B200WhisperFbank()
    assert ext.name == "b200-whisper-fbank" and ext.frame_shift == 0.01 and ext.feature_dim(16000) == 80
    p = ext.plan
    assert (p.L, p.S, p.N, p.K, p.num_filters, p.pad_mode) == (400, 160, 400, 201, 80, PAD_CENTER)
    assert not p.remove_dc_offset and p.preemph_coeff == 0.0 and p.mel_floor == pytest.approx(1e-10)
    assert np.array_equal(p.window, torch.hann_window(400).numpy())  # periodic Hann, whisper_fbank.py:116
    for n, rows in ((16000, 100), (16079, 100), (16080, 101), (201, 1), (160000, 1000)):
        assert p.num_frames(n) == rows == W.num_rows(n)
    # config round trip: the reference's own keys (num_filters, device) + kernel
    d = ext.to_dict()
    assert d == {"num_filters": 80, "device": "cuda", "kernel": "auto", "feature_type": "b200-whisper-fbank"}
    again = type(ext).from_dict(dict(d))
    # (compare by name: other test modules re-import the package once the reference tree is on sys.path)
    assert type(again).__name__ == "B200WhisperFbank" and again.config.to_dict() == ext.config.to_dict()
    assert pickle.loads(pickle.dumps(ext)).config == ext.config
    assert build_plan("whisper-fbank", B200WhisperFbankConfig(num_filters=128)).mel_bank.shape == (201, 128)
    with pytest.raises(AssertionError):
        ext.extract(np.zeros(8000, dtype=np.float32), 8000)  # whisper_fbank.py:141-146
    with pytest.raises(ValueError):
        ext.extract(np.zeros((2, 8000), dtype=np.float32), 16000)  # :54-56 single channel only
    with pytest.raises(NotImplementedError):
        ext.online_inference(torch.zeros(1, 1600))


def test_whisper_registry_alias():
    import lhotse_b200
    from lhotse_b200.base import _REGISTRY, get_extractor_type

    saved = dict(_REGISTRY)
    try:
        lhotse_b200.install_as_default()
        assert get_extractor_type("whisper-fbank").__name__ == "B200WhisperFbank"
    finally:
        _REGISTRY.clear()
        _REGISTRY.update(saved)


# ------------------------------------------------------------------------------------------------ GPU tier
def make(num_filters=80, kernel="auto"):
    B200WhisperFbank, B200WhisperFbankConfig = _classes()
    return B200WhisperFbank(B200WhisperFbankConfig(num_filters=num_filters, kernel=kernel))


@pytest.mark.gpu
@pytest.mark.parametrize("i,c,x,y", GOLD, ids=IDS)
def test_gpu_whisper_golden(i, c, x, y):
    truth = W.extract(x, c["num_filters"], dtype=torch.float64)
    assert make(c["num_filters"]).engine.kernel == "fast"  # AUTO = the N = 400 prime-factor kernel
    for k in ("fast", "generic"):
        got = make(c["num_filters"], k).extract(x, 16000)
        assert got.dtype == np.float32 and got.shape == y.shape, (k, got.shape)  # row counts: bit-exact
        ok, msg = whisper_gate(got, y, truth)
        assert ok, f"kernel={k}: {msg}"
        if c["n"] % 160 >= 80:  # one more row than the stft has frames: a zero row (whisper_fbank.py:73-80)
            assert np.all(got[-1] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["fast", "generic"])
def test_gpu_whisper_ragged_batch(kernel):
    rs = np.random.RandomState(7)
    lens = [201, 640, 16000, 16079, 16080, 23456, 100000, 4000, 31999]
    xs = [((0.3 if i % 2 else 0.01) * rs.randn(n)).astype(np.float32) for i, n in enumerate(lens)]
    ext = make(kernel=kernel)
    batch = ext.extract_batch(xs, 16000)
    assert isinstance(batch, list) and len(batch) == len(xs)
    for x, got in zip(xs, batch):
        ref = W.extract(x)
        ok, msg = whisper_gate(got, ref, W.extract(x, dtype=torch.float64))
        assert got.shape == ref.shape and ok, msg
        assert np.array_equal(got, ext.extract(x, 16000))  # every cut is normalised by its own maximum
    # device-resident route (torch tensors in, CUDA tensors out) == host route, bit for bit
    tb = ext.extract_batch([torch.from_numpy(x) for x in xs], 16000)
    for a, b in zip(batch, tb):
        assert b.is_cuda and np.array_equal(a, b.cpu().numpy())
    # (1, n) input, tensor in -> tensor out
    one = ext.extract(torch.from_numpy(xs[2])[None, :], 16000)
    assert isinstance(one, torch.Tensor) and np.array_equal(one.cpu().numpy(), batch[2])
    # padded collation in the same launch pair: LOG_EPSILON rows past every cut's own rows
    padded, feat_lens = ext.extract_batch_padded([torch.from_numpy(x) for x in xs], 16000)
    assert padded.shape == (len(xs), max(W.num_rows(n) for n in lens), 80)
    pc = padded.cpu().numpy()
    for i, got in enumerate(batch):
        T = int(feat_lens[i])
        assert T == got.shape[0] and np.array_equal(pc[i, :T], got)
        assert np.all(pc[i, T:] == np.float32(LOG_EPSILON))
    # equal-length cuts stack to (B, T, F)
    same = ext.extract_batch(np.stack([xs[2], xs[2][::-1].copy()]), 16000)
    assert same.shape == (2, 100, 80) and np.array_equal(same[0], batch[2])


@pytest.mark.gpu
def test_gpu_whisper_int16_short_and_errors():
    rs = np.random.RandomState(8)
    pcm = np.clip(rs.randn(24000) * 3000, -32768, 32767).astype(np.int16)
    ext = make()
    a = ext.extract(pcm, 16000)
    b = ext.extract(pcm.astype(np.float32) / 32768.0, 16000)
    assert np.array_equal(a, b)  # int16 staging converts as x / 32768 on load
    for n in (1, 80, 200):  # torch's reflect padding needs more than n_fft / 2 samples: the reference raises too
        with pytest.raises(ValueError):
            ext.extract(np.zeros(n, dtype=np.float32), 16000)
    z = ext.extract(np.zeros(8000, dtype=np.float32), 16000)
    assert z.shape == (50, 80) and np.all(z == np.float32(-1.5))  # silence: log10(1e-10) = -10 -> (-10 + 4) / 4


@pytest.mark.gpu
def test_gpu_whisper_properties_at_baseline_size():
    """Size-independent properties on 256 x 10 s cuts (BASELINE-sized batch)."""
    g = torch.Generator(device="cuda").manual_seed(0)
    B, n = 256, 160000
    x = 0.1 * torch.randn(B, n, device="cuda", generator=g)
    ext = make()
    y = ext.extract_batch(x, 16000)
    assert y.shape == (B, 1000, 80) and bool(torch.isfinite(y).all())
    assert torch.equal(y, ext.extract_batch(x, 16000))  # deterministic (the max is order-independent)
    perm = torch.randperm(B, device="cuda", generator=g)
    assert torch.equal(ext.extract_batch(x[perm].contiguous(), 16000), y[perm])  # cuts are independent
    # gain: every mel energy scales by a^2 and so does the maximum, hence (log10 + 4) / 4 moves by log10(a) / 2
    # uniformly (white noise stays far above the 1e-10 floor and inside the max - 8 window)
    y4 = ext.extract_batch(4.0 * x, 16000)
    assert float((y4 - y - 0.5 * np.log10(4.0)).abs().max()) < 5e-6
    # per-cut normalisation: the clamp value of a cut is its own maximum - 8
    assert float(y.amax(dim=(1, 2)).min()) > 0.0 and float((y.amin(dim=(1, 2)) - (y.amax(dim=(1, 2)) - 2.0)).min()) >= -1e-6
    # spot parity with the oracle on four cuts
    for i in (0, 17, 128, 255):
        xi = x[i].cpu().numpy()
        ok, msg = whisper_gate(y[i].cpu().numpy(), W.extract(xi), W.extract(xi, dtype=torch.float64))
        assert ok, msg
