"""Registry-level drop-ins for the torchaudio and kaldifeat config families (lhotse_b200/families.py; SURVEY.md §8a row a2).
CPU tier: config surfaces field-for-field against the reference's dataclasses, YAML/dict round trips, registry aliases,
container rules through the oracle-backed fake engine.  GPU tier: torchaudio golden vectors through the adapter classes,
kaldifeat adapters against B200Fbank / B200Mfcc (the reference anchors kaldifeat on Fbank the same way,
test/features/test_kaldifeat_features.py:103-116)."""
import dataclasses
import json
import os
import pickle

import numpy as np
import pytest
import torch

from helpers import attach_oracle_engine, load_golden_reference_api

HERE = os.path.dirname(os.path.abspath(__file__))


def _lb():
    """Resolved at call time (other test modules reload the package once the reference is importable)."""
    import lhotse_b200.extractors as ex
    import lhotse_b200.families as fam

    return ex, fam


def _ta_golden():
    g = np.load(os.path.join(HERE, "golden", "golden_torchaudio_v1.npz"))
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


TA_GOLD = _ta_golden()


def _ta_spec_golden():
    g = np.load(os.path.join(HERE, "golden", "golden_torchaudio_spec_v1.npz"))
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


TA_SPEC_GOLD = _ta_spec_golden()


# ------------------------------------------------------------------------------------------------ CPU tier
def test_config_surfaces_match_the_reference_field_for_field():
    """Against the reference's config dataclasses as stored in tests/golden/golden_reference_api_v1.npz: field names,
    default values and `to_dict()` output."""
    man, _ = load_golden_reference_api()
    ref = man["config_surfaces"]
    _, fam = _lb()
    pairs = [("TorchaudioFbankConfig", fam.B200TorchaudioFbankConfig), ("TorchaudioMfccConfig", fam.B200TorchaudioMfccConfig),
             ("TorchaudioSpectrogramConfig", fam.B200TorchaudioSpectrogramConfig),
             ("KaldifeatFrameOptions", fam.B200KaldifeatFrameOptions), ("KaldifeatMelOptions", fam.B200KaldifeatMelOptions),
             ("KaldifeatFbankConfig", fam.B200KaldifeatFbankConfig), ("KaldifeatMfccConfig", fam.B200KaldifeatMfccConfig)]
    assert sorted(ref) == sorted(name for name, _ in pairs)
    for ref_name, our_cls in pairs:
        ours = {f.name: f for f in dataclasses.fields(our_cls)}
        ref_fields, ref_defaults = ref[ref_name]["fields"], ref[ref_name]["defaults"]
        our_inst = our_cls()
        for name in ref_fields:
            assert name in ours, (ref_name, name)
            if name in ("device", "frame_opts", "mel_opts"):
                continue
            assert json.loads(json.dumps(getattr(our_inst, name))) == ref_defaults[name], (ref_name, name)
        extra = set(ours) - set(ref_fields)
        assert extra <= {"device", "kernel"}, (our_cls.__name__, extra)
        # a dict written by the reference loads into ours
        loaded = our_cls.from_dict(dict(ref[ref_name]["to_dict"]))
        assert dataclasses.asdict(loaded) == dataclasses.asdict(dataclasses.replace(our_inst, **(
            {"device": "cpu"} if "device" in ref_fields else {})))
    assert fam.B200KaldifeatFrameOptions().to_dict() == ref["KaldifeatFrameOptions"]["to_dict"]  # ms / samp_freq spelling


def test_family_registry_names_and_round_trips(tmp_path):
    import lhotse_b200
    from lhotse_b200.base import _REGISTRY, FeatureExtractor, get_extractor_type

    _, fam = _lb()
    saved = dict(_REGISTRY)
    try:
        lhotse_b200.install_as_default()
        for name, cls in (("fbank", "B200TorchaudioFbank"), ("mfcc", "B200TorchaudioMfcc"), ("spectrogram", "B200TorchaudioSpectrogram"),
                          ("kaldifeat-fbank", "B200KaldifeatFbank"), ("kaldifeat-mfcc", "B200KaldifeatMfcc")):
            assert get_extractor_type(name).__name__ == cls
        # a manifest / YAML produced by the reference ("feature_type: kaldifeat-fbank", device: cpu, ms spellings)
        d = {"feature_type": "kaldifeat-fbank", "frame_opts": {"samp_freq": 8000.0, "frame_shift_ms": 10.0, "frame_length_ms": 25.0},
             "mel_opts": {"num_bins": 40}, "use_energy": True, "device": "cuda"}
        ext = FeatureExtractor.from_dict(dict(d))
        assert type(ext).__name__ == "B200KaldifeatFbank" and ext.config.frame_opts.sampling_rate == 8000
        assert ext.feature_dim(8000) == 40 and ext.frame_shift == 0.01
        plan = ext._inner(8000).plan
        assert (plan.L, plan.S, plan.N, plan.num_filters, plan.use_energy, plan.energy_style) == (200, 80, 256, 40, True, 1)
    finally:
        _REGISTRY.clear()
        _REGISTRY.update(saved)
    sp = fam.B200TorchaudioSpectrogram()
    plan = sp._inner(16000).plan  # kaldi.py spectrogram: log(max(P, eps32)), bin 0 <- Kaldi log-energy
    assert (plan.feature, plan.use_energy, plan.energy_style, sp.feature_dim(16000), sp.feature_dim(8000)) == ("log-spectrogram", True, 1, 257, 129)
    assert plan.log_spec_eps == -float(np.finfo(np.float32).eps)
    for cls in (fam.B200TorchaudioFbank, fam.B200TorchaudioMfcc, fam.B200TorchaudioSpectrogram, fam.B200KaldifeatFbank, fam.B200KaldifeatMfcc):
        ext = cls()
        path = tmp_path / f"{cls.name}.yml"
        ext.to_yaml(path)
        again = FeatureExtractor.from_yaml(path)
        assert type(again).__name__ == cls.__name__ and again.config.to_dict() == ext.config.to_dict()
        assert pickle.loads(pickle.dumps(ext)).config.to_dict() == ext.config.to_dict()
    for bad in (dict(vtln_warp=1.2, vtln_low=10.0), dict(min_duration=0.5), dict(window_type="kaiser")):  # vtln_low below low_freq
        with pytest.raises(ValueError):
            fam.B200TorchaudioFbank(fam.B200TorchaudioFbankConfig(**bad))
    assert fam.B200KaldifeatFbank(fam.B200KaldifeatFbankConfig(htk_compat=True, use_energy=True))._inner(16000).plan.energy_last
    with pytest.raises(ValueError):
        fam.B200KaldifeatFbank(fam.B200KaldifeatFbankConfig(use_log_fbank=False))


def test_vtln_mel_bank_bit_equal_to_torchaudio():
    """`vtln_warp != 1` (TorchaudioFbankConfig.vtln_*, lhotse/features/fbank.py:30-32 -> torchaudio.compliance.kaldi.fbank): the
    warped filter bank is the table torchaudio builds, bit for bit, and the plan carries it."""
    K = pytest.importorskip("torchaudio.compliance.kaldi")
    import lhotse_b200.families as fam
    from lhotse_b200.plan import build_plan, make_mel_bank

    for M, N, sr, lo, hi, vlo, vhi, warp in ((80, 512, 16000, 20.0, -400.0, 100.0, -500.0, 1.1), (40, 512, 16000, 20.0, -400.0, 100.0, -500.0, 0.9),
                                             (23, 256, 8000, 20.0, 3700.0, 200.0, -800.0, 1.15), (80, 1024, 24000, 0.0, 0.0, 60.0, 11000.0, 0.8),
                                             (128, 2048, 44100, 20.0, -400.0, 100.0, -500.0, 1.25)):
        want, _ = K.get_mel_banks(M, N, float(sr), lo, hi, vlo, vhi, warp)
        want = torch.nn.functional.pad(want, (0, 1)).T.numpy()
        got = make_mel_bank(M, N, sr, lo, hi, vtln_low=vlo, vtln_high=vhi, vtln_warp=warp)
        assert got.dtype == np.float32 and got.shape == want.shape == (N // 2 + 1, M)
        assert np.array_equal(got, want), (M, N, warp, float(np.abs(got - want).max()))
        assert not np.array_equal(got, make_mel_bank(M, N, sr, lo, hi))  # the warp does move the filters
    plan = build_plan("fbank", fam.B200TorchaudioFbankConfig(vtln_warp=1.1))
    want, _ = K.get_mel_banks(80, 512, 16000.0, 20.0, -400.0, 100.0, -500.0, 1.1)
    assert np.array_equal(np.asarray(plan.mel_bank), torch.nn.functional.pad(want, (0, 1)).T.numpy())
    inner = fam.B200TorchaudioMfcc(fam.B200TorchaudioMfccConfig(vtln_warp=1.15, vtln_low=200.0, vtln_high=-800.0, device="cpu"))._inner(16000)
    assert (inner.config.vtln_warp, inner.config.vtln_low, inner.config.vtln_high) == (1.15, 200.0, -800.0)


def test_family_container_rules_on_the_oracle_engine():
    """Host logic only (no GPU): the adapters' container / dtype rules, with the CPU oracle standing in for the engine."""
    _, fam = _lb()
    i, c, x, y = TA_GOLD[0]  # torchaudio fbank defaults: no energy term, so the lhotse-convention oracle applies
    ta = fam.B200TorchaudioFbank()
    attach_oracle_engine(ta._inner(16000))
    got = ta.extract(x, 16000)
    assert isinstance(got, np.ndarray) and got.shape == y.shape
    np.testing.assert_allclose(got, y, rtol=1e-3, atol=5e-4)
    got_t = ta.extract(torch.from_numpy(x).unsqueeze(0), 16000)  # (1, n) tensor in -> numpy out (base.py:421-424)
    assert isinstance(got_t, np.ndarray) and np.array_equal(got_t, got)
    batch = ta.extract_batch([x, x[:8000]], 16000)
    assert isinstance(batch, list) and batch[0].shape == y.shape and batch[1].shape == (50, 80)
    assert ta._inner(8000) is not ta._inner(16000) and ta._inner(8000).plan.N == 256  # one handle per sampling rate

    kf = fam.B200KaldifeatFbank()
    attach_oracle_engine(kf._inner(16000))
    single = kf.extract(x, 16000)                      # 1-D array -> array
    assert isinstance(single, np.ndarray) and single.shape == y.shape
    as_list = kf.extract([x], 16000)                   # list of one -> list of one (kaldifeat.py:131-135)
    assert isinstance(as_list, list) and len(as_list) == 1 and np.array_equal(as_list[0], single)
    stacked = kf.extract(np.stack([x, x]), 16000)      # 2-D batch of equal lengths -> stacked (B, T, F)
    assert stacked.shape == (2,) + y.shape and np.array_equal(stacked[1], single)
    ragged = kf.extract([x, x[:4000]], 16000)
    assert isinstance(ragged, list) and [r.shape[0] for r in ragged] == [75, 25]
    trimmed = kf.extract_batch(torch.from_numpy(np.stack([x, x])), 16000, lengths=[12000, 4000])  # kaldifeat.py:84-86
    assert [t.shape[0] for t in trimmed] == [75, 25] and np.allclose(np.asarray(trimmed[1]), ragged[1])
    with pytest.raises(AssertionError):
        kf.extract(x, 8000)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("i,c,x,y", TA_GOLD, ids=[f"{i}-{c['feature']}" for i, c, _, _ in TA_GOLD])
def test_gpu_torchaudio_adapters_golden(i, c, x, y):
    """torchaudio.compliance.kaldi outputs (tests/golden/make_golden_torchaudio.py) through the registry-level adapters,
    built from the reference's own config dict; gate as in test/features/test_kaldi_features.py:116-122."""
    _, fam = _lb()
    cls = fam.B200TorchaudioMfcc if c["feature"] == "mfcc" else fam.B200TorchaudioFbank
    ext = cls(cls.config_type.from_dict(dict(c["cfg"])))
    got = ext.extract(x, 16000)
    assert isinstance(got, np.ndarray) and got.shape == y.shape
    np.testing.assert_allclose(got, y, rtol=1e-3, atol=5e-4)
    assert np.array_equal(ext.extract(torch.from_numpy(x), 16000), got)   # tensor in -> numpy out, same bits
    b = ext.extract_batch([torch.from_numpy(x), torch.from_numpy(x[:5000])], 16000)
    assert b[0].is_cuda and np.array_equal(b[0].cpu().numpy(), got) and b[1].shape[0] == (5000 + 80) // 160


def _htk_golden():
    import json

    g = np.load(os.path.join(HERE, "golden", "golden_kaldi_htk_v1.npz"))
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


HTK_GOLD = _htk_golden()


def test_htk_compat_plan_tables():
    """htk_compat (kaldifeat.py:158, :227) as table permutations: C0's DCT column and lifter slot move last, sqrt(2) rides on the
    lifter slot without use_energy; fbank only flags the energy column."""
    _, fam = _lb()
    base = fam.B200KaldifeatMfcc(fam.B200KaldifeatMfccConfig(device="cpu"))._inner(16000).plan
    htk = fam.B200KaldifeatMfcc(fam.B200KaldifeatMfccConfig(htk_compat=True, device="cpu"))._inner(16000).plan
    C = base.num_ceps
    assert np.array_equal(htk.dct[:, :-1], base.dct[:, 1:]) and np.array_equal(htk.dct[:, -1], base.dct[:, 0])
    assert np.array_equal(htk.lifter[:-1], base.lifter[1:]) and htk.lifter[-1] == np.float32(np.float32(1.0) * np.float32(np.sqrt(2.0)))
    assert htk.energy_last and htk.feature_dim == C
    e = fam.B200KaldifeatMfcc(fam.B200KaldifeatMfccConfig(htk_compat=True, use_energy=True, device="cpu"))._inner(16000).plan
    assert e.energy_last and e.lifter[-1] == np.float32(1.0)
    fb = fam.B200KaldifeatFbank(fam.B200KaldifeatFbankConfig(htk_compat=True, device="cpu"))._inner(16000).plan
    assert not fb.energy_last and fb.feature_dim == 80  # nothing to move without use_energy


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["generic", "fast"])
@pytest.mark.parametrize("i,c,x,y", HTK_GOLD, ids=[f"{i}-{c['feature']}" for i, c, _, _ in HTK_GOLD])
def test_gpu_kaldifeat_htk_compat_golden(kernel, i, c, x, y):
    """Kaldi's htk_compat layout through the kaldifeat adapters against torchaudio's Kaldi-compatible functions
    (tests/golden/make_golden_kaldi_htk.py): energy / C0 last, C0 * sqrt(2) without use_energy."""
    _, fam = _lb()
    k = c["cfg"]
    mel = fam.B200KaldifeatMelOptions(num_bins=k["num_bins"])
    if c["feature"] == "mfcc":
        ext = fam.B200KaldifeatMfcc(fam.B200KaldifeatMfccConfig(mel_opts=mel, num_ceps=k["num_ceps"], cepstral_lifter=k["cepstral_lifter"],
                                                                use_energy=k["use_energy"], htk_compat=True, kernel=kernel))
    else:
        ext = fam.B200KaldifeatFbank(fam.B200KaldifeatFbankConfig(mel_opts=mel, use_energy=k["use_energy"], htk_compat=True, kernel=kernel))
    got = ext.extract(x, 16000)
    assert got.shape == y.shape
    np.testing.assert_allclose(got, y, rtol=1e-3, atol=5e-4)
    plain = type(ext)(type(ext.config).from_dict({**ext.config.to_dict(), "htk_compat": False})).extract(x, 16000)
    if c["feature"] == "fbank" and k["use_energy"]:
        assert np.array_equal(got[:, :-1], plain[:, 1:]) and np.array_equal(got[:, -1], plain[:, 0])  # a pure column move
    elif c["feature"] == "fbank":
        assert np.array_equal(got, plain)


@pytest.mark.gpu
def test_gpu_kaldifeat_adapters_agree_with_fbank_and_mfcc():
    ex, fam = _lb()
    rs = np.random.RandomState(3)
    xs = [(0.1 * rs.randn(n)).astype(np.float32) for n in (16000, 4000, 23456)]
    kf, fb = fam.B200KaldifeatFbank(), ex.B200Fbank()
    got = kf.extract(xs, 16000)
    want = fb.extract_batch(xs, 16000)
    assert isinstance(got, list) and all(np.array_equal(a, b) for a, b in zip(got, want))  # same plan, same kernel
    assert np.array_equal(kf.extract(xs[0], 16000), want[0])
    tens = kf.extract([torch.from_numpy(x) for x in xs], 16000)
    assert all(t.is_cuda and np.array_equal(t.cpu().numpy(), w) for t, w in zip(tens, want))
    trimmed = kf.extract_batch(torch.from_numpy(np.stack([xs[0], xs[0]])), 16000, lengths=[16000, 4000])
    assert np.array_equal(trimmed[0].cpu().numpy(), want[0]) and trimmed[1].shape[0] == 25
    km, mf = fam.B200KaldifeatMfcc(), ex.B200Mfcc()
    np.testing.assert_allclose(km.extract(xs[2], 16000), mf.extract(xs[2], 16000), rtol=1e-3, atol=1e-3)  # decimal=3 upstream
    # Kaldi energy convention (C0 <- log-energy) vs the torchaudio golden of the same settings
    i, c, x, y = next(t for t in TA_GOLD if t[1]["feature"] == "mfcc" and t[1]["cfg"]["use_energy"])
    ke = fam.B200KaldifeatMfcc(fam.B200KaldifeatMfccConfig(use_energy=True))
    np.testing.assert_allclose(ke.extract(x, 16000), y, rtol=1e-3, atol=5e-4)
    # 8 kHz telephone geometry through the ms-spelled dict
    k8 = fam.B200KaldifeatFbank.config_type.from_dict({"frame_opts": {"samp_freq": 8000.0}, "mel_opts": {"num_bins": 40}})
    y8 = fam.B200KaldifeatFbank(k8).extract(xs[0][:8000], 8000)
    assert y8.shape == (100, 40) and np.isfinite(y8).all()


@pytest.mark.gpu
@pytest.mark.parametrize("i,c,x,y", TA_SPEC_GOLD, ids=[f"{i}-sr{c['sampling_rate']}" for i, c, _, _ in TA_SPEC_GOLD])
@pytest.mark.parametrize("kernel", ["auto", "generic"])
def test_gpu_torchaudio_spectrogram_adapter_golden(kernel, i, c, x, y):
    """`torchaudio.compliance.kaldi.spectrogram` (tests/golden/make_golden_torchaudio_spectrogram.py) through
    B200TorchaudioSpectrogram.  Bin 0 is a Kaldi log-energy (compared directly); the other bins are log(max(P, eps32)):
    compared as amplitudes, because an fp32 FFT carries an error ~1e-6 of the frame's largest line whatever the bin's own
    size (the rule of helpers.gate), and checked to sit on the same floor where the reference does."""
    _, fam = _lb()
    ext = fam.B200TorchaudioSpectrogram(fam.B200TorchaudioSpectrogramConfig.from_dict(dict(c["cfg"], kernel=kernel)))
    got = ext.extract(x, c["sampling_rate"])
    assert isinstance(got, np.ndarray) and got.shape == y.shape and np.isfinite(got).all()
    np.testing.assert_allclose(got[:, 0], y[:, 0], rtol=1e-4, atol=2e-4)
    floor = np.log(np.float32(np.finfo(np.float32).eps))
    assert got[:, 1:].min() >= floor - 1e-6
    silent = (y[:, 1:] <= floor + 1e-6).all(axis=1)   # frames of exact silence: every bin on the floor, in both
    np.testing.assert_allclose(got[silent, 1:], y[silent, 1:], rtol=0, atol=4e-6)  # logf(eps32): device vs host libm
    a_got, a_ref = np.exp(0.5 * got[:, 1:].astype(np.float64)), np.exp(0.5 * y[:, 1:].astype(np.float64))
    tol = 1e-4 * a_ref + 4e-6 * a_ref.max(axis=1, keepdims=True) + 1e-9
    assert (np.abs(a_got - a_ref) <= tol).all(), float((np.abs(a_got - a_ref) / tol).max())
