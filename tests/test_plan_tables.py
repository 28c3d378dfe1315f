"""Constant tables built by the product (lhotse_b200/plan.py) are bit-identical to the oracle's
and to the reference module parameters (stored golden data)."""
import math

import numpy as np
import pytest

from helpers import as_config, load_golden_reference_api
from lhotse_b200 import (B200Fbank, B200FbankConfig, B200LogSpectrogramConfig, B200Mfcc, B200MfccConfig,
                         B200Spectrogram, B200SpectrogramConfig, build_plan)
from lhotse_b200.plan import make_window
from oracle import kaldi_oracle as O

CASES = [
    dict(),
    dict(num_filters=40, sampling_rate=8000),
    dict(num_filters=23, low_freq=100.0, high_freq=7000.0),
    dict(round_to_power_of_two=False),
    dict(torchaudio_compatible_mel_scale=False, norm_filters=True, num_filters=40),
    dict(torchaudio_compatible_mel_scale=False, low_freq=0.0, high_freq=0.0),
    dict(sampling_rate=24000, frame_length=0.05),
    dict(sampling_rate=22050, round_to_power_of_two=False, torchaudio_compatible_mel_scale=False, num_filters=40),
    dict(sampling_rate=44100, num_filters=128),
]


@pytest.mark.parametrize("kw", CASES)
def test_mel_bank_equals_oracle(kw):
    plan = build_plan("fbank", B200FbankConfig(**kw))
    ocfg = O.OracleConfig(feature="fbank", **kw)
    L, S, N = O.layer_sizes(ocfg)
    assert (plan.L, plan.S, plan.N) == (L, S, N)
    ref = O.make_mel_bank(ocfg, N).numpy()
    assert plan.mel_bank.shape == ref.shape == (N // 2 + 1, ocfg.num_filters)
    assert np.array_equal(plan.mel_bank, ref)


@pytest.mark.parametrize("w", ["povey", "hanning", "hamming", "rectangular", "blackman"])
@pytest.mark.parametrize("L", [200, 400, 551, 1200])
def test_window_equals_oracle(w, L):
    assert np.array_equal(make_window(L, w), O.make_window(L, w).numpy())


def test_dct_lifter_equal_oracle():
    plan = build_plan("mfcc", B200MfccConfig())
    assert np.array_equal(plan.dct, O.make_dct(13, 23).numpy())
    assert np.array_equal(plan.lifter, O.make_lifter(13, 22).numpy())
    assert build_plan("mfcc", B200MfccConfig(cepstral_lifter=0)).lifter is None


def test_headline_bank_structure():
    # SURVEY.md §2b: 477 non-zeros, <=16 per filter, rows 1..243 for 16 kHz / N=512 / M=80
    fb = build_plan("fbank", B200FbankConfig()).mel_bank
    nz = fb != 0
    assert nz.sum() == 477 and nz.sum(axis=0).max() <= 16
    rows = np.where(nz.any(axis=1))[0]
    assert rows.min() == 1 and rows.max() == 243


def test_plan_dims_and_validation():
    assert build_plan("fbank", B200FbankConfig(use_energy=True)).feature_dim == 81
    assert build_plan("mfcc", B200MfccConfig()).feature_dim == 13
    assert build_plan("spectrogram", B200SpectrogramConfig()).feature_dim == 257
    assert build_plan("log-spectrogram", B200LogSpectrogramConfig(round_to_power_of_two=False)).feature_dim == 201
    assert B200Fbank(B200FbankConfig(num_mel_bins=40)).config.num_filters == 40
    with pytest.raises(ValueError):
        build_plan("fbank", B200FbankConfig(dither=-1.0))
    assert build_plan("fbank", B200FbankConfig(dither=1.0)).dither == 1.0
    with pytest.raises(ValueError):
        build_plan("fbank", B200FbankConfig(window_type="kaiser"))
    with pytest.raises(ValueError):
        build_plan("fbank", B200FbankConfig(sampling_rate=22050, round_to_power_of_two=False))  # odd N, torchaudio mel
    p = build_plan("fbank", B200FbankConfig())
    for n in (159, 16000, 16079, 16080, 160000):
        assert p.num_frames(n) == O.num_frames_api(n, 0.01, 16000)
    blob = p.tables_blob()
    q = build_plan("fbank", B200FbankConfig())
    q.window[:] = 0
    q.load_tables_blob(blob)
    assert np.array_equal(q.window, p.window) and np.array_equal(q.mel_bank, p.mel_bank)


def test_tables_equal_live_reference_and_foreign_configs():
    """Against the reference module parameters and config objects stored in tests/golden/golden_reference_api_v1.npz."""
    man, arr = load_golden_reference_api()
    assert len(man["fbank_configs"]) == 7 and all(man["fbank_configs"][i][k] == v for i, kw in enumerate(CASES[:7]) for k, v in kw.items())
    for i, d in enumerate(man["fbank_configs"]):
        plan = build_plan("fbank", as_config(d))  # the reference's own config fields are accepted
        assert np.array_equal(plan.mel_bank, arr[f"fbank{i}_mel_bank"])
        assert np.array_equal(plan.window, arr[f"fbank{i}_window"])
    plan = build_plan("mfcc", as_config(man["mfcc_config"]))
    assert np.array_equal(plan.dct, arr["mfcc_dct"]) and np.array_equal(plan.lifter, arr["mfcc_lifter"])
    # torchaudio / kaldifeat config families normalise onto the same plan
    fam = {k: as_config(v) for k, v in man["family_configs"].items()}
    p = build_plan("fbank", fam["TorchaudioFbankConfig"])
    assert (p.L, p.S, p.N, p.num_filters, p.preemph_coeff, p.energy_style) == (400, 160, 512, 80, 0.97, 1)
    p = build_plan("mfcc", fam["TorchaudioMfccConfig"])
    assert (p.num_filters, p.num_ceps) == (23, 13)
    p = build_plan("fbank", fam["KaldifeatFbankConfig"])
    assert (p.L, p.S, p.N, p.num_filters, p.snip_edges) == (400, 160, 512, 80, False)
    p = build_plan("mfcc", fam["KaldifeatMfccConfig"])
    assert (p.num_filters, p.num_ceps) == (23, 13) and math.isclose(p.lifter[1], 1 + 11 * math.sin(math.pi / 22), rel_tol=1e-6)


def test_compat_flag_and_foreign_config_conversion():
    from dataclasses import dataclass

    from lhotse_b200 import from_reference_config

    p = build_plan("fbank", B200FbankConfig(compat="torchaudio", window_type="blackman"))
    q = build_plan("fbank", B200FbankConfig(window_type="blackman"))
    assert p.energy_style == 1 and q.energy_style == 0
    assert not np.array_equal(p.window, q.window)  # 2*pi/(L-1) vs 2*pi/L (kaldi.py:104 vs layers.py:931)
    with pytest.raises(ValueError):
        build_plan("fbank", B200FbankConfig(compat="htk"))

    @dataclass
    class TorchaudioMfccConfig:  # stand-in with the reference's field names (lhotse/features/mfcc.py:9-39)
        dither: float = 0.0
        window_type: str = "povey"
        frame_length: float = 0.025
        frame_shift: float = 0.01
        remove_dc_offset: bool = True
        round_to_power_of_two: bool = True
        energy_floor: float = 1e-10
        min_duration: float = 0.0
        preemphasis_coefficient: float = 0.97
        raw_energy: bool = True
        low_freq: float = 20.0
        high_freq: float = -400.0
        num_mel_bins: int = 23
        use_energy: bool = False
        vtln_low: float = 100.0
        vtln_high: float = -500.0
        vtln_warp: float = 1.0
        cepstral_lifter: float = 22.0
        num_ceps: int = 13

    ext = from_reference_config(TorchaudioMfccConfig(use_energy=True), sampling_rate=8000)
    assert type(ext).__name__ == "B200Mfcc" and ext.config.compat == "torchaudio" and ext.config.sampling_rate == 8000
    assert ext.plan.energy_style == 1 and ext.plan.num_filters == 23 and ext.plan.use_energy
    assert ext.config.preemph_coeff == 0.97 and (ext.plan.L, ext.plan.S, ext.plan.N) == (200, 80, 256)
