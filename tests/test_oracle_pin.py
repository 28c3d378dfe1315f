"""Pins the oracle against the committed golden vectors produced by the REAL reference
(tests/golden/make_golden.py, make_golden_reference_api.py): within the parity gate, and bit for bit."""
import hashlib

import numpy as np
import pytest
import torch

from helpers import gate, load_golden, load_golden_reference_api, oracle_cfg
from oracle import kaldi_oracle as O

GOLD = load_golden()


@pytest.mark.parametrize("i,c,x,y", GOLD, ids=[f"{i}-{c['feature']}-{c['kind']}-{c['n']}" for i, c, _, _ in GOLD])
def test_oracle_matches_golden(i, c, x, y):
    cfg = oracle_cfg(c["feature"], c["cfg"])
    got = O.extract(x, cfg)
    assert got.shape == tuple(c["shape"]) == y.shape and got.dtype == np.float32
    if np.array_equal(got, y):
        return  # bit-identical (same CPU / BLAS path as the generator)
    truth = O.extract(x, cfg, dtype=torch.float64)
    ok, msg = gate(got, y, truth, c["feature"], c["cfg"].get("use_energy", False), c["cfg"].get("use_fft_mag", False))
    assert ok, msg
    # different BLAS kernels (other CPU, other thread count) may move the last bits only
    np.testing.assert_allclose(got, y, rtol=1e-4, atol=1e-3 if c["feature"] == "mfcc" else 1e-4)


def test_frame_count_contract():
    # utils.py:424-434 and layers.py:753 agree for the standard geometry
    for n in list(range(15995, 16006)) + [159, 160, 239, 240, 16079, 16080, 160000]:
        assert O.num_frames_api(n, 0.01, 16000) == O.num_frames_layer(n, 400, 160, False)
    assert O.num_frames_layer(160000, 400, 160, False) == 1000
    assert O.num_frames_layer(16079, 400, 160, False) == 100
    assert O.num_frames_layer(16080, 400, 160, False) == 101
    assert O.num_frames_layer(159, 400, 160, False) == 1
    # test/known_issues/test_cut_consistency.py:77-105: 24 kHz, 50 ms window, 4.7 s -> 470 frames
    assert O.num_frames_layer(int(4.7 * 24000), 1200, 240, False) == 470
    with pytest.raises(ValueError):
        O.frame_index_matrix(100, 400, 160, False)  # too short for one reflection
    with pytest.raises(ValueError):
        O.frame_index_matrix(10, 400, 160, False)  # no frames


def test_reflect_indices_match_padding_semantics():
    # closed form == flip/cat construction of layers.py:753-766, exhaustively for small n
    for n in (159, 200, 399, 400, 1000, 1037):
        L, S = 400, 160
        idx = O.frame_index_matrix(n, L, S, False)
        T = idx.shape[0]
        left = (L - S) // 2
        right = (T - 1) * S + L - n - left
        base = np.arange(n)
        padded = np.concatenate((base[:left][::-1], base, base[n - right:][::-1] if right > 0 else base[:0]))
        want = np.stack([padded[t * S: t * S + L] for t in range(T)])
        assert np.array_equal(idx, want)


def test_oracle_bit_identical_to_live_reference():
    """Every golden input, bit for bit against the reference's own `Fbank / Mfcc / Spectrogram / LogSpectrogram.extract`:
    the SHA-256 of each reference output is stored in golden_reference_api_v1.npz (make_golden_reference_api.py).
    Oracle and reference run the same torch ops, but a CPU whose kernels order a sum differently moves the last bit of
    both (measured: 1 ulp, across CPUs and torch thread counts): there the oracle must stay within 2 ulp of the
    reference's stored output."""
    want = load_golden_reference_api()[0]["kaldi_sha256"]
    assert len(want) == len(GOLD)
    for (i, c, x, ref), h in zip(GOLD, want):
        got = O.extract(x, oracle_cfg(c["feature"], c["cfg"]))
        if hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() != h:
            np.testing.assert_array_max_ulp(got, ref, maxulp=2)


def test_strided_view_equals_closed_form_gather():
    rs = np.random.RandomState(0)
    for n, L, S, snip in ((159, 400, 160, False), (1000, 400, 160, False), (16080, 400, 160, False),
                          (5000, 200, 80, False), (3000, 400, 160, True), (11025, 551, 220, False)):
        x = torch.from_numpy(rs.randn(n).astype(np.float32))
        a = O._frames_view(x, L, S, snip)
        b = x[torch.from_numpy(O.frame_index_matrix(n, L, S, snip))]
        assert torch.equal(a, b)


from helpers import load_golden_stream  # noqa: E402

STREAM = load_golden_stream()


@pytest.mark.parametrize("i,m,x,y,r", STREAM, ids=[f"{i}-{m['feature']}" for i, m, _, _, _ in STREAM])
def test_oracle_streaming_matches_golden(i, m, x, y, r):
    """`online_inference` chunk by chunk against the reference's own streaming runs (layers.py:199-224, :326-333,
    :775-857): frame counts per call and the final remainder exactly, values like the offline goldens."""
    cfg = oracle_cfg(m["feature"], m["cfg"])
    rem, feats, counts = None, [], []
    for a, b in zip(m["bounds"][:-1], m["bounds"][1:]):
        f, rem = O.online_inference(x[a:b], cfg, context=rem)
        feats.append(f)
        counts.append(f.shape[0])
    assert counts == m["counts"]
    assert np.array_equal(rem, r)
    got = np.concatenate(feats, axis=0)
    assert got.shape == y.shape
    if not np.array_equal(got, y):
        np.testing.assert_allclose(got, y, rtol=1e-4, atol=1e-3 if m["feature"] in ("mfcc", "spectrogram") else 1e-4)
    S = O.layer_sizes(cfg)[1]
    if not m["cfg"].get("snip_edges", False) and m["n"] % S == 0:
        # test_kaldi_layers.py:199-235: streaming + one flipped tail chunk reproduces the offline frames
        tail, rem2 = O.online_inference(x[-S:][::-1].copy(), cfg, context=rem)
        online = np.concatenate([got, tail], axis=0)
        offline = O.extract(x, cfg)
        assert online.shape == offline.shape
        np.testing.assert_allclose(online, offline, rtol=1e-4, atol=1e-3 if m["feature"] in ("mfcc", "spectrogram") else 1e-4)
