"""Features that every kernel implements in its own epilogue or launch code, run on every kernel.

The per-kernel oracle sweeps (test_gpu_parity.py) pin the arithmetic of each kernel on its default path.  Three features
are handled separately by each kernel and are checked here across the whole kernel table:
  A. the output affine (`Engine.set_output_affine`, the fused GlobalMVN) at every store site of every epilogue, padding
     rows included;
  B. the htk_compat layout (energy / C0 column last) through the kaldifeat adapters;
  C. the chunked host pipelines (`extract_host` / `extract_host_list`), whose launches are the only ones that start at a
     nonzero cut and tile (`batch_first`, `tile_base`) and that offset whisper-fbank's per-cut maximum scratch.
Every case asserts the kernel and FFT size it landed on, so that a plan silently served by another kernel fails instead
of passing untested."""
import math
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

from helpers import gate, oracle_cfg
from lhotse_b200 import build_plan
from lhotse_b200.engine import OUT_PADDED, B200FeatError, Engine, pack_device, stage_host
from lhotse_b200.extractors import (B200FbankConfig, B200LibrosaFbankConfig, B200LogSpectrogramConfig, B200MfccConfig,
                                    B200SpectrogramConfig, B200WhisperFbankConfig)
from lhotse_b200.families import (B200KaldifeatFbank, B200KaldifeatFbankConfig, B200KaldifeatFrameOptions,
                                  B200KaldifeatMelOptions, B200KaldifeatMfcc, B200KaldifeatMfccConfig)
from oracle import kaldi_oracle as O
from oracle import librosa_oracle as LO
from oracle import whisper_oracle as W
from test_librosa import librosa_gate
from test_whisper import whisper_gate

pytestmark = pytest.mark.gpu

PAD = -7.25  # a padding value other than the extractors' LOG_EPSILON default


@dataclass(frozen=True)
class Row:
    """One kernel of the table: the plan geometry that selects it and what the handle must report."""
    id: str
    kernel: str        # Engine.kernel expected
    N: int             # plan.N expected
    sr: int
    request: str = "auto"
    frame: dict = field(default_factory=dict)


ROWS = [
    Row("generic", "generic", 512, 16000, request="generic"),
    Row("fast256", "fast", 256, 8000),
    Row("fast400", "fast", 400, 16000, frame={"round_to_power_of_two": False}),
    Row("fast512", "fast", 512, 16000),
    Row("fast1024-24k", "fast", 1024, 24000),
    Row("fast1024-22k", "fast", 1024, 22050),   # L = 551: odd frame length
    Row("fast2048-44k", "fast", 2048, 44100),   # S = 441: every other frame starts on an odd sample
    Row("fast2048-48k", "fast", 2048, 48000),
    Row("tc", "tc", 512, 16000, request="tc"),
]
ROW = {r.id: r for r in ROWS}

CONFIGS = {"fbank": B200FbankConfig, "mfcc": B200MfccConfig, "spectrogram": B200SpectrogramConfig,
           "log-spectrogram": B200LogSpectrogramConfig}

# feature kinds of part A: (feature, config fields); the tensor-core kernel serves fbank / mfcc without an energy column
KINDS = {
    "fbank": ("fbank", {}),
    "fbank-energy": ("fbank", {"use_energy": True}),                        # energy in column 0, mel bins shifted by one
    "fbank-htk": ("fbank", {"use_energy": True, "htk_compat": True}),       # energy in the last column
    "mfcc": ("mfcc", {}),
    "mfcc-energy": ("mfcc", {"use_energy": True}),                          # C0 <- log-energy
    "mfcc-htk-energy": ("mfcc", {"use_energy": True, "htk_compat": True}),  # log-energy in the last column
    "spectrogram-energy": ("spectrogram", {"use_energy": True}),            # bin 0 <- log-energy
    "log-spectrogram-energy": ("log-spectrogram", {"use_energy": True}),
}
TC_KINDS = ("fbank", "mfcc")


def kaldi_cfg(row: Row, feature: str, extra: dict) -> dict:
    cfg = dict(sampling_rate=row.sr, **row.frame, **extra)
    if feature == "fbank" and row.sr == 8000:
        cfg["num_filters"] = 40  # 80 filters are too narrow for the 4 kHz band at N = 256
    return cfg


def make_engine(plan, row: Row) -> Engine:
    eng = Engine(plan, kernel=row.request)
    assert eng.kernel == row.kernel and plan.N == row.N, (row.id, eng.kernel, plan.N)
    return eng


def edge_lengths(L: int, S: int, sr: int):
    """Frame-count edges as in the per-kernel sweeps: one frame, one sample more, just below half a hop past ten hops,
    a few seconds, and an odd length."""
    return [L, L + 1, 10 * S + S // 2 - 1, 3 * sr + S // 3, (41 * S + 7) | 1]


def seeded_cuts(lens, seed):
    rs = np.random.RandomState(seed)
    return [(0.1 * rs.randn(n)).astype(np.float32) for n in lens]


def ordered(a: np.ndarray) -> np.ndarray:
    """float32 bit patterns as integers that order like the values (so that a difference counts ulps, across 0 too)."""
    i = np.ascontiguousarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.where(i < 0, np.int64(-(2 ** 31)) - i, i)


def affine_tables(F: int):
    """Differs in every column and changes sign column to column, so that a value stored under a neighbour's column (or
    column 0's) transforms visibly differently."""
    c = np.arange(F, dtype=np.float64)
    return ((-1.0) ** c * (0.5 + c / F)).astype(np.float32), (3.0 * c - F).astype(np.float32)


def assert_affine(got, plain, scale, shift, what):
    """got == float32(float64(plain) * scale + shift) within 1 ulp: the kernels fuse it into one fmaf, the reference
    rounds the float64 result once more."""
    got, plain = np.asarray(got), np.asarray(plain)
    assert got.shape == plain.shape, (what, got.shape, plain.shape)
    want = (plain.astype(np.float64) * scale.astype(np.float64) + shift.astype(np.float64)).astype(np.float32)
    assert np.isfinite(got).all() and np.isfinite(want).all(), what
    ulps = np.abs(ordered(got) - ordered(want))
    bad = np.argwhere(ulps > 1)
    assert bad.size == 0, f"{what}: {len(bad)} values off by more than 1 ulp, first at (row, col) {tuple(bad[0])}"


def kaldi_reference(x, feature, cfg):
    """(fp32 oracle, float64 oracle) of one cut in the layout the plan produces: with htk_compat the energy / C0 column
    moves last, and an MFCC without energy has C0 * sqrt(2) there."""
    c = {k: v for k, v in cfg.items() if k != "htk_compat"}
    ocfg = oracle_cfg(feature, c)
    ref, truth = O.extract(x, ocfg), O.extract(x, ocfg, dtype=torch.float64)
    if cfg.get("htk_compat"):
        perm = list(range(1, ref.shape[1])) + [0]
        ref, truth = ref[:, perm].copy(), truth[:, perm].copy()
        if feature == "mfcc" and not cfg.get("use_energy"):
            ref[:, -1] *= np.float32(math.sqrt(2.0))
            truth[:, -1] *= math.sqrt(2.0)
    return ref, truth


def check_affine_on_engines(plain, aff, xs, scale, shift, gate_cut):
    """Part A's assertions for one plan: packed and padded device paths, padding rows, switching the affine off again,
    and the plain output of two cuts against the float64 oracle (`gate_cut(i, rows)` raises on failure)."""
    dev = plain.device
    buf, lens, offs = pack_device([torch.from_numpy(x) for x in xs], dev)
    p_packed, prefix = plain.extract_device(buf, lens, offsets=offs)
    a_packed, a_prefix = aff.extract_device(buf, lens, offsets=offs)
    p_packed, a_packed = p_packed.cpu().numpy(), a_packed.cpu().numpy()
    assert np.array_equal(prefix, a_prefix)
    assert_affine(a_packed, p_packed, scale, shift, "packed")

    p_pad, _ = plain.extract_device(buf, lens, offsets=offs, out_mode=OUT_PADDED, pad_value=PAD)
    a_pad, _ = aff.extract_device(buf, lens, offsets=offs, out_mode=OUT_PADDED, pad_value=PAD)
    p_pad, a_pad = p_pad.cpu().numpy(), a_pad.cpu().numpy()
    pad_row = (np.float64(PAD) * scale.astype(np.float64) + shift.astype(np.float64)).astype(np.float32)
    assert p_pad.shape == a_pad.shape == (len(xs), int(np.diff(prefix).max()), plain.feature_dim)
    for i in range(len(xs)):
        T = int(prefix[i + 1] - prefix[i])
        assert np.array_equal(p_pad[i, :T], p_packed[prefix[i]: prefix[i + 1]]), f"cut {i}: padded rows != packed rows"
        assert_affine(a_pad[i, :T], p_pad[i, :T], scale, shift, f"padded, cut {i}")
        assert np.all(p_pad[i, T:] == np.float32(PAD)), f"cut {i}: plain padding"
        assert np.array_equal(a_pad[i, T:], np.broadcast_to(pad_row, a_pad[i, T:].shape)), f"cut {i}: affine padding"

    aff.set_output_affine(None, None)
    again, _ = aff.extract_device(buf, lens, offsets=offs)
    assert np.array_equal(again.cpu().numpy(), p_packed), "affine switched off: output differs from the plain handle"

    for i in (1, len(xs) - 1):
        gate_cut(i, p_packed[prefix[i]: prefix[i + 1]])


# ---------------------------------------------------------------------------------------------- A. output affine
A_CASES = [(r.id, k) for r in ROWS for k in KINDS if r.kernel != "tc" or k in TC_KINDS]


@pytest.mark.parametrize("row_id,kind", A_CASES, ids=[f"{r}-{k}" for r, k in A_CASES])
def test_output_affine_every_epilogue(row_id, kind):
    row = ROW[row_id]
    feature, extra = KINDS[kind]
    cfg = kaldi_cfg(row, feature, extra)
    plan = build_plan(feature, CONFIGS[feature](**cfg))
    plain, aff = make_engine(plan, row), make_engine(plan, row)
    F = plain.feature_dim
    scale, shift = affine_tables(F)
    aff.set_output_affine(scale, shift)
    xs = seeded_cuts(edge_lengths(plan.L, plan.S, row.sr), seed=ROWS.index(row))

    def gate_cut(i, rows):
        ref, truth = kaldi_reference(xs[i], feature, cfg)
        assert rows.shape == ref.shape, (i, rows.shape, ref.shape)
        ok, msg = gate(rows, ref, truth, feature, use_energy=bool(cfg.get("use_energy")))
        assert ok, f"cut {i}: {msg}"

    check_affine_on_engines(plain, aff, xs, scale, shift, gate_cut)


@pytest.mark.parametrize("fft_size", [256, 512, 1024, 2048])
def test_output_affine_librosa_fbank(fft_size):
    """The log10 mel epilogue of the fast kernels (librosa-fbank, centred framing)."""
    cfg = dict(sampling_rate=22050, fft_size=fft_size, hop_size=fft_size // 4)
    plan = build_plan("librosa-fbank", B200LibrosaFbankConfig(**cfg))
    row = Row(f"librosa{fft_size}", "fast", fft_size, 22050)
    plain, aff = make_engine(plan, row), make_engine(plan, row)
    scale, shift = affine_tables(plain.feature_dim)
    aff.set_output_affine(scale, shift)
    N, S = fft_size, plan.S
    xs = seeded_cuts([N // 2 + 1, N + 1, 10 * S + S // 2 - 1, 3 * 22050 + S // 3, (41 * S + 7) | 1], seed=fft_size)
    full = B200LibrosaFbankConfig(**cfg).to_dict()

    def gate_cut(i, rows):
        truth = LO.extract(xs[i], float64=True, **cfg)
        assert rows.shape == truth.shape, (i, rows.shape, truth.shape)
        ok, msg = librosa_gate(rows, truth, full)
        assert ok, f"cut {i}: {msg}"

    check_affine_on_engines(plain, aff, xs, scale, shift, gate_cut)


def test_whisper_fbank_refuses_the_output_affine():
    """Its normalise pass clamps against each cut's own maximum, so a column affine cannot be fused into it."""
    plan = build_plan("whisper-fbank", B200WhisperFbankConfig())
    for row in (Row("whisper-generic", "generic", 400, 16000, request="generic"), Row("whisper-fast400", "fast", 400, 16000)):
        eng = make_engine(plan, row)
        scale, shift = affine_tables(eng.feature_dim)
        with pytest.raises(B200FeatError) as e:
            eng.set_output_affine(scale, shift)
        assert e.value.code == -2, row.id


# ---------------------------------------------------------------------------------------------- B. htk layout
B_CASES = [(r.id, f, e) for r in ROWS for f, e in (("fbank", True), ("mfcc", True), ("mfcc", False))
           if r.kernel != "tc" or (f == "mfcc" and not e)]


def kaldifeat_pair(row: Row, feature: str, use_energy: bool):
    frame = B200KaldifeatFrameOptions(sampling_rate=row.sr, round_to_power_of_two=row.frame.get("round_to_power_of_two", True))
    if feature == "fbank":
        mel = B200KaldifeatMelOptions(num_bins=40 if row.sr == 8000 else 80)
        mk = lambda htk: B200KaldifeatFbank(B200KaldifeatFbankConfig(frame_opts=frame, mel_opts=mel, use_energy=use_energy,
                                                                     htk_compat=htk, kernel=row.request))
    else:
        mk = lambda htk: B200KaldifeatMfcc(B200KaldifeatMfccConfig(frame_opts=frame, use_energy=use_energy, htk_compat=htk,
                                                                   kernel=row.request))
    return mk(True), mk(False)


@pytest.mark.parametrize("row_id,feature,use_energy", B_CASES,
                         ids=[f"{r}-{f}{'-energy' if e else ''}" for r, f, e in B_CASES])
def test_htk_compat_column_move_every_kernel(row_id, feature, use_energy):
    row = ROW[row_id]
    htk_ext, plain_ext = kaldifeat_pair(row, feature, use_energy)
    for ext in (htk_ext, plain_ext):
        inner = ext._inner(row.sr)
        assert inner.engine.kernel == row.kernel and inner.plan.N == row.N, (row.id, inner.engine.kernel, inner.plan.N)
    hplan = htk_ext._inner(row.sr).plan
    assert hplan.energy_last
    xs = seeded_cuts(edge_lengths(hplan.L, hplan.S, row.sr), seed=100 + ROWS.index(row))
    htk, plain = htk_ext.extract(xs, row.sr), plain_ext.extract(xs, row.sr)
    assert len(htk) == len(plain) == len(xs)
    for i, (h, p) in enumerate(zip(htk, plain)):
        assert h.shape == p.shape, (i, h.shape, p.shape)
        if use_energy:  # a pure column move; the DCT sums over m run in the same order for every column
            assert np.array_equal(h[:, :-1], p[:, 1:]), f"cut {i}: columns 1.. did not move left by one"
            assert np.array_equal(h[:, -1], p[:, 0]), f"cut {i}: energy column"
        else:  # C0 moves last and takes sqrt(2) through the lifter slot (Kaldi's lifter[0] is 1)
            assert np.array_equal(h[:, :-1], p[:, 1:]), f"cut {i}: C1.. did not move left by one"
            assert np.array_equal(h[:, -1], p[:, 0] * np.float32(math.sqrt(2.0))), f"cut {i}: C0 * sqrt(2)"
    # the permuted output against the float64 oracle on one cut (the adapters use Kaldi's log-energy convention, which
    # equals the oracle's log(E + 1e-15) on noise far above the floor)
    cfg = dict(sampling_rate=row.sr, use_energy=use_energy, htk_compat=True, **row.frame)
    if feature == "fbank":
        cfg["num_filters"] = 40 if row.sr == 8000 else 80
    i = len(xs) - 1
    ref, truth = kaldi_reference(xs[i], feature, cfg)
    ok, msg = gate(htk[i], ref, truth, feature, use_energy=use_energy)
    assert ok, msg


# ---------------------------------------------------------------------------------------------- C. chunked host pipelines
CHUNK_BYTES = 32 << 20  # b200feat.cu: the host pipelines cut a batch into chunks of 32 MB of samples


def chunk_count(lens, offs, esz):
    """The host pipelines' greedy split: a chunk takes cuts while their span stays within CHUNK_BYTES of samples."""
    cap, n, b0 = CHUNK_BYTES // esz, 0, 0
    while b0 < len(lens):
        b1 = b0 + 1
        while b1 < len(lens) and offs[b1] + lens[b1] - offs[b0] <= cap:
            b1 += 1
        n, b0 = n + 1, b1
    return n


def aligned_offsets(lens, align=1):
    """Start of every cut when staged in order, each start rounded up to `align` elements."""
    offs, cur = [], 0
    for n in lens:
        cur = (cur + align - 1) // align * align
        offs.append(cur)
        cur += n
    return offs


def make_chunked_batch(esz, seed):
    """Cuts for three chunks of `esz`-byte samples: two chunks of long cuts (1-2.5 M samples, quiet noise with a stretch
    of digital silence) interleaved with short odd-length loud cuts, each chunk closed by a long cut sized to leave a gap
    smaller than any short cut, then a last chunk of short cuts only.  Back to back, the odd lengths put later cuts on odd
    offsets.  The silence makes whisper-fbank's output depend on each cut's own maximum (its clamp at max - 8)."""
    rs = np.random.RandomState(seed)
    cap = CHUNK_BYTES // esz
    lens, loud = [], []

    def short():
        lens.append(int(rs.randint(2500, 30000)) * 2 + 1)
        loud.append(True)

    for _ in range(2):
        span = 0
        while True:
            if rs.rand() < 0.6:
                short()
                span += lens[-1]
            room = cap - span - 4000  # far above the alignment gaps of the staged layouts, below any short cut
            n = room if room <= 3_500_000 else int(rs.randint(1_000_000, min(2_500_000, room - 1_000_000)))
            lens.append(n)
            loud.append(False)
            span += n
            if n == room:
                break
    for _ in range(4):
        short()
    cuts = []
    for n, is_loud in zip(lens, loud):
        if is_loud:
            x = (0.3 * rs.randn(n)).astype(np.float32)
        else:
            x = (0.02 * rs.randn(n)).astype(np.float32)
            a = int(rs.randint(0, n // 2))
            x[a: a + n // 3] = 0.0
        cuts.append(x)
    if esz == 2:
        cuts = [np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16) for x in cuts]
    return cuts


@pytest.fixture(scope="module")
def chunked_batches():
    batches = {np.float32: make_chunked_batch(4, 21), np.int16: make_chunked_batch(2, 22)}
    for dt, cuts in batches.items():
        esz = np.dtype(dt).itemsize
        lens = [len(c) for c in cuts]
        assert chunk_count(lens, aligned_offsets(lens), esz) >= 3 and sum(lens) * esz < (100 << 20)
    return batches


def _kaldi_plan(row: Row):
    cfg = kaldi_cfg(row, "fbank", {})
    return build_plan("fbank", B200FbankConfig(**cfg)), ("fbank", cfg)


C_PLANS = {r.id: (lambda r=r: (r,) + _kaldi_plan(r)) for r in ROWS}
C_PLANS["whisper-generic"] = lambda: (Row("whisper-generic", "generic", 400, 16000, request="generic"),
                                      build_plan("whisper-fbank", B200WhisperFbankConfig()), ("whisper-fbank", None))
C_PLANS["whisper-fast400"] = lambda: (Row("whisper-fast400", "fast", 400, 16000),
                                      build_plan("whisper-fbank", B200WhisperFbankConfig()), ("whisper-fbank", None))
C_PLANS["librosa-fast1024"] = lambda: (Row("librosa-fast1024", "fast", 1024, 22050),
                                       build_plan("librosa-fbank", B200LibrosaFbankConfig()), ("librosa-fbank", None))


def _gate_against_oracle(kind, x, rows):
    feature, cfg = kind
    if feature == "whisper-fbank":
        ok, msg = whisper_gate(rows, W.extract(x), W.extract(x, dtype=torch.float64))
    elif feature == "librosa-fbank":
        ok, msg = librosa_gate(rows, LO.extract(x, float64=True), B200LibrosaFbankConfig().to_dict())
    else:
        ref, truth = kaldi_reference(x, feature, cfg)
        assert rows.shape == ref.shape
        ok, msg = gate(rows, ref, truth, feature)
    assert ok, msg


@pytest.mark.parametrize("dtype", [np.float32, np.int16], ids=["float32", "int16"])
@pytest.mark.parametrize("plan_id", list(C_PLANS))
def test_chunked_host_routes_match_one_device_launch(plan_id, dtype, chunked_batches, monkeypatch):
    monkeypatch.delenv("B200FEAT_PY_GATHER", raising=False)  # extract_host_list: the C pointer-list route
    row, plan, kind = C_PLANS[plan_id]()
    eng = make_engine(plan, row)
    per_chunk = 2 if plan.feature == "whisper-fbank" else 1  # whisper-fbank: fused kernel + normalise pass
    cuts = chunked_batches[dtype]
    esz = np.dtype(dtype).itemsize
    lens = [len(c) for c in cuts]
    staged, _, offs = stage_host(cuts, dtype=dtype)  # pinned, every cut on a 4-element boundary

    # the yardstick: the whole batch in one launch on the device
    dev = staged.to(eng.device)
    want, prefix = eng.extract_device(dev, lens, offsets=offs)
    want = want.cpu().numpy()
    want_pad, _ = eng.extract_device(dev, lens, offsets=offs, out_mode=OUT_PADDED, pad_value=PAD)
    want_pad = want_pad.cpu().numpy()
    del dev

    def launches():
        return eng.stats()["kernel_launches"]

    # 1. extract_host, cuts back to back (pageable memory)
    flat = np.concatenate(cuts)
    k0 = launches()
    got, got_prefix = eng.extract_host(flat, lens)
    n1 = chunk_count(lens, aligned_offsets(lens), esz)
    assert n1 >= 3 and launches() - k0 >= per_chunk * n1
    assert np.array_equal(got_prefix, prefix) and np.array_equal(got, want), "extract_host, packed back to back"

    # 2. extract_host at the aligned offsets of stage_host, padded output
    k0 = launches()
    got, _ = eng.extract_host(staged, lens, out_mode=OUT_PADDED, pad_value=PAD, offsets=offs)
    n2 = chunk_count(lens, offs, esz)
    assert n2 >= 3 and launches() - k0 >= per_chunk * n2
    assert got.shape == want_pad.shape and np.array_equal(got, want_pad), "extract_host, staged, padded"

    # 3. extract_host_list: the library gathers the cuts itself (16-byte aligned starts)
    k0 = launches()
    got, got_prefix = eng.extract_host_list(cuts, dtype=dtype)
    n3 = chunk_count(lens, aligned_offsets(lens, 16 // esz), esz)
    assert n3 >= 3 and launches() - k0 >= per_chunk * n3
    assert np.array_equal(got_prefix, prefix) and np.array_equal(got, want), "extract_host_list"

    # two cuts of the last chunk against the CPU oracle: the host and the device path cannot both be wrong the same way
    for i in (len(cuts) - 2, len(cuts) - 1):
        x = cuts[i].astype(np.float32) / 32768.0 if dtype == np.int16 else cuts[i]
        _gate_against_oracle(kind, x, want[prefix[i]: prefix[i + 1]])

