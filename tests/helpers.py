"""Shared test utilities: golden fixtures, tolerance gates, the oracle-backed fake engine."""
import json
import os

import numpy as np
import torch

from oracle import kaldi_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "golden_v1.npz")

# north_star: "within 1e-4 relative (float32)".  Element-wise that cannot hold against an fp32
# reference whose own distance to the float64 truth reaches 8e-4 abs on log-mel values
# (measured: profiles/r2_parity_report.json, DESIGN.md "Parity tolerance"), so the gate is, per element,
#   |ours - truth64| / tol <= max(1, NOISE_X * N(frame)),   tol = ATOL + RTOL*|truth64|
# where N(frame) is the largest |ref32 - truth64| / tol over the element's own frame and its two neighbours: a noisy
# frame of the reference (a near-cancelling bin, a frame at the mel floor) relaxes the bound for that neighbourhood
# only, not for the whole case.  NOISE_X = 2 as SURVEY.md §7 asks.
RTOL, ATOL, NOISE_X = 1e-4, 2e-4, 2.0


def load_golden():
    g = np.load(GOLDEN)
    man = json.loads(bytes(g["manifest"]).decode())
    return [(i, c, g[f"x{i}"], g[f"y{i}"]) for i, c in enumerate(man)]


def load_golden_stream():
    """tests/golden/golden_stream_v1.npz (make_golden_stream.py): reference `online_inference` runs."""
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "golden_stream_v1.npz"))
    meta = json.loads(bytes(g["meta"]).decode())
    return [(i, m, g[f"x{i}"], g[f"y{i}"], g[f"r{i}"]) for i, m in enumerate(meta)]


def load_golden_reference_api():
    """tests/golden/golden_reference_api_v1.npz (make_golden_reference_api.py): (manifest dict, arrays by name)."""
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "golden_reference_api_v1.npz"))
    return json.loads(bytes(g["manifest"]).decode()), {k: g[k] for k in g.files if k != "manifest"}


def as_config(d):
    """A reference config stored as a dict, back as an object with the same attributes (kaldifeat's nested options
    included): `build_plan` reads configs by field name."""
    from types import SimpleNamespace

    return SimpleNamespace(**{k: as_config(v) if isinstance(v, dict) else v for k, v in d.items()})


def oracle_cfg(feature, cfg):
    return O.OracleConfig(feature=feature, **cfg)


def _unit_tolerance(truth64, feature, use_energy, use_fft_mag):
    """Element-wise tolerance 'unit' for one case (float64 arrays)."""
    if feature in ("spectrogram", "log-spectrogram"):
        # judge spectra in the linear domain: an fp32 FFT carries an amplitude error ~1e-6 of the
        # frame's largest line, whatever the bin's own size (log() would blow that up arbitrarily)
        lin = np.exp(truth64) if feature == "log-spectrogram" else truth64.copy()
        body = lin[:, 1:] if use_energy else lin
        peak = np.sqrt(np.abs(body).max(axis=1, keepdims=True)) if not use_fft_mag else np.abs(body).max(axis=1, keepdims=True)
        delta = 2e-6 * peak
        amp = np.sqrt(np.abs(lin)) if not use_fft_mag else np.abs(lin)
        tol = RTOL * np.abs(lin) + (delta if use_fft_mag else 2 * amp * delta + delta ** 2) + 1e-30
        return lin, tol
    return truth64, ATOL + RTOL * np.abs(truth64)


def gate_stats(ours, ref32, truth64, feature, use_energy=False, use_fft_mag=False):
    """Everything the parity report records for one case: tolerance units of ours / of the fp32 reference against the
    float64 truth, plain differences against the reference, and the gate's verdict."""
    ours = np.asarray(ours, dtype=np.float64)
    ref32 = np.asarray(ref32, dtype=np.float64)
    truth64 = np.asarray(truth64, dtype=np.float64)
    if ours.shape != ref32.shape:
        return {"ok": False, "msg": f"shape {ours.shape} != {ref32.shape}"}
    if not np.all(np.isfinite(ours)):
        return {"ok": False, "msg": "non-finite values"}
    tdom, tol = _unit_tolerance(truth64, feature, use_energy, use_fft_mag)
    to_dom = (lambda a: np.exp(a)) if feature == "log-spectrogram" else (lambda a: a)
    o, r = to_dom(ours), to_dom(ref32)
    if use_energy and feature in ("spectrogram", "log-spectrogram"):  # column 0 is a log-energy
        o[:, 0], r[:, 0], tdom = ours[:, 0], ref32[:, 0], tdom.copy()
        tdom[:, 0] = truth64[:, 0]
        tol[:, 0] = ATOL + RTOL * np.abs(truth64[:, 0])
    err = np.abs(o - tdom) / tol
    noise = np.abs(r - tdom) / tol
    if err.ndim == 1:
        err, noise = err[None, :], noise[None, :]
    frame_noise = noise.max(axis=1)
    nb = frame_noise.copy()  # the frame and its two neighbours
    nb[1:] = np.maximum(nb[1:], frame_noise[:-1])
    nb[:-1] = np.maximum(nb[:-1], frame_noise[1:])
    limit = np.maximum(1.0, NOISE_X * nb)[:, None]
    bad = int((err > limit).sum())
    diff = np.abs(ours - ref32)
    st = {
        "ok": bool(bad == 0 and noise.max() <= 50),
        "ours_max_units": float(err.max()), "ours_p99_units": float(np.percentile(err, 99)),
        "ref32_max_units": float(noise.max()), "ref32_p99_units": float(np.percentile(noise, 99)),
        "worst_ratio_to_limit": float((err / limit).max()), "bad": bad, "n": int(err.size),
        "max_abs_diff_vs_ref32": float(diff.max()),
        "max_rel_diff_vs_ref32": float((diff / np.maximum(np.abs(ref32), 1.0)).max()),
    }
    if noise.max() > 50:
        st["msg"] = f"reference itself is {noise.max():.1f} tolerance units from the float64 truth: wrong config?"
    else:
        st["msg"] = (f"max err/tol ours={st['ours_max_units']:.3f} ref32={st['ref32_max_units']:.3f} worst err/limit={st['worst_ratio_to_limit']:.3f} "
                     f"max|ours-ref32|={st['max_abs_diff_vs_ref32']:.3e} bad={bad}/{err.size}")
    return st


def gate(ours, ref32, truth64, feature, use_energy=False, use_fft_mag=False):
    """Returns (ok, message): every element of ours within max(1, NOISE_X * neighbourhood noise of the fp32 reference)
    tolerance units of the float64 truth (see the header)."""
    st = gate_stats(ours, ref32, truth64, feature, use_energy, use_fft_mag)
    return st["ok"], st["msg"]


class OracleEngine:
    """TEST-ONLY stand-in for lhotse_b200.engine.Engine backed by the CPU oracle, used to exercise
    the host-side container logic of the extractors where no GPU exists.  Never shipped."""

    def __init__(self, plan, feature, cfg_dict):
        self.plan = plan
        self.device = torch.device("cpu")
        self.cfg = O.OracleConfig(feature=feature, **cfg_dict)
        self.feature_dim = plan.feature_dim
        self.kernel = "oracle"

    def num_frames(self, n):
        return plan_num_frames(self.plan, n)

    def _run(self, chunks):
        outs = [O.extract(np.asarray(c, dtype=np.float32) if c.dtype != np.int16 else c.astype(np.float32) / 32768.0,
                          self.cfg) for c in chunks]
        prefix = np.concatenate(([0], np.cumsum([o.shape[0] for o in outs]))).astype(np.int64)
        return outs, prefix

    def extract_host(self, samples, num_samples, out_mode=0, pad_value=0.0, out=None, offsets=None):
        flat = samples.numpy() if isinstance(samples, torch.Tensor) else np.asarray(samples)
        chunks, o = [], 0
        for i, n in enumerate(num_samples):
            if offsets is not None:
                o = int(offsets[i])
            chunks.append(flat[o:o + int(n)])
            o += int(n)
        outs, prefix = self._run(chunks)
        if out_mode == 1:
            T = max(x.shape[0] for x in outs)
            res = np.full((len(outs), T, self.feature_dim), pad_value, dtype=np.float32)
            for i, x in enumerate(outs):
                res[i, : x.shape[0]] = x
            return res, prefix
        return np.concatenate(outs, axis=0), prefix

    def extract_host_list(self, arrays, dtype=np.float32, sub_bytes=0):
        outs, prefix = self._run([np.asarray(a) for a in arrays])
        return np.concatenate(outs, axis=0), prefix

    def extract_device(self, samples, num_samples, offsets=None, out_mode=0, pad_value=0.0, **kw):
        flat = samples.cpu().numpy()
        if offsets is None:
            offsets, cur = [], 0
            for n in num_samples:
                cur = (cur + 3) // 4 * 4
                offsets.append(cur)
                cur += n
        chunks = [flat[o:o + int(n)] for o, n in zip(offsets, num_samples)]
        outs, prefix = self._run(chunks)
        if out_mode == 1:
            T = max(x.shape[0] for x in outs)
            res = np.full((len(outs), T, self.feature_dim), pad_value, dtype=np.float32)
            for i, x in enumerate(outs):
                res[i, : x.shape[0]] = x
            return torch.from_numpy(res), prefix
        return torch.from_numpy(np.concatenate(outs, axis=0)), prefix

    def close(self):
        pass


def plan_num_frames(plan, n):
    return plan.num_frames(n)


def attach_oracle_engine(extractor):
    """Injects the fake engine into a lhotse_b200 extractor (tests of host logic only)."""
    cfg = {k: v for k, v in extractor.config.to_dict().items()
           if k in O.OracleConfig.__dataclass_fields__ and k not in ("feature",)}
    extractor._engine = OracleEngine(extractor.plan, extractor.feature_kind, cfg)
    import dataclasses

    from lhotse_b200.plan import build_plan
    snip_plan = build_plan(extractor.feature_kind, dataclasses.replace(extractor.config, snip_edges=True))
    extractor._stream_eng = OracleEngine(snip_plan, extractor.feature_kind, dict(cfg, snip_edges=True))
    return extractor
