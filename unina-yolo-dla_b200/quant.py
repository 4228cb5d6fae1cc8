"""INT8 execution of the QAT graph (reference: qat.py:91-126 quantiser configuration, qat.py:700-753
precision carve-out, train.py:721-725 ``quant_modules.initialize()``).

Every ``nn.Conv2d`` outside the float layers is a QuantConv2d: 8-bit, narrow range, per-tensor scales for
inputs *and* weights.  With static ``_amax`` the fake-quant convolution is an integer computation:

    q_x = clamp(rne(x * 127 / amax_x), -127, 127)        (uyd_plan_add_quantize, from the bf16 activation)
    q_w = clamp(rne(w * 127 / amax_w), -127, 127)        (here, on the host)
    acc = sum q_x * q_w                                   (int32, exact: tcgen05 kind::i8 / dp4a)
    y   = float(acc) * m_c + b_c ; ReLU ; (+ residual) ; round to bf16     (conv epilogue)
          m_c = (amax_x / 127) (amax_w / 127) gamma_c / sqrt(var_c + eps),  b_c = beta_c - mu_c gamma_c / sqrt(var_c + eps)

BN, ReLU, residual adds, concat, max-pool and upsample stay floating point (bf16 activations), exactly as
in the QAT graph.  The arithmetic of every step is fixed (fp32 round-to-nearest operations in a fixed order),
so the outputs are bit-exact with respect to the integer reference of the test-suite.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

IN_SUFFIX = "._input_quantizer._amax"
W_SUFFIX = "._weight_quantizer._amax"


@dataclass
class QuantSpec:
    amax: dict = field(default_factory=dict)          # conv module name -> (input amax, weight amax)
    # kept in floating point (qat.py:700-753): an int i names the layer model.{i} (YAML network), a str any conv whose
    # module name contains it (model.py network, e.g. "stem" or "head_p2")
    float_layers: tuple = (0, 1, 2)

    def covers(self, name: str) -> bool:
        if name not in self.amax:
            return False
        parts = name.split(".")
        layer = int(parts[1]) if len(parts) > 1 and parts[0] == "model" and parts[1].isdigit() else None
        return not any(f in name if isinstance(f, str) else f == layer for f in self.float_layers)


def amax_state_dict(spec: QuantSpec | None) -> dict:
    """The ``_amax`` buffers of a quantisation in pytorch-quantization's naming."""
    out = {}
    for n, (ai, aw) in (spec.amax if spec else {}).items():
        out[n + IN_SUFFIX] = torch.tensor(ai)
        out[n + W_SUFFIX] = torch.tensor(aw)
    return out


def scale_of(amax: float) -> np.float32:
    return np.float32(127.0) / np.float32(amax)


def quantize_weights(w: torch.Tensor, amax: float) -> np.ndarray:
    """Weight quantiser: per-tensor, fp32 multiply, round half to even, narrow range."""
    s = scale_of(amax)
    return np.clip(np.rint(w.detach().float().cpu().numpy().astype(np.float32) * s), -127, 127).astype(np.int8)


def requant_params(amax_x: float, amax_w: float, bn: torch.nn.BatchNorm2d | None, conv_bias: torch.Tensor | None):
    """Per-channel (m_c, b_c) of the requant epilogue, fp32."""
    sx = np.float32(amax_x) / np.float32(127.0)
    sw = np.float32(amax_w) / np.float32(127.0)
    if bn is None:
        b = conv_bias.detach().float().cpu().numpy().astype(np.float32)
        return np.full(b.shape[0], sx * sw, np.float32), b
    g = bn.weight.detach().double().cpu().numpy() / np.sqrt(bn.running_var.detach().double().cpu().numpy() + bn.eps)
    m = (np.float64(sx) * np.float64(sw) * g).astype(np.float32)
    b = (bn.bias.detach().double().cpu().numpy() - bn.running_mean.detach().double().cpu().numpy() * g).astype(np.float32)
    return m, b


def split_state_dict(sd: dict):
    """Separates pytorch-quantization ``_amax`` buffers from the module parameters."""
    plain, amax_in, amax_w = {}, {}, {}
    for k, v in sd.items():
        if k.endswith(IN_SUFFIX):
            amax_in[k[: -len(IN_SUFFIX)]] = float(torch.as_tensor(v).max())
        elif k.endswith(W_SUFFIX):
            amax_w[k[: -len(W_SUFFIX)]] = float(torch.as_tensor(v).max())
        else:
            plain[k] = v
    amax = {n: (amax_in[n], amax_w[n]) for n in amax_in if n in amax_w}
    return plain, amax


def calibration_rule(method: str) -> str:
    """The amax rule of a ``calibrate_int8`` method ("histogram" is the reference's entropy rule)."""
    rule = {"histogram": "entropy"}.get(method, method)
    if rule not in ("max", "entropy", "percentile", "mse"):
        raise ValueError(f"unknown calibration method {method!r}")
    return rule


def collect_input_amax(p, x_all: torch.Tensor, batch: int, names: list, rule: str, percentile: float = 99.99,
                       per_batch=None) -> list:
    """Input amax of every conv in ``names`` over the frames ``x_all``, run through the bf16 plan ``p`` in chunks of
    ``batch``; ``p.conv_inputs`` maps each name to the bf16 slice the conv reads.  Per chunk: one max |x| reduction
    (uyd_plan_slice_absmax) per input and, unless ``rule`` is "max", one |x| histogram (uyd_plan_slice_histogram);
    ``per_batch(x, nb)`` runs after them."""
    from ._lib import UydError

    vmax = [0.0] * len(names)
    cal = [HistogramCalibrator() for _ in names] if rule != "max" else None
    for b0 in range(0, x_all.shape[0], batch):
        x = x_all[b0:b0 + batch].contiguous()
        nb = x.shape[0]
        p.run(x)
        bits = torch.zeros(len(names), dtype=torch.int32, device=x.device)
        for i, n in enumerate(names):
            p.slice_absmax(p.conv_inputs[n], nb, bits[i:i + 1])
        vals = bits.view(torch.float32).cpu().tolist()
        vmax = [max(a, b) for a, b in zip(vmax, vals)]
        if cal is not None:
            nbins = [c.bins_for(v) for c, v in zip(cal, vals)]
            if max(nbins) > 12288:
                raise UydError("histogram calibration: a later batch exceeds 6x the first batch's range; "
                               "put representative frames first")
            offs = np.concatenate(([0], np.cumsum(nbins)))
            hist = torch.zeros(int(offs[-1]), dtype=torch.int32, device=x.device)
            for i, n in enumerate(names):
                p.slice_histogram(p.conv_inputs[n], nb, 1.0 / cal[i].width, hist[int(offs[i]):int(offs[i + 1])])
            h = hist.cpu().numpy()
            for i in range(len(names)):
                cal[i].add(h[int(offs[i]):int(offs[i + 1])])
        if per_batch is not None:
            per_batch(x, nb)
    return [vmax[i] if rule == "max" else cal[i].compute_amax(rule, percentile) for i in range(len(names))]


def weight_amax(w: torch.Tensor, rule: str, percentile: float = 99.99) -> float:
    """Weight amax on the host with the same rule as the inputs."""
    if rule == "max":
        return float(w.detach().abs().max())
    c = HistogramCalibrator()
    c.collect_host(w.detach().float().cpu().numpy())
    return c.compute_amax(rule, percentile)


# ------------------------------------------------------------------------------------------------------
# Histogram calibration (SURVEY 8f-4).  qat.py:91-126 configures pytorch-quantization's HistogramCalibrator for
# inputs AND weights ("histogram" is the default of initialize_quantization), qat.py:676-697 selects "entropy" as
# the amax method; the reference never materialises the scales (SURVEY 3.5).  pytorch-quantization (2.1.2,
# demo.ipynb) is not vendored: the collection rule and the three amax methods below restate its published
# calib/histogram.py; the GPU part is uyd_plan_slice_absmax + uyd_plan_slice_histogram.  PARITY UNPINNED w.r.t. the
# library itself; pinned against a loop-form restatement kept with the test infrastructure.
# ------------------------------------------------------------------------------------------------------
NUM_BINS = 2048


class HistogramCalibrator:
    """|x| histogram of one tensor over several batches: ``NUM_BINS`` bins over [0, max of the first batch]; a later
    batch with a larger maximum extends the range by whole bins of the same width (HistogramCalibrator.collect)."""

    def __init__(self, num_bins: int = NUM_BINS):
        self.num_bins = num_bins
        self.width = None            # bin width, fixed by the first batch
        self.hist = None             # int64 counts

    def bins_for(self, batch_max: float) -> int:
        """Number of bins the next batch needs (>= the current length)."""
        if self.width is None:
            self.width = max(float(batch_max), 1e-12) / self.num_bins
            return self.num_bins
        cur = len(self.hist) if self.hist is not None else self.num_bins
        need = int(np.ceil(float(batch_max) / self.width - 1e-9))
        return max(cur, need)

    def add(self, counts: np.ndarray) -> None:
        counts = np.asarray(counts, dtype=np.int64)
        if self.hist is None:
            self.hist = counts.copy()
        else:
            if len(counts) > len(self.hist):
                self.hist = np.concatenate((self.hist, np.zeros(len(counts) - len(self.hist), np.int64)))
            self.hist[: len(counts)] += counts

    def collect_host(self, x: np.ndarray) -> None:
        """Host-side collection (weights): same binning rule as the GPU kernel."""
        a = np.abs(np.asarray(x, dtype=np.float32)).reshape(-1)
        n = self.bins_for(float(a.max()) if a.size else 0.0)
        inv = np.float32(1.0 / self.width)
        idx = np.minimum((a * inv).astype(np.int64), n - 1)
        self.add(np.bincount(idx, minlength=n))

    @property
    def edges(self) -> np.ndarray:
        return np.arange(len(self.hist) + 1, dtype=np.float64) * self.width

    def compute_amax(self, method: str = "entropy", percentile: float = 99.99) -> float:
        if method == "entropy":
            return amax_entropy(self.hist, self.edges)
        if method == "percentile":
            return amax_percentile(self.hist, self.edges, percentile)
        if method == "mse":
            return amax_mse(self.hist, self.edges)
        if method == "max":
            nz = np.nonzero(self.hist)[0]
            return float(self.edges[nz[-1] + 1]) if len(nz) else 0.0
        raise ValueError(f"unknown amax method {method!r}")


def _kl(p: np.ndarray, q: np.ndarray) -> float:
    """scipy.stats.entropy(p, q): both normalised, 0 log 0 = 0, p > 0 = q gives inf."""
    p = p / p.sum()
    q = q / q.sum()
    m = p > 0
    if np.any(q[m] == 0):
        return float("inf")
    return float(np.sum(p[m] * np.log(p[m] / q[m])))


def amax_entropy(hist, edges, num_bits: int = 8, unsigned: bool = False, stride: int = 1, start_bin: int = 128) -> float:
    """KL-divergence threshold search (_compute_amax_entropy): for every candidate length i the first i bins are
    merged into 2^(bits-1) quantisation levels (empty source bins stay empty, a level's mass is spread evenly over
    its non-empty source bins) and compared with the reference distribution whose last bin absorbs the outliers;
    the LAST minimum wins."""
    bins = np.asarray(hist, dtype=np.float64).copy()
    bins[0] = bins[1]
    total = bins.sum()
    nlev = 1 << (num_bits - 1 + int(unsigned))
    stop = len(bins)
    tail = np.concatenate((np.cumsum(bins[::-1])[::-1], [0.0]))   # tail[i] = sum(bins[i:])
    div = []
    for i in range(start_bin, stop + 1, stride):
        space = np.linspace(0, i, num=nlev + 1)
        lev = np.digitize(np.arange(i), space) - 1
        src = bins[:i]
        nz = src != 0
        mass = np.bincount(lev[nz], weights=src[nz], minlength=nlev)
        cnt = np.bincount(lev[nz], minlength=nlev)
        per = np.divide(mass, cnt, out=np.zeros(nlev), where=cnt > 0)
        new = np.where(nz, per[lev], 0.0)
        ref = src.copy()
        ref[-1] += tail[i]
        if round(new.sum() + tail[i]) != round(total) or round(ref.sum()) != round(total):
            raise RuntimeError("entropy calibration: count mismatch")
        div.append(_kl(ref, new) if new.sum() > 0 else float("inf"))
    div = np.asarray(div)
    last_argmin = len(div) - 1 - int(np.argmin(div[::-1]))
    return float(edges[last_argmin * stride + start_bin])


def amax_percentile(hist, edges, percentile: float) -> float:
    if not 0 <= percentile <= 100:
        raise ValueError("percentile must be in [0, 100]")
    h = np.asarray(hist, dtype=np.float64)
    cdf = np.cumsum(h / h.sum())
    return float(edges[int(np.searchsorted(cdf, percentile / 100.0))])


def amax_mse(hist, edges, num_bits: int = 8, unsigned: bool = False, stride: int = 1, start_bin: int = 128) -> float:
    counts = np.asarray(hist, dtype=np.float64)
    centers = (edges[1:] + edges[:-1]) / 2
    bound = (1 << (num_bits - 1 + int(unsigned))) - 1
    best, arg = None, start_bin
    for i in range(start_bin, len(centers), stride):
        amax = centers[i]
        scale = bound / amax
        q = np.clip(np.rint(centers.astype(np.float32) * np.float32(scale)), -bound, bound) / np.float32(scale)
        mse = float((((q - centers) ** 2) * counts).mean())
        if best is None or mse < best:
            best, arg = mse, i
    return float(centers[arg])
