import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Sampled:
    """A golden array stored as every `stride`-th element of its flattened form (tools/make_golden.py samples the large gradient
    arrays so that each fixture stays under 1 MB).  `absmax` is max|.| over the whole array."""

    def __init__(self, values, shape, stride, absmax):
        self.values, self.shape, self.stride, self.absmax = values, tuple(int(s) for s in shape), int(stride), float(absmax)

    def take(self, t):
        """The elements of a whole array `t` (of this array's shape) at the stored positions, as float64."""
        t = torch.as_tensor(t).detach().double().cpu()
        assert tuple(t.shape) == self.shape, (tuple(t.shape), self.shape)
        return t.reshape(-1)[::self.stride]

    def like(self, t):
        """A whole array `t` reduced to the same positions."""
        t = torch.as_tensor(t).detach().double().cpu()
        return Sampled(self.take(t).numpy(), self.shape, self.stride, t.abs().max().item())


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = {k: z[k] for k in z.files if "@" not in k}
    for k in g:
        if k + "@stride" in z.files:
            g[k] = Sampled(g[k], z[k + "@shape"], z[k + "@stride"], z[k + "@absmax"])
    return g


def T(a, dtype=None, device=None):
    t = torch.from_numpy(np.asarray(a))
    if dtype is not None:
        t = t.to(dtype)
    if device is not None:
        t = t.to(device)
    return t


def rel_err(a, b):
    """per-tensor max|a-b| / max|b|  (the metric SURVEY §8(d) fixes for every float comparison).  With a `Sampled` golden on either
    side the maximum runs over its stored elements; the denominator stays max|b| over the whole array."""
    if isinstance(a, Sampled) or isinstance(b, Sampled):
        s = a if isinstance(a, Sampled) else b
        a, b = (x if isinstance(x, Sampled) else s.like(x) for x in (a, b))
        assert (a.shape, a.stride) == (b.shape, b.stride)
        d = np.abs(a.values.astype(np.float64) - b.values.astype(np.float64)).max()
        return float(d) / (b.absmax if b.absmax > 0 else 1.0)
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    den = b.abs().max().item()
    return (a - b).abs().max().item() / (den if den > 0 else 1.0)


def close_vs_truth(got, ref32, truth64, tol=1e-5, slack=None, name=None):
    """Parity criterion for ill-conditioned fp32 reductions (pose / bias gradients: sums with heavy cancellation,
    where the fp32 reference itself is only accurate to ~1e-4 of its own value).  `truth64` is the fp64 oracle;
    `ref32` the fp32 reference (golden or fp32 oracle).  Pass iff the kernel is within `tol` of the fp32 reference, or within
    `tol` of the truth, or no further from it than `slack` x the fp32 reference's own distance.  Recorded in the parity ledger.
    Returns (ok, err_got_vs_truth, err_ref_vs_truth)."""
    truth64 = _on_golden_elements(ref32, truth64)
    e_got = rel_err(got, truth64)
    e_ref = rel_err(ref32, truth64)
    try:
        parity(name or _auto_name(), got, ref32, tol, truth=truth64, slack=TRUTH_SLACK if slack is None else slack)
        ok = True
    except AssertionError:
        ok = False
    return ok, e_got, e_ref


def _on_golden_elements(ref, truth):
    """A whole `truth` against a `Sampled` reference is reduced to the reference's stored elements, so that the kernel, the
    reference and the truth are judged on the same elements."""
    if isinstance(ref, Sampled) and truth is not None and not isinstance(truth, Sampled):
        return ref.like(truth)
    return truth


_AUTO = {}


def _auto_name():
    t = _current_test()
    _AUTO[t] = _AUTO.get(t, 0) + 1
    return "tensor_%d" % _AUTO[t]


def parity_ok(name, got, ref, tol, truth=None, outliers=0.0):
    """bool form of `parity` for compound asserts: records the comparison, returns whether it passed."""
    try:
        parity(name, got, ref, tol, truth=truth, outliers=outliers)
        return True
    except AssertionError:
        return False


# ---------------------------------------------------------------------------------------------------------------------
# Parity ledger: every float comparison of the -m gpu tests goes through `parity(...)`, which applies the stated tolerance
# (1e-5 fp32 mode / 2e-2 bf16 mode, north star) and appends the MEASURED error to gpurun_out/parity_r2.jsonl
# (tools/parity_report.py folds the lines into profiles/parity_r2.json).
# ---------------------------------------------------------------------------------------------------------------------
PARITY_LOG = os.environ.get("SNB_PARITY_LOG", os.path.join(ROOT, "gpurun_out", "parity_r2.jsonl"))
TRUTH_SLACK = 1.5   # an ill-conditioned fp32 reduction may be at most this much further from the fp64 truth than the fp32 reference is


def _current_test():
    return os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0]


ADAM_OUTLIERS = 0.02   # see `outliers` below


def rel_err_without_outliers(a, b, frac):
    """max|a-b| / max|b| after setting aside the ceil(frac * n) largest differences."""
    a = torch.as_tensor(a).detach().double().cpu().reshape(-1)
    b = torch.as_tensor(b).detach().double().cpu().reshape(-1)
    k = int(-(-frac * a.numel() // 1))
    d = torch.sort((a - b).abs())[0]
    den = b.abs().max().item()
    return (d[-1 - k].item() if k < d.numel() else 0.0) / (den if den > 0 else 1.0)


def parity(name, got, ref, tol, truth=None, slack=TRUTH_SLACK, rows=None, floor=None, floor_slack=1.25, info=False, outliers=0.0):
    """Record and judge one per-tensor comparison.  metric = max|a-b| / max|b|.
    * no `truth`: pass iff err(got, ref) <= tol.
    * `truth` (fp64 result of the same computation: the reference run in float64, or the fp64 oracle): pass iff
      err(got, ref) <= tol, or err(got, truth) <= max(tol, slack x err(ref, truth)) -- i.e. where the fp32 reference's OWN
      rounding error exceeds the tolerance the kernel must be about as close to the exact value as the reference is.
    * `floor` (bf16 mode, adversarial inputs only): the error of the CPU EMULATION of the prescribed bf16 rounding points
      against the same reference -- what any faithful bf16-MLP implementation shows on these inputs; pass iff
      err(got, ref) <= max(tol, floor_slack x floor).  Recorded as `bf16_emulation_err`.
    * `info`: record only, never fail (a second view of a tensor already judged elsewhere).
    * `outliers` (AdamW-updated parameters compared between two summation orders only): the fraction of elements set aside before
      the maximum is taken.  AdamW's first steps are ~ lr * sign(g): an element whose gradient is at summation-noise level
      (|g| <~ 1e-7 * sqrt(n_samples) of the typical one: a few 1e-5 of the elements per iteration) may step 2 lr apart in two
      orders and never come back -- the loss does not see it.  The error over ALL elements is recorded as `err_all_elements`.
    Returns the error that decided (so a test can print it)."""
    import json
    truth = _on_golden_elements(ref, truth)
    e = rel_err(got, ref)
    rec = {"test": _current_test(), "tensor": name, "tol": tol, "err_vs_ref": e}
    if outliers > 0:
        rec.update(err_all_elements=e, outliers_set_aside=outliers)
        e = rel_err_without_outliers(got, ref, outliers)
        rec["err_vs_ref"] = e
    ok = e <= tol
    if truth is not None:
        e_got, e_ref = rel_err(got, truth), rel_err(ref, truth)
        rec.update(err_vs_truth64=e_got, ref_err_vs_truth64=e_ref, slack=slack)
        ok = ok or e_got <= max(tol, slack * e_ref)
    if floor is not None:
        rec.update(bf16_emulation_err=floor, floor_slack=floor_slack)
        ok = ok or e <= max(tol, floor_slack * floor)
    if rows is not None:
        rec["rows"] = rows
    if info:
        rec["info_only"] = True
        ok = True
    rec["pass"] = bool(ok)
    try:
        os.makedirs(os.path.dirname(PARITY_LOG), exist_ok=True)
        with open(PARITY_LOG, "a") as f:
            f.write(json.dumps(rec) + "\n")
    except OSError:
        pass
    assert ok, rec
    return rec.get("err_vs_truth64", e) if not (e <= tol) else e
