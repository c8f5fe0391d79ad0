"""Loading of the committed golden vectors (tests/golden/*.npz, made by oracle/make_golden.py)."""
import hashlib
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_case(name):
    """The arrays of one case.  Reduced parts (oracle/make_golden.py) come back as follows: `features` is redrawn from
    its seed and checked against its SHA-256; a matrix stored as `<k>/rows` + `<k>/values` is rebuilt with zeros in the
    rows the case never reads; a [.., V] output listed under `vocab_axis/<k>` holds the entries `vocab_sample` only --
    compare it with golden_rel_err / golden_grad_close."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    out = {}
    for k in z.files:
        v = z[k]
        out[k] = v if v.dtype.kind in "US" else torch.from_numpy(v)
    if "features/seed" in out:
        g = torch.Generator().manual_seed(int(out.pop("features/seed")))
        f = torch.randn(out.pop("features/shape").tolist(), generator=g)
        assert hashlib.sha256(f.numpy().tobytes()).hexdigest() == str(out.pop("features/sha256")), \
            "torch.randn no longer reproduces the golden features from their seed"
        out["features"] = f
    for k in [k[:-len("/rows")] for k in out if k.endswith("/rows")]:
        full = torch.zeros(out.pop(k + "/shape").tolist(), dtype=out[k + "/values"].dtype)
        full[out.pop(k + "/rows")] = out.pop(k + "/values")
        out[k] = full
    return out


def params_of(case):
    return {k[3:]: v.clone() for k, v in case.items() if k.startswith("sd/")}


def rel_err(a, b, scale=None):
    """max|a-b| / max|b|  (the tolerance form of SURVEY.md 8(d)); `scale` replaces max|b|."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    d = (a - b).abs().max().item()
    s = b.abs().max().item() if scale is None else float(scale)
    return d / s if s > 0 else d


def grad_close(a, b, rtol, atol=1e-7, scale=None):
    """Gradient comparison: relative to max|ref| (or `scale`), with an absolute floor for gradients that are
    analytically zero (e.g. d/d v_a.bias -- softmax is shift invariant -- which come out as 1e-9 rounding noise)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    d = (a - b).abs().max().item()
    return d <= atol or d <= rtol * (b.abs().max().item() if scale is None else float(scale))


def _stored_part(case, key, x):
    """x reduced the way the case stores `key`, and the scale max|ref| of the full reference array (None: x is whole)."""
    if "vocab_axis/" + key not in case:
        return x, None
    idx = case["vocab_sample"].to(x.device)
    return x.index_select(int(case["vocab_axis/" + key]), idx), case["absmax/" + key]


def golden_rel_err(case, key, x):
    """rel_err(x, case[key]) for a full-size x, also where the case keeps a vocabulary sample of `key`."""
    part, scale = _stored_part(case, key, x)
    return rel_err(part, case[key], scale)


def golden_grad_close(case, key, x, rtol, atol=1e-7):
    """grad_close(x, case[key], rtol, atol) for a full-size x, also where the case keeps a vocabulary sample of `key`."""
    part, scale = _stored_part(case, key, x)
    return grad_close(part, case[key], rtol, atol, scale)


def same_greedy_paths(a, b, tol=1e-4, min_frac=0.5):
    """Two greedy decodes a, b [B,T,V] (logits or probabilities) of the same model by two numerically different routes.
    Greedy feedback amplifies rounding: once a near-tie flips, the trajectories legitimately diverge (and with
    probabilities the argmax of the output need not even be the token that was fed back when the top two round to the
    same value).  So a step counts as certainly-identical only if both outputs name the same token AND its top-2 margin
    exceeds 2*tol of the score scale; wherever all earlier steps are certainly-identical the scores must agree within
    ``tol`` of the scale, any disagreement there must be a near-tie, and most trajectories must stay identical."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    ta, tb = a.argmax(-1), b.argmax(-1)
    same = ta == tb
    scale = a.abs().max().item()
    top2 = a.topk(2, -1).values
    margin = top2[..., 0] - top2[..., 1]
    certain = same & (margin > 2 * tol * scale)
    hist = torch.cumprod(torch.cat([torch.ones_like(certain[:, :1]), certain[:, :-1]], 1).long(), 1).bool()
    diff = (a - b).abs().amax(-1)
    if not bool((diff[hist] <= tol * scale).all()):
        return False, f"scores differ by {diff[hist].max().item() / scale:.2e} of scale with identical history"
    flips = hist & ~same
    if flips.any() and not bool((margin[flips] <= 2 * tol * scale).all()):
        return False, f"token flip at margin {margin[flips].max().item() / scale:.2e} of scale"
    frac = hist.double().mean().item()
    why = f"identical-history fraction {frac:.3f}, first flips {int(flips.sum())}"
    report(f"same_greedy_paths: {why} (B={a.shape[0]}, T={a.shape[1]}, V={a.shape[2]})")
    return frac > min_frac, why


def report(line):
    """Measured margins / fractions of the decode-parity tests: printed (pytest -s / -rP) and appended to
    gpurun_out/parity_report.txt when that directory exists, so a passing run still shows the numbers."""
    print(line)
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(d):
        try:
            with open(os.path.join(d, "parity_report.txt"), "a") as fh:
                fh.write(line + "\n")
        except OSError:
            pass
