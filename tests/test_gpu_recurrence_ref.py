"""The GRU and LSTM recurrence kernels against a float64 cell (tests/recurrence_ref.py) at every hidden size their plans
dispatch on.

Kernels and the hidden sizes that select each instantiation (confirmed against gr_plan / gr_plan_bwdc in
csrc/gru_resident.cu and pick_cluster in csrc/gru_cluster.cu):

    resident forward   KR = 0 / 12 / 24 / 36 / 48 / 60        H = 1-21 / 22-45 / 46-69 / 70-93 / 94-117 / 118-160
    resident backward  KR = 0 / 12 / 24 / 36                  H = 1-23 / 24-47 / 48-71 / 72-95
                       column-blocked C = 3 with KS = 0       H = 96 (every weight in registers)
                       column-blocked C = 4 / C = 5           H = 97-128 / 129-155
                       KR = 60                                H = 156-160
    resident refused                                          H >= 161
    cluster size 2 / 4 / 8 / refused                          H <= 167 / 168-235 / 236-328 / >= 329
    streaming GRU      forward H <= 2074, backward H <= 1452 (shared-memory checks of caphn_gru_seq_fwd / _bwd)
    streaming LSTM     forward H <= 1452, backward H <= 1816

Every output is compared on its own with rel_err = max|kernel - ref| / max|ref|: forward outputs (states, saved gates,
Hmid, cT) within FWD, gradients within BWD.  Hall[0] must keep h0, the batch-major copy Hbm must be Hall[1:] transposed and
the inference form (no saved gates, no Hbm) must write the same Hall, all bit for bit.  Batch sizes leave row tails: the
resident and streaming kernels own 4 rows per CTA, the cluster kernels 8."""
import pytest
import torch

import recurrence_ref as R
from golden_util import rel_err, report

gpu = pytest.mark.gpu

FWD, BWD = 5e-6, 2e-5          # the float32 bounds that hold at T <= 5
FWD_KEYS = ("Hall", "Hmid", "cT", "saved")

CLUSTER_TABLE = {(1, 167): 2, (168, 235): 4, (236, 328): 8, (329, 400): 0}
GRU_SEQ_FWD_MAX, GRU_SEQ_BWD_MAX = 2074, 1452
LSTM_SEQ_FWD_MAX, LSTM_SEQ_BWD_MAX = 1452, 1816
SEQ_H = (1, 3, 4, 5, 150, 200, 329, 512)
GROUP_COUNTS = (1, 8, 13)      # 8-row tiles: a 1-row tile, a full tile, a full tile plus a 5-row tail

GRU_GATES = ("r", "z", "n", "gh_n")
LSTM_GATES = ("i", "f", "g", "o", "c_prev", "tanh_c")


def _ops():
    from hypernet_image_captioning_b200 import ops
    return ops


def _seed(family, B, T, H, NL):
    return {"gru": 1, "lstm": 2, "grouped": 3}[family] * 10_000_000 + NL * 1_000_000 + H * 1000 + T * 50 + B


def bound(key):
    return FWD if key.split("[")[0].split(".")[0] in FWD_KEYS else BWD


def flat(r, gates):
    """Result dict (reference or kernel) -> one tensor per compared output: Hall[1:], each saved gate of each layer, ..."""
    out = {}
    for k, v in r.items():
        if k == "Hall":
            out[k] = v[1:]
        elif k == "saved":
            for l in range(v.shape[0]):
                for q, name in enumerate(gates):
                    out[f"saved[{l}].{name}"] = v[l, q]
        elif k in ("Hmid", "xdGI", "xdGH", "dG"):
            for l in range(v.shape[0]):
                out[f"{k}[{l}]"] = v[l]
        else:
            out[k] = v
    return out


def errors(got, ref, gates):
    g, r = flat(got, gates), flat(ref, gates)
    return {k: rel_err(g[k], r[k]) for k in g}


def compare(got, ref, gates, where, bounds=None):
    """rel_err of every output of ``got`` against ``ref``; fails listing every output over its bound."""
    errs = errors(got, ref, gates)
    bounds = bounds or {}
    bad = {k: e for k, e in errs.items() if not e < bounds.get(k, bound(k))}
    assert not bad, f"{where}: " + ", ".join(f"{k} rel err {e:.3e} (bound {bounds.get(k, bound(k)):.0e})"
                                             for k, e in sorted(bad.items()))
    return errs


def _param_grads(r):
    """The parameter gradients the backward's callers form from the kernel outputs, in float64 on the host."""
    H = r["Hall"].shape[2]
    Hprev = r["Hall"][:-1].reshape(-1, H).double()
    r["dW_hh"] = r["dGH"].double().t() @ Hprev
    r["db_hh"] = r["dGH"].double().sum(0)
    for l in range(r["xdGI"].shape[0] if "xdGI" in r else 0):
        Hin = r["Hmid"][l].reshape(-1, H).double()
        dGI, dGH = r["xdGI"][l].double(), r["xdGH"][l].double()
        r[f"x{l + 1}.dW_ih"], r[f"x{l + 1}.dW_hh"] = dGI.t() @ Hin, dGH.t() @ Hin
        r[f"x{l + 1}.db_ih"], r[f"x{l + 1}.db_hh"] = dGI.sum(0), dGH.sum(0)


def run_gru(kind, d):
    """Forward (training and inference form) + backward of one kernel family on the inputs ``d``; kernel outputs on the
    CPU in the layout of recurrence_ref.gru().  Also checks the bitwise contracts."""
    ops = _ops()
    T, B, H3 = d["GI"].shape
    H = H3 // 3
    GI = d["GI"].reshape(T * B, H3).cuda()
    W, b, h0, dH = d["W_hh"].cuda(), d["b_hh"].cuda(), d["h0"].cuda(), d["dH"].cuda()
    if kind == "seq":
        ld3, ldh = ops.round4(H3), ops.round4(H)
        ex = [tuple(t.cuda() for t in cell) for cell in d["extra"]]
        xf = [(ops.transpose_pad(Wi, ld3), ops.transpose_pad(Wh, ld3), bi, bh) for Wi, Wh, bi, bh in ex]
        xb = [(ops.copy_pad(Wi, ldh), ops.copy_pad(Wh, ldh)) for Wi, Wh, _, _ in ex]
        WhhT = ops.transpose_pad(W, ld3)
        Hall, Hbm, saved, Hmid = ops.gru_seq_fwd(GI, WhhT, b, h0, T, extra=xf)
        dGI, dGH, xdGI, xdGH, dh0 = ops.gru_seq_bwd(dH, saved, Hall, Hmid, ops.copy_pad(W, ldh), extra=xb)
        Hinf, Hbm2, sv2, Hmid2 = ops.gru_seq_fwd(GI, WhhT, b, h0, T, save=False, want_bm=False, extra=xf)
    else:
        fwd, bwd = {"resident": (ops.gru_resident_fwd, ops.gru_resident_bwd),
                    "cluster": (ops.gru_cluster_fwd, ops.gru_cluster_bwd)}[kind]
        Hall, Hbm, saved, Hmid = fwd(GI, W, b, h0, T)
        dGI, dGH, xdGI, xdGH, dh0 = bwd(dH, saved, Hall, W)
        Hinf, Hbm2, sv2, Hmid2 = fwd(GI, W, b, h0, T, save=False, want_bm=False)
    assert Hbm2 is None and sv2 is None and Hmid2 is None
    torch.cuda.synchronize()
    assert torch.equal(Hall[0].cpu(), d["h0"]), "Hall[0] no longer holds h0"
    assert torch.equal(Hbm, Hall[1:].permute(1, 0, 2)), "Hbm is not Hall[1:] transposed"
    assert torch.equal(Hinf, Hall), "the inference form computes a different Hall"
    r = {"Hall": Hall.cpu(), "saved": saved.cpu(), "dGI": dGI.cpu(), "dGH": dGH.cpu(), "dh0": dh0.cpu()}
    if Hmid is not None:
        r.update(Hmid=Hmid.cpu(), xdGI=xdGI.cpu(), xdGH=xdGH.cpu())
    _param_grads(r)
    return r


def check_gru(kind, B, T, H, NL=1, bounds=None):
    d = R.inputs(B, T, H, NL, 3, _seed("gru", B, T, H, NL))
    return compare(run_gru(kind, d), R.gru(d), GRU_GATES, f"{kind} GRU B={B} T={T} H={H} NL={NL}", bounds)


def run_lstm(d, want_c=False):
    ops = _ops()
    T, B, H4 = d["GI"].shape
    H = H4 // 4
    ld4, ldh = ops.round4(H4), ops.round4(H)
    GI = d["GI"].reshape(T * B, H4).cuda()
    W, b, h0, dH = d["W_hh"].cuda(), d["b_hh"].cuda(), d["h0"].cuda(), d["dH"].cuda()
    c0 = d["c0"].cuda() if "c0" in d else None
    ex = [tuple(t.cuda() for t in cell) for cell in d["extra"]]
    xf = [(ops.transpose_pad(Wi, ld4), ops.transpose_pad(Wh, ld4), bi, bh) for Wi, Wh, bi, bh in ex]
    xb = [(ops.copy_pad(Wi, ldh), ops.copy_pad(Wh, ldh)) for Wi, Wh, _, _ in ex]
    WhhT = ops.transpose_pad(W, ld4)
    out = ops.lstm_seq_fwd(GI, WhhT, b, h0, T, extra=xf, c0=c0, want_c=want_c)
    Hall, Hbm, saved, Hmid = out[:4]
    dG, dh0 = ops.lstm_seq_bwd(dH, saved, Hall, ops.copy_pad(W, ldh), extra=xb)
    inf = ops.lstm_seq_fwd(GI, WhhT, b, h0, T, save=False, want_bm=False, extra=xf, c0=c0, want_c=want_c)
    assert inf[1] is None and inf[2] is None and inf[3] is None
    torch.cuda.synchronize()
    assert torch.equal(Hall[0].cpu(), d["h0"]), "Hall[0] no longer holds h0"
    assert torch.equal(Hbm, Hall[1:].permute(1, 0, 2)), "Hbm is not Hall[1:] transposed"
    assert torch.equal(inf[0], Hall), "the inference form computes a different Hall"
    r = {"Hall": Hall.cpu(), "saved": saved.cpu(), "dG": dG.cpu(), "dh0": dh0.cpu()}
    if want_c:
        assert torch.equal(inf[4], out[4]), "the inference form computes a different cT"
        r["cT"] = out[4].cpu()
    if Hmid is not None:
        r["Hmid"] = Hmid.cpu()
    return r


def check_lstm(B, T, H, NL=1, c0=False, bounds=None):
    d = R.inputs(B, T, H, NL, 4, _seed("lstm", B, T, H, NL + 10 * c0), c0=c0)
    ref = R.lstm(d)
    if not c0:
        del ref["cT"]
    return compare(run_lstm(d, want_c=c0), ref, LSTM_GATES, f"LSTM B={B} T={T} H={H} NL={NL} c0={c0}", bounds)


# ----------------------------------------------------------------------------------------------------------------------
# plans (host functions of the library: no device needed)
# ----------------------------------------------------------------------------------------------------------------------
def test_resident_and_cluster_plans_cover_the_swept_hidden_sizes():
    ops = _ops()
    assert all(ops.gru_resident_ok(H) for H in range(1, 161))
    assert not ops.gru_resident_ok(161)
    for (lo, hi), cs in CLUSTER_TABLE.items():
        got = {H: ops.gru_cluster_size(H) for H in range(lo, hi + 1)}
        assert all(v == cs for v in got.values()), f"cluster sizes over H = {lo}..{hi}: {sorted(set(got.values()))}"


# ----------------------------------------------------------------------------------------------------------------------
# sweeps
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("H", range(1, 161))
def test_resident_gru_every_hidden_size(H):
    for B in (1, 5):
        for T in (1, 3):
            check_gru("resident", B, T, H)


@gpu
def test_resident_gru_refuses_161():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    H, B, T = 161, 2, 1
    GI, W, b, h0 = (torch.zeros(T * B, 3 * H).cuda(), torch.zeros(3 * H, H).cuda(), torch.zeros(3 * H).cuda(),
                    torch.zeros(B, H).cuda())
    with pytest.raises(CaphnError):
        ops.gru_resident_fwd(GI, W, b, h0, T)
    with pytest.raises(CaphnError):
        ops.gru_resident_bwd(torch.zeros(B, T, H).cuda(), torch.zeros(1, 4, T, B, H).cuda(),
                             torch.zeros(T + 1, B, H).cuda(), W)


@gpu
@pytest.mark.parametrize("H", range(1, 329))
def test_cluster_gru_every_hidden_size(H):
    for B in (1, 9):
        check_gru("cluster", B, 3, H)


@gpu
def test_cluster_gru_refuses_329():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    H, B, T = 329, 2, 1
    W = torch.zeros(3 * H, H).cuda()
    with pytest.raises(CaphnError):
        ops.gru_cluster_fwd(torch.zeros(T * B, 3 * H).cuda(), W, torch.zeros(3 * H).cuda(), torch.zeros(B, H).cuda(), T)
    with pytest.raises(CaphnError):
        ops.gru_cluster_bwd(torch.zeros(B, T, H).cuda(), torch.zeros(1, 4, T, B, H).cuda(),
                            torch.zeros(T + 1, B, H).cuda(), W)


@gpu
@pytest.mark.parametrize("H", [36, 167, 168, 235, 236, 328])
def test_grouped_cluster_gru_per_style_reference(H):
    """caphn_gru_cluster_{fwd,bwd}_grouped called as grouped.py calls them: rows sorted by style, 8-row tiles from
    GroupPlan, each style's W_hh / b_hh in its own row of one packed buffer.  Each style is compared with its own float64
    reference."""
    ops = _ops()
    from hypernet_image_captioning_b200.grouped import GroupPlan
    G, T, H3 = len(GROUP_COUNTS), 3, 3 * H
    B = sum(GROUP_COUNTS)
    groups = torch.cat([torch.full((n,), g, dtype=torch.int64) for g, n in enumerate(GROUP_COUNTS)])
    plan = GroupPlan.get(groups, G, T, torch.device("cuda"))
    styles = [R.inputs(n, T, H, 1, 3, _seed("grouped", n, T, H, g + 1)) for g, n in enumerate(GROUP_COUNTS)]
    stride = H3 * H + H3 + 1                      # odd: every style's W_hh starts at a different alignment
    pack = torch.zeros(G, stride)
    for g, d in enumerate(styles):
        pack[g, :H3 * H] = d["W_hh"].reshape(-1)
        pack[g, H3 * H:H3 * H + H3] = d["b_hh"]
    pack = pack.cuda()
    GI = torch.cat([d["GI"] for d in styles], 1).reshape(T * B, H3).cuda()
    h0 = torch.cat([d["h0"] for d in styles], 0).cuda()
    dH = torch.cat([d["dH"] for d in styles], 0).cuda()
    Hall = torch.empty(T + 1, B, H, device="cuda")
    Hall[0].copy_(h0)
    Hbm = torch.empty(B, T, H, device="cuda")
    saved = torch.empty(1, 4, T, B, H, device="cuda")
    ops._cabi.call("caphn_gru_cluster_fwd_grouped", GI.data_ptr(), pack.data_ptr(), pack.data_ptr() + 4 * H3 * H,
                   Hall.data_ptr(), Hbm.data_ptr(), saved.data_ptr(), B, T, H, plan.tiles8.data_ptr(),
                   plan.tiles8.shape[0], stride, stride, ops._stream())
    dGI = torch.empty(T * B, H3, device="cuda")
    dGH = torch.empty(T * B, H3, device="cuda")
    dh0 = torch.empty(B, H, device="cuda")
    ops._cabi.call("caphn_gru_cluster_bwd_grouped", dH.data_ptr(), saved.data_ptr(), Hall.data_ptr(), pack.data_ptr(),
                   dGI.data_ptr(), dGH.data_ptr(), dh0.data_ptr(), B, T, H, plan.tiles8.data_ptr(),
                   plan.tiles8.shape[0], stride, ops._stream())
    torch.cuda.synchronize()
    assert torch.equal(Hall[0], h0) and torch.equal(Hbm, Hall[1:].permute(1, 0, 2))
    Hall, saved, dGI, dGH, dh0 = Hall.cpu(), saved.cpu(), dGI.cpu().view(T, B, H3), dGH.cpu().view(T, B, H3), dh0.cpu()
    r0 = 0
    for g, d in enumerate(styles):
        rows = slice(r0, r0 + GROUP_COUNTS[g])
        got = {"Hall": Hall[:, rows], "saved": saved[:, :, :, rows], "dGI": dGI[:, rows].reshape(-1, H3),
               "dGH": dGH[:, rows].reshape(-1, H3), "dh0": dh0[rows]}
        _param_grads(got)
        compare(got, R.gru(d), GRU_GATES, f"grouped cluster GRU H={H} style {g} ({GROUP_COUNTS[g]} rows)")
        r0 += GROUP_COUNTS[g]


@gpu
@pytest.mark.parametrize("H", SEQ_H + (GRU_SEQ_BWD_MAX,))
@pytest.mark.parametrize("NL", [1, 2, 3, 4])
def test_streaming_gru(NL, H):
    for B in (1, 5):
        check_gru("seq", B, 3, H, NL)


@gpu
@pytest.mark.parametrize("NL", [1, 4])
def test_streaming_gru_forward_at_its_largest_hidden_size(NL):
    """H = 2074 passes the forward's shared-memory check only (the per-step decode fallback runs the forward alone)."""
    ops = _ops()
    B, T, H = 5, 3, GRU_SEQ_FWD_MAX
    d = R.inputs(B, T, H, NL, 3, _seed("gru", B, T, H, NL))
    ref = R.gru(d)
    ld3 = ops.round4(3 * H)
    xf = [(ops.transpose_pad(Wi.cuda(), ld3), ops.transpose_pad(Wh.cuda(), ld3), bi.cuda(), bh.cuda())
          for Wi, Wh, bi, bh in d["extra"]]
    Hall, Hbm, saved, Hmid = ops.gru_seq_fwd(d["GI"].reshape(T * B, 3 * H).cuda(), ops.transpose_pad(d["W_hh"].cuda(), ld3),
                                             d["b_hh"].cuda(), d["h0"].cuda(), T, extra=xf)
    assert torch.equal(Hbm, Hall[1:].permute(1, 0, 2))
    got = {"Hall": Hall.cpu(), "saved": saved.cpu()}
    want = {"Hall": ref["Hall"], "saved": ref["saved"]}
    if NL > 1:
        got["Hmid"], want["Hmid"] = Hmid.cpu(), ref["Hmid"]
    compare(got, want, GRU_GATES, f"streaming GRU forward H={H} NL={NL}")


@gpu
def test_streaming_gru_refuses_one_above_its_largest_hidden_size():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    B, T = 1, 1
    H = GRU_SEQ_FWD_MAX + 1
    with pytest.raises(CaphnError):
        ops.gru_seq_fwd(torch.zeros(T * B, 3 * H).cuda(), torch.zeros(H, ops.round4(3 * H)).cuda(),
                        torch.zeros(3 * H).cuda(), torch.zeros(B, H).cuda(), T)
    H = GRU_SEQ_BWD_MAX + 1
    with pytest.raises(CaphnError):
        ops.gru_seq_bwd(torch.zeros(B, T, H).cuda(), torch.zeros(1, 4, T, B, H).cuda(), torch.zeros(T + 1, B, H).cuda(),
                        None, torch.zeros(3 * H, ops.round4(H)).cuda())


@gpu
@pytest.mark.parametrize("H", SEQ_H + (LSTM_SEQ_FWD_MAX,))
@pytest.mark.parametrize("NL", [1, 2, 3, 4])
def test_streaming_lstm(NL, H):
    for B in (1, 5):
        check_lstm(B, 3, H, NL)


@gpu
@pytest.mark.parametrize("H", [1, 5, 150, 512])
def test_streaming_lstm_one_step_with_cell_state(H):
    """T = 1 with a non-zero c0 and want_c: the per-step call of DecoderRNN.infer (modules.py), also in its inference
    form (save=False, want_bm=False), which must return the same h and cT bit for bit."""
    for B in (1, 5):
        check_lstm(B, 1, H, 1, c0=True)
    check_lstm(5, 3, H, 2, c0=True)


@gpu
def test_streaming_lstm_backward_at_its_largest_hidden_size():
    """H = 1816 passes the backward's shared-memory check but not the forward's: the backward runs on the reference's
    saved gates (rounded to float32)."""
    ops = _ops()
    B, T, H = 5, 3, LSTM_SEQ_BWD_MAX
    d = R.inputs(B, T, H, 1, 4, _seed("lstm", B, T, H, 1))
    ref = R.lstm(d)
    dG, dh0 = ops.lstm_seq_bwd(d["dH"].cuda(), ref["saved"].float().cuda(), ref["Hall"].float().cuda(),
                               ops.copy_pad(d["W_hh"].cuda(), ops.round4(H)))
    compare({"dG": dG.cpu(), "dh0": dh0.cpu()}, {"dG": ref["dG"], "dh0": ref["dh0"]}, LSTM_GATES,
            f"streaming LSTM backward H={H}")


@gpu
def test_streaming_lstm_refuses_one_above_its_largest_hidden_size():
    ops = _ops()
    from hypernet_image_captioning_b200._cabi import CaphnError
    B, T = 1, 1
    H = LSTM_SEQ_FWD_MAX + 1
    with pytest.raises(CaphnError):
        ops.lstm_seq_fwd(torch.zeros(T * B, 4 * H).cuda(), torch.zeros(H, ops.round4(4 * H)).cuda(),
                         torch.zeros(4 * H).cuda(), torch.zeros(B, H).cuda(), T)
    H = LSTM_SEQ_BWD_MAX + 1
    with pytest.raises(CaphnError):
        ops.lstm_seq_bwd(torch.zeros(B, T, H).cuda(), torch.zeros(1, 6, T, B, H).cuda(), torch.zeros(T + 1, B, H).cuda(),
                         torch.zeros(4 * H, ops.round4(H)).cuda())


# ----------------------------------------------------------------------------------------------------------------------
# drift at the benchmark's batch and hidden size, 64 steps
# ----------------------------------------------------------------------------------------------------------------------
DRIFT_BOUNDS = {"Hall": 8e-7, "saved[0].r": 6e-7, "saved[0].z": 6e-7, "saved[0].n": 1.3e-6, "saved[0].gh_n": 1e-6,
                "dGI": 6e-7, "dGH": 6e-7, "dh0": 5e-7, "dW_hh": 4e-7, "db_hh": 4e-7}


@gpu
@pytest.mark.parametrize("kind", ["resident", "seq"])
def test_drift_at_64_steps(kind):
    """H = 150, B = 512, T = 64: the benchmark's batch and hidden size over a long caption.

    rel_err measured on one NVIDIA B200 (1000 W power limit), resident / streaming kernel:
        Hall 2.18e-7 / 2.02e-7, r 1.54e-7 / 1.39e-7, z 1.53e-7 / 1.36e-7, n 3.38e-7 / 2.77e-7, gh_n 2.75e-7 / 1.98e-7,
        dGI 1.64e-7 / 1.66e-7, dGH 1.72e-7 / 1.57e-7, dh0 1.36e-7 / 1.34e-7, dW_hh 1.11e-7 / 1.04e-7,
        db_hh 1.04e-7 / 9.8e-8.
    Each bound in DRIFT_BOUNDS is at most 4x the larger of the two.  Relative to max|ref| the float32 error does not grow
    over 64 steps: it stays below the T <= 5 bounds of the sweeps."""
    B, T, H = 512, 64, 150
    d = R.inputs(B, T, H, 1, 3, _seed("gru", B, T, H, 1))
    errs = compare(run_gru(kind, d), R.gru(d), GRU_GATES, f"{kind} GRU B={B} T={T} H={H}", DRIFT_BOUNDS)
    report(f"drift {kind} GRU B={B} T={T} H={H}: " + ", ".join(f"{k} {e:.3e}" for k, e in errs.items()))
    assert set(errs) == set(DRIFT_BOUNDS)


# ----------------------------------------------------------------------------------------------------------------------
# the tolerances discriminate (CPU only)
# ----------------------------------------------------------------------------------------------------------------------
def _worst_ratio(mut, ref, gates, bounds=None):
    bounds = bounds or {}
    return max(e / bounds.get(k, bound(k)) for k, e in errors(mut, ref, gates).items())


@pytest.mark.parametrize("mutant", R.GRU_MUTANTS + tuple("lstm: " + m for m in R.LSTM_MUTANTS))
def test_tolerances_catch_planted_defects(mutant):
    """Each defect planted in the float64 reference moves at least one compared output by more than 10x its bound, on
    inputs of the sweeps above (same shapes, same seeds)."""
    if mutant.startswith("lstm: "):
        m = mutant[len("lstm: "):]
        NLs = (2, 3, 4) if m == "extra layer fed the step input" else (1, 2)
        cases = [(B, 3, H, NL) for H in (1, 5, 150) for NL in NLs for B in (1, 5)]
        for B, T, H, NL in cases:
            d = R.inputs(B, T, H, NL, 4, _seed("lstm", B, T, H, NL))
            ref = R.lstm(d)
            ratio = _worst_ratio(R.lstm(d, m), ref, LSTM_GATES)
            assert ratio > 10, f"{m}: B={B} T={T} H={H} NL={NL} moves the outputs by only {ratio:.1f}x the bound"
        return
    if mutant == "extra layer fed the step input":
        cases = [(B, 3, H, NL) for H in (1, 5, 150) for NL in (2, 3, 4) for B in (1, 5)]
    else:
        cases = [(B, T, H, 1) for H in (1, 24, 36, 96, 160) for B in (1, 5) for T in (1, 3)]
        cases += [(B, 3, H, 1) for H in (167, 236, 328) for B in (1, 9)] + [(5, 3, 150, 2)]
    for B, T, H, NL in cases:
        d = R.inputs(B, T, H, NL, 3, _seed("gru", B, T, H, NL))
        ratio = _worst_ratio(R.gru(d, mutant), R.gru(d), GRU_GATES)
        assert ratio > 10, f"{mutant}: B={B} T={T} H={H} NL={NL} moves the outputs by only {ratio:.1f}x the bound"
