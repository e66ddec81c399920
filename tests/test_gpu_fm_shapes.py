"""The sparse FM step at every embedding size, field count and run length its kernels accept.

fm_step.cu, fm_backward.cu and online.cu take any k <= 124 and F < 512, and their geometry changes with both: the fused
kernel has a compile-time row width for k = 8..11 only, `fit` takes the templated entry kernel up to k = 15, the run
kernel's old-row prefetch covers 32 components, the sample tile shrinks with k * F (down to one sample with the >48 KB
shared-memory opt-in), and the run kernel changes code path at run lengths 32 / 64 / 128 / 1 024 and with the run's start
modulo 4.  These tests drive each of those paths through the public classes and compare with the C oracle bit for bit
(every coordinate of every row, after every step), check every constructed batch's premise on the run list the sort
produced, compare oracle and CUDA step with an independent float64 restatement, and check that refused shapes leave the
table and the process intact.

CPU tests (no mark): the premises against numpy's stable argsort, the tile geometry, and the oracle against float64."""
import ctypes as C

import numpy as np
import pytest
import torch

from _util import synth
from test_gpu_fm import _pair, pull, push

KS = [1, 2, 3, 7, 8, 11, 12, 15, 16, 31, 32, 33, 63, 64, 65, 124]
SIZES39 = [3, 7, 50, 200] * 9 + [1, 11] + [2000]    # the last field has >= 16 B rows at B = 99: the sort's sparse-field pass
B39 = 99                                            # ragged last tile at every SB
F_SHAPES = [(1, 124, 99), (2, 124, 99), (200, 64, 40), (511, 32, 24), (120, 124, 40), (300, 124, 40)]
RUN_NS = [2, 31, 32, 33, 64, 65, 127, 128, 129, 1023, 1024, 1025, 1028, 2049, 4100]
PAD = np.float32(-7.25)                             # padding columns k+1 .. rowp-1: must never be written
EPS32 = float(np.finfo(np.float32).eps)             # 2^-23


def _sizes_f(F):
    if F == 1:
        return [40]
    if F == 2:
        return [40, 2000]
    return ([3, 7, 50, 200] * 128)[:F]


def _fused_tile(F, k):
    """(samples per tile, dynamic shared memory bytes) of fm_step_fused_kernel: the host code of fm_step.cu restated."""
    kp4, cu = (k + 3) // 4 * 4, (k + 4) // 4
    sb = max(4, min(32, 256 >> (kp4 - 1).bit_length()))
    nbytes = lambda s: 4 * (s * F * cu * 4 + 4 * s * F + s * k + s * cu * 4 + s)
    while sb > 1 and nbytes(sb) > 48 * 1024:
        sb >>= 1
    while sb > 8:
        sb >>= 1
    return sb, nbytes(sb)


# ---------------------------------------------------------------------------------------------------------------------
# constructed runs: one hot row hit exactly n times in each of three fields
#   field 1 (dense, B + 4 rows): the hot row has `above` larger ids in the batch -> the run starts at B + B - n - above
#   field 2 (16 B rows): sparse for the step's sort (only multi-hit entries are placed: the run starts at 2 B), dense for
#            the sort of `fit` (the run starts at 2 B + B - n)
#   field 4 (dense, B + 4 rows): the hot row is the field's largest id -> the run ends at the last sorted position N - 1
# the other entries of those fields are distinct ids; fields 0 and 3 are random (their own long runs ride along)
# ---------------------------------------------------------------------------------------------------------------------
def _run_sizes(B):
    return [5, B + 4, 16 * B, 3, B + 4]


def _run_B(n):
    return n + 8


def _run_batch(n, above, seed, real_xv=False):
    B = _run_B(n)
    sizes = _run_sizes(B)
    rng = np.random.RandomState(seed)
    Xi = np.stack([rng.randint(0, fs, size=B) for fs in sizes], 1).astype(np.int64)
    hot = {}
    for f, a in ((1, above), (2, 0), (4, 0)):
        h = sizes[f] - 1 - a
        others = np.concatenate([rng.choice(h, size=B - n - a, replace=False), np.arange(h + 1, sizes[f])])
        col = np.concatenate([np.full(n, h), others])
        Xi[:, f] = col[rng.permutation(B)]
        hot[f] = h
    Xv = rng.uniform(0.25, 2.0, size=Xi.shape).astype(np.float32) if real_xv else np.ones(Xi.shape, np.float32)
    Y = (rng.uniform(size=B) < 0.3).astype(np.float32)
    return Xi, Xv, Y, hot


def _intended_runs(n, above, sparse):
    """{field: (start, length)} the construction aims at"""
    B = _run_B(n)
    return {1: (2 * B - n - above, n), 2: ((2 * B, n) if sparse else (3 * B - n, n)), 4: (5 * B - n, n)}


def _numpy_runs(Xi, sizes, sparse_rows):
    """runs of >= 2 equal keys after the per-field sort, as {key: (start, length)}: numpy's stable argsort of the flat id
    matrix; fields with >= sparse_rows rows hold only their multi-hit entries, in (key, sample) order, at the head of
    the field's range (radix_sort.cu sparse_fields_kernel)"""
    B, F = Xi.shape
    off = np.concatenate([[0], np.cumsum(sizes)])
    ids = Xi + off[:-1][None, :]
    flat = ids.reshape(-1)
    sk = flat[np.argsort(flat, kind="stable")]
    for f in range(F):
        if sizes[f] >= sparse_rows:
            seg = sk[f * B:(f + 1) * B]
            u, c = np.unique(seg, return_counts=True)
            keep = seg[np.isin(seg, u[c > 1])]
            sk[f * B:(f + 1) * B] = -1
            sk[f * B:f * B + len(keep)] = keep
    out = {}
    i = 0
    while i < len(sk):
        j = i
        while j + 1 < len(sk) and sk[j + 1] == sk[i]:
            j += 1
        if sk[i] >= 0 and j > i:
            out[int(sk[i])] = (i, j - i + 1)
        i = j + 1
    return out


def _check_premise(runs, Xi, hot, n, above, sparse):
    """the hot rows' runs are where the case needs them: start, length, long-run flag (>= 128), start modulo 4"""
    B = Xi.shape[0]
    off = np.concatenate([[0], np.cumsum(_run_sizes(B))])
    want = _intended_runs(n, above, sparse)
    for f, (s, ln) in want.items():
        key = int(off[f] + hot[f])
        assert key in runs, (f, n)
        got = runs[key]
        assert got[0] == s and got[1] == ln, (f, n, above, got, (s, ln))
        if len(got) > 2:           # the run list's own fields
            assert got[2] == min(ln, 32) and got[3] == int(ln >= 128), (f, got)
    assert want[4][0] + want[4][1] == Xi.size                        # field 4's run ends at the last sorted position
    return {f: s % 4 for f, (s, _) in want.items()}


# ---------------------------------------------------------------------------------------------------------------------
# float64 restatement of one SGD step (update mode 1, loss on z_fm) and its error bound
# ---------------------------------------------------------------------------------------------------------------------
def sgd_step_fp64(V, w1, bias, ids, xv, y, lr):
    """One update_embedding step in update mode 1, in float64: z = bias + sum_f w x + 1/2 sum_j (S_j^2 - Q_j),
    d = (sigmoid(z) - y) / B, per row the sum of its entries' contributions x (d S_j - d v_j x) and d x, p - lr g.

    Returns (V', w1', bias', tolerance of V', of w1', of bias').  With every fp32 operation rounded once
    (relative error <= eps = 2^-23) the fp32 step differs from this one by at most, per coordinate,

        ulp(p') + lr * c * eps * M,    c = 2 (F + k + n_r) + 16,

    n_r the number of entries of the row, and M the sum over the row's entries of |x| * D_b * (sum_f' |e_f'j| + |e_j|)
    (component j) or |x| * D_b (w1), where e = v x and D_b = |d_b| + (Z_b / 4 + 1) / B with
    Z_b = |bias| + sum_f |w x| + sum_j (sum_f |e_fj|)^2 -- the magnitudes behind z_b.  The terms: z_b's sums
    (F + k terms, error <= (F + k + 4) eps Z_b) move d_b by at most a quarter of that over B (sigmoid' <= 1/4), the
    sigmoid and the division add a few eps / B; S_j carries <= F eps sum_f |e_fj|; each contribution's products round
    3 more times, the row's sum of n_r contributions n_r times; `fma(g, -lr, p)` rounds once (half an ulp of p')."""
    f64 = np.float64
    B, F = ids.shape
    k = V.shape[1]
    lr = f64(np.float32(lr))
    x = xv.astype(f64)
    E = V[ids].astype(f64) * x[:, :, None]                    # [B,F,k]
    S = E.sum(1)
    Q = (E * E).sum(1)
    first = w1[ids].astype(f64) * x
    z = f64(bias) + first.sum(1) + 0.5 * (S * S - Q).sum(1)
    d = (1.0 / (1.0 + np.exp(-z)) - y.astype(f64)) / B
    cV = (d[:, None, None] * (S[:, None, :] - E)) * x[:, :, None]
    cw = d[:, None] * x
    R = V.shape[0]
    flat = ids.reshape(-1)
    gV = np.zeros((R, k))
    gw = np.zeros(R)
    np.add.at(gV, flat, cV.reshape(-1, k))
    np.add.at(gw, flat, cw.reshape(-1))
    absE = np.abs(E)
    A = absE.sum(1)
    Z = abs(f64(bias)) + np.abs(first).sum(1) + (A * A).sum(1)
    D = np.abs(d) + (Z / 4 + 1) / B
    MV = np.zeros((R, k))
    Mw = np.zeros(R)
    np.add.at(MV, flat, (np.abs(x)[:, :, None] * D[:, None, None] * (A[:, None, :] + absE)).reshape(-1, k))
    np.add.at(Mw, flat, (np.abs(x) * D[:, None]).reshape(-1))
    cnt = np.bincount(flat, minlength=R).astype(f64)
    c = 2 * (F + k + cnt) + 16
    Vn = V.astype(f64) - lr * gV
    wn = w1.astype(f64) - lr * gw
    bn = f64(bias) - lr * d.sum()
    ulp = lambda a: np.spacing(np.abs(a).astype(np.float32)).astype(f64)
    tolV = ulp(Vn) + lr * c[:, None] * EPS32 * MV
    tolw = ulp(wn) + lr * c * EPS32 * Mw
    tolb = ulp(np.array(bn)) + lr * (2 * (F + k + B) + 16) * EPS32 * D.sum()
    return Vn, wn, bn, tolV, tolw, float(tolb)


def _within(got, want, tol, what):
    err = np.abs(got.astype(np.float64) - want)
    bad = err > tol
    assert not bad.any(), (what, int(bad.sum()), float((err / np.maximum(tol, 1e-300)).max()))


def _fp64_cases():
    cases = [("k", SIZES39, k, B39) for k in KS]
    cases += [("F", _sizes_f(F), k, B) for F, k, B in F_SHAPES]
    return cases


def _oracle_sgd(sizes, k, seed):
    from oracle.deep import OracleDeep
    orc = OracleDeep("FMAdam", sizes, k, lr=0.05, update_mode=1, seed=seed)
    orc.V *= np.float32(0.1)
    orc.w1 *= np.float32(0.1)
    orc.bias[:] = np.float32(0.1)
    return orc


def _fp64_vs_oracle(orc, Xi, Xv, Y):
    ids = orc.global_ids(Xi)
    want = sgd_step_fp64(orc.V.copy(), orc.w1.copy(), float(orc.bias[0]), ids, Xv, Y, 0.05)
    orc.update_embedding(Xi, Xv, Y)
    return want


def _assert_fp64(want, V, w1, bias):
    Vn, wn, bn, tolV, tolw, tolb = want
    _within(V, Vn, tolV, "V")
    _within(w1, wn, tolw, "w1")
    assert abs(float(bias) - bn) <= tolb, (float(bias), bn, tolb)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def test_tile_geometry_reaches_every_path():
    """the sweep's shapes reach 8-, 4-, 2- and 1-sample tiles, the >48 KB opt-in, and one refused tile"""
    sbs = {k: _fused_tile(39, k)[0] for k in KS}
    assert {sbs[k] for k in KS} == {8, 4, 2}
    assert sbs[31] == 8 and sbs[32] == 4 and sbs[124] == 2
    for F, k, _ in F_SHAPES[2:]:
        sb, nbytes = _fused_tile(F, k)
        assert sb == 1 and 48 * 1024 < nbytes <= 200 * 1024, (F, k, nbytes)
    assert _fused_tile(511, 124)[1] > 200 * 1024


@pytest.mark.parametrize("n", RUN_NS)
def test_constructed_runs_premise_numpy(n):
    """every constructed batch puts its hot runs where the case needs them, per numpy's stable argsort: all four start
    offsets modulo 4 in field 1, the last run ending at N - 1, the long-run flag exactly from n >= 128"""
    B = _run_B(n)
    mods = set()
    for above in range(4):
        Xi, Xv, Y, hot = _run_batch(n, above, seed=1000 * n + above)
        for sparse in (False, True):
            runs = _numpy_runs(Xi, _run_sizes(B), 16 * B if sparse else 1 << 40)
            m = _check_premise(runs, Xi, hot, n, above, sparse)
            mods.add(m[1])
    assert mods == {0, 1, 2, 3}


@pytest.mark.parametrize("kind,sizes,k,B", _fp64_cases())
def test_oracle_sgd_step_within_fp64_bound(kind, sizes, k, B):
    orc = _oracle_sgd(sizes, k, seed=k)
    for step in range(2):
        Xi, Xv, Y = synth(sizes, B, 300 + step, real_xv=(step == 1), zipf=(step == 0))
        want = _fp64_vs_oracle(orc, Xi, Xv, Y)
        _assert_fp64(want, orc.V, orc.w1, orc.bias[0])


@pytest.mark.parametrize("k", [10, 33, 124])
@pytest.mark.parametrize("n", RUN_NS)
def test_oracle_sgd_step_within_fp64_bound_on_constructed_runs(n, k):
    B = _run_B(n)
    orc = _oracle_sgd(_run_sizes(B), k, seed=n)
    for above in (0, 3):
        Xi, Xv, Y, _ = _run_batch(n, above, seed=1000 * n + above, real_xv=(above == 3))
        _assert_fp64(_fp64_vs_oracle(orc, Xi, Xv, Y), orc.V, orc.w1, orc.bias[0])


def test_fp64_bound_is_tight_enough_to_see_one_dropped_contribution():
    """the bound is not vacuous: removing one entry's contribution from a hot row's sum leaves it"""
    n = 129
    B = _run_B(n)
    orc = _oracle_sgd(_run_sizes(B), 33, seed=5)
    Xi, Xv, Y, hot = _run_batch(n, 0, seed=7)
    ids = orc.global_ids(Xi)
    Vn, wn, bn, tolV, tolw, _ = sgd_step_fp64(orc.V.copy(), orc.w1.copy(), float(orc.bias[0]), ids, Xv, Y, 0.05)
    r = int(orc.offsets[1] + hot[1])
    b = int(np.flatnonzero(Xi[:, 1] == hot[1])[-1])
    Eb = orc.V[ids[b]].astype(np.float64) * Xv[b][:, None]          # sample b's embeddings, [F,k]
    S = Eb.sum(0)
    z = float(orc.bias[0]) + (orc.w1[ids[b]] * Xv[b].astype(np.float64)).sum() + 0.5 * (S * S - (Eb * Eb).sum(0)).sum()
    d = (1 / (1 + np.exp(-z)) - Y[b]) / B
    lr = np.float64(np.float32(0.05))
    dropped = lr * d * (S - Eb[1]) * Xv[b, 1]                       # entry (b, field 1)'s share of the row's step
    assert (np.abs(dropped) > tolV[r]).mean() > 0.5, (np.abs(dropped), tolV[r])
    assert abs(lr * d * Xv[b, 1]) > tolw[r]


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _lib():
    import fm_for_online_recommendation_b200 as pkg
    return pkg.require_cuda()


def _push_padded(m, orc):
    push(m, orc)
    with torch.no_grad():
        m._table[:, orc.k + 1:] = float(PAD)


def _same(m, orc, step=None):
    """every coordinate of V, w1, bias (and the tower, alpha, FTRL state where present); padding untouched"""
    p = pull(m)
    for key in ("V", "w1", "bias"):
        a, b = p[key], getattr(orc, key)
        assert np.array_equal(a, b), (step, key, int((a != b).sum()), a.size)
    if orc.L:
        assert np.array_equal(p["mlp"], orc.mlp), (step, "mlp", int((p["mlp"] != orc.mlp).sum()))
    if hasattr(m, "alpha"):
        assert np.array_equal(p["alpha"], orc.alpha[:orc.L]), (step, "alpha")
    pad = m._table[:, orc.k + 1:]
    assert bool((pad == float(PAD)).all()), (step, "padding written", int((pad != float(PAD)).sum().item()))
    if m.update_mode == 2:
        k = orc.k
        zn = m._ftrl_zn.cpu().numpy()
        assert np.array_equal(zn[:, 0, :k], orc.fz_V) and np.array_equal(zn[:, 1, :k], orc.fn_V), (step, "ftrl V")
        assert np.array_equal(zn[:, 0, k], orc.fz_w1) and np.array_equal(zn[:, 1, k], orc.fn_w1), (step, "ftrl w1")
        assert np.array_equal(m._ftrl_bias.cpu().numpy(), orc.f_bias), (step, "ftrl bias")


def _model(kind, sizes, k, mode, L=0, H=0, lr=None, **kw):
    lr = lr if lr is not None else (0.05 if mode else 1e-3)
    m, orc = _pair(kind, sizes, k, L, H, lr=lr, scale=0.1, update_mode=min(mode, 1), **kw)
    m.update_mode = min(mode, 1)
    orc.bias[:] = np.float32(0.1)
    _push_padded(m, orc)
    if mode == 2:
        orc.enable_ftrl(1.0, 2e-3, 1e-3)
        m.enable_ftrl(1.0, 2e-3, 1e-3)
    return m, orc


def _ue_steps(m, orc, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        got = m.update_embedding(Xi, Xv, Y).item()
        want = orc.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), (i, got, want)
        _same(m, orc, i)


def _fit_steps(m, orc, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        m.fit(Xi, Xv, Y)
        orc.fit(Xi, Xv, Y)
        _same(m, orc, i)


def _sweep_batches(sizes, B, seed, n=6):
    """three all-ones steps then three real-valued ones: per value kind, the eager first call, the graph capture and a
    replay re-pointed at a new batch; Zipf ids on every other step (long runs, multi-hit rows in the sparse field)"""
    return [synth(sizes, B, seed + i, real_xv=(i >= n // 2), zipf=(i % 2 == 0)) for i in range(n)]


def _gpu_runs(m, e, sparse):
    """{key: (start, length among the first 32 positions, n0, long flag)} from the sort's run list"""
    from fm_for_online_recommendation_b200._lib import RunList
    lib = m._lib
    B, F = e.B, m.field_size
    N = B * F
    nseg, cap = C.c_int(), C.c_int()
    lib.fmb_runlist_shape(B, F, C.byref(nseg), C.byref(cap))
    nseg, cap = nseg.value, cap.value
    dev = lambda n: torch.zeros(n, dtype=torch.int32, device="cuda")
    sk, pm, pf = dev(N), dev(N), dev(N)
    rl = torch.full((nseg * cap, 4), -1, dtype=torch.int32, device="cuda")
    cnt = dev(2 * nseg)
    desc = RunList(rl.data_ptr(), cnt.data_ptr(), nseg, cap)
    p = lambda t: C.c_void_p(t.data_ptr())
    assert lib.fmb_sort_fields_ex(p(e.ids), B, F, p(m._field_off_dev), p(sk), p(pm), p(pf), C.byref(desc),
                                  1 if sparse else 0, None) == 0, lib.fmb_last_error()
    torch.cuda.synchronize()
    c, r = cnt.cpu().numpy(), rl.cpu().numpy()
    ent = [r[g * cap:g * cap + c[g]] for g in range(nseg)] + [r[(g + 1) * cap - c[nseg + g]:(g + 1) * cap] for g in range(nseg)]
    ent = np.concatenate(ent + [np.zeros((0, 4), np.int32)])
    skn = sk.cpu().numpy()
    out = {}
    for s, key, n0, lng in ent:
        ln = 1
        while s + ln < N and skn[s + ln] == key:
            ln += 1
        out[int(key)] = (int(s), ln, int(n0), int(lng))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# 1. shape sweep, bit for bit against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("k", KS)
def test_update_embedding_every_k(k, mode):
    assert _lib().fmb_sort_fields_sparse_min_rows(B39) <= SIZES39[-1]
    m, orc = _model("FMAdam", SIZES39, k, mode)
    _ue_steps(m, orc, _sweep_batches(SIZES39, B39, 10 * k))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 16), ("NFMAdam", 2, 24)])
@pytest.mark.parametrize("k", KS)
def test_fit_every_k(k, kind, L, H, mode):
    """FMAdam.fit (the step with the loss on sigmoid(z)), DeepFMAdam.fit (two gradient chains per row: nv = 2k + 1
    virtual lanes, several 32-lane passes from k = 16) and NFMAdam.fit (the tower chain alone); the SIMT tower
    (B * H * H far below the tensor-core threshold) is bit-exact too"""
    m, orc = _model(kind, SIZES39, k, mode, L, H)
    _fit_steps(m, orc, _sweep_batches(SIZES39, B39, 20 * k))


@pytest.mark.gpu
@pytest.mark.parametrize("F,k,B", F_SHAPES)
def test_field_counts(F, k, B):
    """F = 1, 2 at k = 124 and the one-sample tiles behind the >48 KB shared-memory opt-in; F = 511 makes 2 044
    run-list segments"""
    sizes = _sizes_f(F)
    for mode in (1, 0):
        m, orc = _model("FMAdam", sizes, k, mode)
        _ue_steps(m, orc, _sweep_batches(sizes, B, 40 + F))
    m, orc = _model("DeepFMAdam", sizes, k, 1, 2, 16)
    _fit_steps(m, orc, _sweep_batches(sizes, B, 50 + F))


@pytest.mark.gpu
def test_batch_above_per_field_sort_limit_k33():
    """B > 65 536: the generic radix sort, pos_flags_kernel's one-segment run list, long-run chains of ~1 000 entries"""
    sizes, k, B = [70, 9, 40000, 3000, 150000], 33, 70001
    assert B > _lib().fmb_sort_fields_max_batch()
    for mode in (1, 0):
        m, orc = _model("FMAdam", sizes, k, mode)
        _ue_steps(m, orc, [synth(sizes, B, 80 + i, real_xv=(i == 1), zipf=(i == 0)) for i in range(3)])


@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 39])
@pytest.mark.parametrize("k", [1, 33, 124])
@pytest.mark.parametrize("kind,L,H,mode", [("FMAdam", 0, 0, 1), ("DeepFMAdam", 2, 8, 1), ("NFMOnn", 3, 10, 0)])
def test_run_experiment_shapes(kind, L, H, mode, k, F):
    sizes = SIZES39 if F == 39 else [40]
    kw = dict(batch_size=1) if kind.endswith("Onn") else {}
    m, orc = _model(kind, sizes, k, mode, L, H, **kw)
    Xi, Xv, Y = synth(sizes, 60, 7 + k, real_xv=True)
    _, _, _, conf = m.run_experiment(Xi.tolist(), Xv.tolist(), [int(v) for v in Y])
    oconf, opreds = orc.run_experiment(Xi, Xv, Y)
    assert conf == oconf
    assert np.array_equal(m._last_online_preds, opreds)
    _same(m, orc)


# ---------------------------------------------------------------------------------------------------------------------
# 2. constructed run lengths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 33, 124])
@pytest.mark.parametrize("n", RUN_NS)
def test_update_embedding_run_lengths(n, k):
    """SGD steps (a value error in a run's sum cannot hide behind a sign step); four batches move field 1's run through
    every start offset modulo 4; field 2's run is placed by the sparse-field pass; field 4's run ends at N - 1"""
    B = _run_B(n)
    sizes = _run_sizes(B)
    assert _lib().fmb_sort_fields_sparse_min_rows(B) == 16 * B      # field 2 is sparse for the step's sort
    m, orc = _model("FMAdam", sizes, k, 1)
    mods = set()
    for above in range(4):
        Xi, Xv, Y, hot = _run_batch(n, above, seed=1000 * n + above, real_xv=(above % 2 == 1))
        e = m.encode(Xi, Xv, Y)
        mods.add(_check_premise(_gpu_runs(m, e, sparse=True), Xi, hot, n, above, sparse=True)[1])
        got = m.update_embedding(e, None, None).item()
        want = orc.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), (above, got, want)
        _same(m, orc, above)
    assert mods == {0, 1, 2, 3}


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16, 33])
@pytest.mark.parametrize("n", RUN_NS)
def test_deepfm_fit_run_lengths(n, k):
    """two chains per row: nv = 21, 33, 67 virtual lanes (one, two, three 32-lane passes over each run)"""
    B = _run_B(n)
    m, orc = _model("DeepFMAdam", _run_sizes(B), k, 1, 1, 8)
    mods = set()
    for above in range(4):
        Xi, Xv, Y, hot = _run_batch(n, above, seed=2000 * n + above, real_xv=(above % 2 == 1))
        e = m.encode(Xi, Xv, Y)
        mods.add(_check_premise(_gpu_runs(m, e, sparse=False), Xi, hot, n, above, sparse=False)[1])
        m.fit(e, None, None)
        orc.fit(Xi, Xv, Y)
        _same(m, orc, above)
    assert mods == {0, 1, 2, 3}


# ---------------------------------------------------------------------------------------------------------------------
# 3. the CUDA step against the float64 restatement
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["k1", "k33", "k124", "F511", "run1025"])
def test_cuda_sgd_step_within_fp64_bound(case):
    if case.startswith("run"):
        n = int(case[3:])
        sizes, k = _run_sizes(_run_B(n)), 33
        batches = [_run_batch(n, a, seed=a, real_xv=(a == 1))[:3] for a in (0, 1)]
    else:
        if case == "F511":
            sizes, k, B = _sizes_f(511), 32, 24
        else:
            sizes, k, B = SIZES39, int(case[1:]), B39
        batches = [synth(sizes, B, 300 + s, real_xv=(s == 1), zipf=(s == 0)) for s in range(2)]
    m, orc = _model("FMAdam", sizes, k, 1)
    for Xi, Xv, Y in batches:
        ids = orc.global_ids(Xi)
        p = pull(m)
        want = sgd_step_fp64(p["V"], p["w1"], float(p["bias"][0]), ids, Xv, Y, m._lr)
        m.update_embedding(Xi, Xv, Y)
        p = pull(m)
        _assert_fp64(want, p["V"], p["w1"], p["bias"][0])


# ---------------------------------------------------------------------------------------------------------------------
# 4. refusals leave nothing behind
# ---------------------------------------------------------------------------------------------------------------------
def _refused(m, call, *names):
    t0 = m._table.clone()
    b0 = m.bias.clone()
    with pytest.raises(RuntimeError) as ei:
        call()
    msg = str(ei.value)
    for s in names:
        assert s in msg, (s, msg)
    torch.cuda.synchronize()
    assert torch.equal(m._table, t0) and torch.equal(m.bias, b0)


def _still_trains():
    """a valid model in the same process still trains bit-exact: update_embedding (eager, captured, replayed; one >48 KB
    tile), DeepFM fit, run_experiment"""
    sizes = _sizes_f(200)
    m, orc = _model("FMAdam", sizes, 64, 1)
    _ue_steps(m, orc, _sweep_batches(sizes, 40, 600, n=3))
    m, orc = _model("DeepFMAdam", SIZES39, 33, 1, 2, 8)
    _fit_steps(m, orc, _sweep_batches(SIZES39, B39, 610, n=3))
    Xi, Xv, Y = synth(SIZES39, 30, 620, real_xv=True)
    _, _, _, conf = m.run_experiment(Xi, Xv, Y)
    assert conf == orc.run_experiment(Xi, Xv, Y)[0]
    _same(m, orc)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["k125", "F512", "F511k124", "online_tower"])
def test_refused_shapes_leave_table_and_process_intact(case):
    import fm_for_online_recommendation_b200 as pkg
    if case == "k125":
        sizes, k, names = [5, 9, 40], 125, ("k=125",)
    elif case == "F512":
        sizes, k, names = [3] * 512, 4, ("F=512",)
    elif case == "F511k124":
        sizes, k, names = [3] * 511, 124, ("F=511", "k=124")
    else:
        sizes, k, names = [2] * 300, 124, ("F=300", "k=124", "L=24", "H=500")
    Xi, Xv, Y = synth(sizes, 16, 1, real_xv=True)
    if case == "online_tower":
        # the step takes this shape (a one-sample tile of 156 KB); the persistent kernel's one CTA cannot hold the rows
        # and a 24 x 500 tower's activations
        m = pkg.DeepFMAdam(sizes, embedding_size=k, num_hidden_layers=24, neuron_per_hidden_layer=500, n=0.01)
        _refused(m, lambda: m.run_experiment(Xi, Xv, Y), *names)
        m.update_embedding(Xi, Xv, Y)
        torch.cuda.synchronize()
    else:
        m = pkg.FMAdam(sizes, embedding_size=k, n=0.01)
        _refused(m, lambda: m.update_embedding(Xi, Xv, Y), *names)
        _refused(m, lambda: m.fit(Xi, Xv, Y), *names)
        _refused(m, lambda: m.run_experiment(Xi, Xv, Y), *names)
    _still_trains()
