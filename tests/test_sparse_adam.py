"""Update mode 4 on the CPU: the oracle's update rules and the host's per-step scalars pinned on torch and CPython, and the
oracle's trajectories against the torch harness stepped by torch.optim.SparseAdam (tables) and torch.optim.Adam (bias):
every loss, both tables, the bias, both moments and the step counters, bit for bit."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from _util import GOLDEN, synth
from sparse_adam_ref import OracleSparseAdam, TorchSparseAdam, scalars, vec_adam, vec_sparse_adam
from test_adagrad import CASE_NAMES, _case
from traj_common import digest, init_tables

avx512 = pytest.mark.skipif(torch.backends.cpu.get_cpu_capability() != "AVX512",
                            reason="the oracle restates torch's AVX-512 dispatch")
BETAS, EPS = (0.9, 0.999), 1e-8
STEPS = list(range(1, 11)) + [100, 1000, 10_000, 1_000_000]


@pytest.fixture(autouse=True)
def _one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _grads(n, rng):
    """gradients from 1e-30 to 1e15 in magnitude, both signs, exact zeros and -0"""
    g = rng.standard_normal(n) * 10.0 ** rng.uniform(-30, 15, n)
    g[rng.uniform(size=n) < 0.1] = 0.0
    g[rng.uniform(size=n) < 0.05] = -0.0
    if n >= 7:
        g[5], g[6] = 0.0, -0.0      # hit coordinates without gradient whose moments are not zero
    return g.astype(np.float32)


def _state(n, rng):
    m = (rng.standard_normal(n) * 10.0 ** rng.uniform(-20, 3, n)).astype(np.float32)
    v = (np.abs(rng.standard_normal(n)) * 10.0 ** rng.uniform(-30, 6, n)).astype(np.float32)
    m[:5] = 0.0
    v[:5] = 0.0
    return m, v


# ------------------------------------------------------------------------------------------------ the per-step scalars
@pytest.mark.parametrize("lr", [1e-3, 0.01, 0.05])
def test_host_scalars_are_cpythons(lr):
    """fmb_adam_scalars (the library) and the oracle's: CPython's double expressions of sparse_adam and
    _single_tensor_adam, rounded to float"""
    import fm_for_online_recommendation_b200._lib as L
    lib = L.load()
    lr32 = float(np.float32(lr))
    out = (C.c_float * 3)()
    for t in STEPS + [2 ** 31 + 5]:
        b1, b2 = BETAS
        want = np.array([-(lr32 * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)), -(lr32 / (1 - b1 ** t)), (1 - b2 ** float(t)) ** 0.5],
                        np.float32)
        lib.fmb_adam_scalars(lr32, b1, b2, t, out)
        assert np.array_equal(_bits(np.array(out, np.float32)), _bits(want)), t
        assert np.array_equal(_bits(scalars(lr32, t)), _bits(want)), t


# ------------------------------------------------------------------------------------------------ the update rules
@avx512
@pytest.mark.parametrize("t", STEPS)
@pytest.mark.parametrize("n", [7, 4099])
def test_sparse_adam_rule_is_torch(n, t):
    """orc_sparse_adam_update against torch.optim.SparseAdam at step t (state seeded with moments of every size), every
    row hit, zero gradients included: those rows step too"""
    rng = np.random.RandomState(n * 31 + t % 1000)
    p0 = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 3, n)).astype(np.float32)
    m0, v0 = _state(n, rng)
    g = _grads(n, rng)
    tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    lr = float(np.float32(0.01))
    opt = torch.optim.SparseAdam([tp], lr=lr, betas=BETAS, eps=EPS)
    opt.state[tp] = {"step": t - 1, "exp_avg": torch.from_numpy(m0.copy()), "exp_avg_sq": torch.from_numpy(v0.copy())}
    tp.grad = torch.sparse_coo_tensor(torch.arange(n)[None], torch.from_numpy(g.copy()), (n,))
    opt.step()
    p, m, v = p0.copy(), m0.copy(), v0.copy()
    vec_sparse_adam(p, g, m, v, scalars(lr, t)[0])
    st = opt.state[tp]
    assert np.array_equal(_bits(m), _bits(st["exp_avg"].numpy())), "m"
    assert np.array_equal(_bits(v), _bits(st["exp_avg_sq"].numpy())), "v"
    assert np.array_equal(_bits(p), _bits(tp.detach().numpy())), ("p", int((p != tp.detach().numpy()).sum()))
    assert m[5] != m0[5] and m[6] != m0[6]   # a hit coordinate without gradient still steps: its moments decay


@avx512
@pytest.mark.parametrize("t", STEPS)
@pytest.mark.parametrize("n", [1, 7, 4099])
def test_adam_rule_is_torch(n, t):
    """orc_adam_update against torch.optim.Adam (foreach=False: _single_tensor_adam) at step t; n = 1 is the bias"""
    rng = np.random.RandomState(n * 17 + t % 1000)
    p0 = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 3, n)).astype(np.float32)
    m0, v0 = _state(n, rng)
    g = _grads(n, rng)
    tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    lr = float(np.float32(0.01))
    opt = torch.optim.Adam([tp], lr=lr, betas=BETAS, eps=EPS, foreach=False)
    opt.state[tp] = {"step": torch.tensor(float(t - 1)), "exp_avg": torch.from_numpy(m0.copy()),
                     "exp_avg_sq": torch.from_numpy(v0.copy())}
    tp.grad = torch.from_numpy(g.copy())
    opt.step()
    p, m, v = p0.copy(), m0.copy(), v0.copy()
    s = scalars(lr, t)
    vec_adam(p, g, m, v, s[1], s[2])
    st = opt.state[tp]
    assert np.array_equal(_bits(m), _bits(st["exp_avg"].numpy())), "m"
    assert np.array_equal(_bits(v), _bits(st["exp_avg_sq"].numpy())), "v"
    assert np.array_equal(_bits(p), _bits(tp.detach().numpy())), ("p", int((p != tp.detach().numpy()).sum()))


# ------------------------------------------------------------------------------------------------ oracle vs torch
def _pair(kind, sizes, L, H, lr, cfg, bias):
    from oracle.deep import OracleDeep
    orc = OracleDeep(kind, sizes, 10, L, H, lr=lr)
    orc.w1[:], orc.V[:] = init_tables(cfg)
    orc.bias[:] = bias
    return OracleSparseAdam(orc), TorchSparseAdam(sizes, *init_tables(cfg), bias, lr)


def _assert_same(sa, h, what):
    V, w1, bias = h.m.tables()
    o = sa.o
    assert digest(o.V, o.w1, o.bias.reshape(1)) == digest(V, w1, bias), (what, int((o.V != V).sum()))
    assert np.array_equal(_bits(o.bias), _bits(bias)), what
    mV, vV, mw1, vw1, mb, vb = h.moments()
    for got, want, name in ((sa.mV, mV, "mV"), (sa.vV, vV, "vV"), (sa.mw1, mw1, "mw1"), (sa.vw1, vw1, "vw1"),
                            (sa.mbias, mb, "m bias"), (sa.vbias, vb, "v bias")):
        assert np.array_equal(_bits(got), _bits(want)), (what, name, int((got != want).sum()))
    steps, bias_steps = h.counters()
    assert steps == {sa.step} and bias_steps == sa.step, (what, steps, bias_steps, sa.step)


@avx512
@pytest.mark.parametrize("name", CASE_NAMES)
def test_oracle_update_embedding_is_torch_sparse_adam(name):
    g = dict(np.load(GOLDEN + "/traj_sgd.npz"))
    kind, sizes, B, zipf, L, H, lr, cfg = _case(name)
    sa, h = _pair(kind, sizes, L, H, lr, cfg, g[name + "_init_bias"][0])
    for s in range(120):
        Xi, Xv, Y = synth(sizes, B, 9000 + s, real_xv=name.endswith("_xv"), zipf=zipf)
        want = h.step(Xi, Xv, Y, kind == "NFMAdam")
        got = np.float32(sa.update_embedding(Xi, Xv, Y))
        assert _bits(got) == _bits(want), (s, got, want)
        if s + 1 in (1, 2, 10, 120):
            _assert_same(sa, h, s + 1)
    assert sa.mlp_step == 0


@avx512
def test_oracle_fm_fit_interleaved_with_update_embedding_is_torch():
    """FMAdam.fit (loss on sigmoid(z)) and update_embedding (loss on z) interleaved: both step the tables and the bias,
    which share one counter"""
    kind, sizes, B, zipf, L, H, lr, cfg = _case("frappe_zipf")
    sa, h = _pair("FMAdam", sizes, 0, 0, lr, cfg, 0.3)
    for s in range(60):
        Xi, Xv, Y = synth(sizes, 250, 11000 + s, zipf=True, real_xv=(s % 2 == 1))
        if s % 3 == 2:
            h.step(Xi, Xv, Y, False)
            sa.update_embedding(Xi, Xv, Y)
        else:
            h.step(Xi, Xv, Y, True)
            sa.fit(Xi, Xv, Y)
        if s + 1 in (1, 3, 60):
            _assert_same(sa, h, s + 1)
    assert sa.step == 60


@avx512
def test_oracle_fm_run_experiment_is_torch():
    """FMAdam.run_experiment over 200 examples: predict sigmoid(z) > 0.5, then fit on the one example"""
    kind, sizes, B, zipf, L, H, lr, cfg = _case("cfg1")
    sa, h = _pair("FMAdam", sizes, 0, 0, lr, cfg, 0.0)
    Xi, Xv, Y = synth(sizes, 200, 12000, zipf=True)
    conf, preds = sa.run_experiment(Xi, Xv, Y)
    want = []
    for i in range(200):
        with torch.no_grad():
            want.append(bool(torch.sigmoid(h.m.forward_fm(Xi[i:i + 1], Xv[i:i + 1]))[0] > 0.5))
        h.step(Xi[i:i + 1], Xv[i:i + 1], Y[i:i + 1], True)
    assert np.array_equal(preds, np.asarray(want))
    assert sum(conf.values()) == 200
    _assert_same(sa, h, "end")


@pytest.mark.parametrize("kind,L,H", [("DeepFMAdam", 2, 8), ("NFMAdam", 1, 12)])
def test_oracle_two_counters(kind, L, H):
    """update_embedding leaves the tower without a gradient: its counter and moments stay; fit steps both counters, and
    the tower's moments follow torch.optim.Adam's rule at the tower's own step"""
    from oracle.deep import OracleDeep
    sizes = [30, 50, 7]
    orc = OracleDeep(kind, sizes, 4, L, H, lr=0.01)
    sa = OracleSparseAdam(orc)
    seq = "uufuff"
    for i, c in enumerate(seq):
        Xi, Xv, Y = synth(sizes, 16, 100 + i, zipf=True)
        mlp0, mm0 = orc.mlp.copy(), sa.mmlp.copy()
        (sa.update_embedding if c == "u" else sa.fit)(Xi, Xv, Y)
        if c == "u":
            assert np.array_equal(_bits(orc.mlp), _bits(mlp0)) and np.array_equal(_bits(sa.mmlp), _bits(mm0))
    assert sa.step == len(seq) and sa.mlp_step == seq.count("f")


@avx512
def test_sparse_true_pipeline_matches_on_batches_without_repeated_rows():
    """nn.Embedding(sparse=True) + SparseAdam coalesces the gradient, and CPU coalesce sums a row's repeated entries in the
    order of an unstable sort.  On batches that hit no row twice there is nothing to sum, and that pipeline equals the
    target (dense gradient of the hit rows) bit for bit"""
    rng = np.random.RandomState(3)
    sizes, B, k, lr = [400, 300, 500], 64, 6, 0.01
    w1 = rng.standard_normal(sum(sizes)).astype(np.float32) * 0.1
    V = rng.standard_normal((sum(sizes), k)).astype(np.float32) * 0.1
    h = TorchSparseAdam(sizes, w1, V, 0.1, lr)
    sp = TorchSparseAdam(sizes, w1, V, 0.1, lr)
    for mods in (sp.m.first_order_embeddings, sp.m.second_order_embeddings):
        for e in mods:
            e.sparse = True
    for s in range(10):
        Xi = np.stack([rng.permutation(n)[:B] for n in sizes], 1)      # no row twice within a field
        Xv = rng.uniform(0.5, 1.5, Xi.shape).astype(np.float32)
        Y = rng.randint(0, 2, B).astype(np.float32)
        h.step(Xi, Xv, Y, False)
        sp.opt_e.zero_grad()
        sp.opt_d.zero_grad()
        z = sp.m.forward_fm(Xi, Xv)
        torch.nn.functional.binary_cross_entropy_with_logits(z, torch.from_numpy(Y)).backward()
        assert all(e.weight.grad.is_sparse for e in sp.m.second_order_embeddings)
        sp.opt_e.step()
        sp.opt_d.step()
    for a, b in zip(h.m.tables(), sp.m.tables()):
        assert np.array_equal(_bits(a), _bits(b))
