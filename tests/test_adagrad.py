"""Update mode 3 (torch.optim.Adagrad) on the CPU: the oracle's update rule pinned on torch, a torch harness pinned on the
live reference's SGD trajectories, and the oracle's Adagrad trajectories against that harness stepped by
torch.optim.Adagrad.

Adagrad keeps a sum per coordinate and leaves a coordinate whose gradient is zero exactly as it is, so the oracle (and the
CUDA step), which update only the rows a batch hits, must reproduce ONE torch.optim.Adagrad over the dense tables bit for
bit: every loss, the whole table, the bias and the sums."""
import numpy as np
import pytest
import torch

from _util import GOLDEN, synth
from adagrad_ref import OracleAdagrad, TorchFM, adagrad, vec_adagrad
from traj_common import digest, init_tables

avx512 = pytest.mark.skipif(torch.backends.cpu.get_cpu_capability() != "AVX512",
                            reason="the oracle restates torch's AVX-512 dispatch")

CASE_NAMES = ["cfg1", "frappe_zipf", "deepfm_fm_part", "nfm_loss_of_sigmoid", "frappe_zipf_xv"]
CKPT = (1, 100, 300)


@pytest.fixture(autouse=True)
def _one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


# ------------------------------------------------------------------------------------------------ the update rule
def _grads(n, step, rng):
    """gradients of every magnitude from 1e-30 to 1e15, both signs, exact zeros (and -0) sprinkled in"""
    g = rng.standard_normal(n) * 10.0 ** rng.uniform(-30, 15, n)
    g[rng.uniform(size=n) < 0.1] = 0.0
    g[rng.uniform(size=n) < 0.05] = -0.0
    if step % 5 == 4:
        g[:] = 0.0            # a whole step without gradient
    return g.astype(np.float32)


@avx512
@pytest.mark.parametrize("init", [0.0, 0.1])
@pytest.mark.parametrize("eps", [1e-10, 1e-6])
@pytest.mark.parametrize("lr", [1e-3, 0.05])
@pytest.mark.parametrize("n", [7, 4096, 4099])
def test_oracle_update_rule_is_torch_adagrad(n, lr, eps, init):
    """orc_adagrad_update against torch.optim.Adagrad (foreach=False: _single_tensor_adagrad) over 20 steps with state
    kept: n covers torch's vector body and its tail; p = +-0 and s = 0 on the first step are in the inputs"""
    rng = np.random.RandomState(n + int(lr * 1e4) + int(eps * 1e12) + int(init * 10))
    p0 = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 3, n)).astype(np.float32)
    p0[::7] = 0.0
    p0[3::7] = -0.0
    tp = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = torch.optim.Adagrad([tp], lr=float(np.float32(lr)), eps=eps, initial_accumulator_value=init, foreach=False)
    p, s = p0.copy(), np.full(n, np.float32(init), np.float32)
    for step in range(20):
        g = _grads(n, step, rng)
        tp.grad = torch.from_numpy(g.copy())
        opt.step()
        vec_adagrad(p, g, s, float(np.float32(lr)), float(np.float32(eps)))
        assert np.array_equal(_bits(s), _bits(opt.state[tp]["sum"].numpy())), (step, "sum")
        assert np.array_equal(_bits(p), _bits(tp.detach().numpy())), (step, "param", int((p != tp.detach().numpy()).sum()))


# ------------------------------------------------------------------------------------------------ the torch harness
def _case(name):
    from golden.make_trajectory_sgd import CASES, cfg_of
    kind, sizes, B, zipf, (L, H), lr, steps = CASES[name]
    return kind, sizes, B, zipf, L, H, lr, cfg_of(name)


@pytest.mark.parametrize("name", CASE_NAMES)
def test_torch_harness_reproduces_the_reference_sgd_trajectories(name):
    """The harness (per-field nn.Embedding, the reference's forward_fm, BCE-with-logits, autograd) with torch.optim.SGD
    gives the live reference's losses and whole-table digests (tests/golden/traj_sgd.npz): it IS the reference's step, so
    with torch.optim.Adagrad in place of SGD it is the ground truth of mode 3."""
    g = dict(np.load(GOLDEN + "/traj_sgd.npz"))
    kind, sizes, B, zipf, L, H, lr, cfg = _case(name)
    m = TorchFM(sizes, *init_tables(cfg), g[name + "_init_bias"][0])
    opt = torch.optim.SGD(m.parameters(), lr=lr)
    losses = []
    for s in range(100):
        Xi, Xv, Y = synth(sizes, B, 7000 + s, real_xv=name.endswith("_xv"), zipf=zipf)
        losses.append(m.step(opt, Xi, Xv, Y, kind == "NFMAdam"))
        if s + 1 in (1, 100):
            assert digest(*m.tables()) == str(g["%s_s%d_digest" % (name, s + 1)]), s + 1
    assert np.array_equal(np.asarray(losses, np.float32), g[name + "_losses"][:100])


# ------------------------------------------------------------------------------------------------ oracle vs torch Adagrad
def _oracle(kind, sizes, L, H, lr, cfg, bias, eps, init):
    from oracle.deep import OracleDeep
    orc = OracleDeep(kind, sizes, 10, L, H, lr=lr)
    orc.w1[:], orc.V[:] = init_tables(cfg)
    orc.bias[:] = bias
    return OracleAdagrad(orc, eps=eps, init=init)


def _assert_same(orc, ada, m, opt, what):
    V, w1, bias = m.tables()
    assert digest(orc.V, orc.w1, orc.bias.reshape(1)) == digest(V, w1, bias), (what, int((orc.V != V).sum()))
    assert np.array_equal(_bits(orc.bias), _bits(bias)), what
    sV, sw1, sb = m.adagrad_sums(opt)
    assert np.array_equal(_bits(ada.sV), _bits(sV)) and np.array_equal(_bits(ada.sw1), _bits(sw1)), (what, "sums")
    assert np.array_equal(_bits(ada.sbias), _bits(sb)), (what, "bias sum")


@avx512
@pytest.mark.parametrize("name", CASE_NAMES)
def test_oracle_update_embedding_is_torch_adagrad(name):
    g = dict(np.load(GOLDEN + "/traj_sgd.npz"))
    kind, sizes, B, zipf, L, H, lr, cfg = _case(name)
    eps, init = (1e-10, 0.0) if name != "frappe_zipf" else (1e-6, 0.1)
    bias = g[name + "_init_bias"][0]
    ada = _oracle(kind, sizes, L, H, lr, cfg, bias, eps, init)
    m = TorchFM(sizes, *init_tables(cfg), bias)
    opt = adagrad(m, lr, eps, init)
    for s in range(300):
        Xi, Xv, Y = synth(sizes, B, 9000 + s, real_xv=name.endswith("_xv"), zipf=zipf)
        want = m.step(opt, Xi, Xv, Y, kind == "NFMAdam")
        got = np.float32(ada.update_embedding(Xi, Xv, Y))
        assert _bits(got) == _bits(want), (s, got, want)
        if s + 1 in CKPT:
            _assert_same(ada.o, ada, m, opt, s + 1)


@avx512
def test_oracle_fm_fit_is_torch_adagrad():
    """FMAdam.fit: BCE-with-logits on sigmoid(z) (fm_adam.py:80), B = 250 (torch.sigmoid's scalar tail every step)"""
    kind, sizes, B, zipf, L, H, lr, cfg = _case("frappe_zipf")
    ada = _oracle("FMAdam", sizes, 0, 0, lr, cfg, 0.3, 1e-10, 0.0)
    m = TorchFM(sizes, *init_tables(cfg), 0.3)
    opt = adagrad(m, lr)
    for s in range(300):
        Xi, Xv, Y = synth(sizes, 250, 11000 + s, zipf=True, real_xv=(s % 2 == 1))
        m.step(opt, Xi, Xv, Y, True)
        ada.fit(Xi, Xv, Y)
        if s + 1 in CKPT:
            _assert_same(ada.o, ada, m, opt, s + 1)


@avx512
def test_oracle_fm_run_experiment_is_torch_adagrad():
    """FMAdam.run_experiment over 300 examples: predict sigmoid(z) > 0.5, then fit on the one example"""
    kind, sizes, B, zipf, L, H, lr, cfg = _case("cfg1")
    ada = _oracle("FMAdam", sizes, 0, 0, lr, cfg, 0.0, 1e-10, 0.0)
    m = TorchFM(sizes, *init_tables(cfg), 0.0)
    opt = adagrad(m, lr)
    Xi, Xv, Y = synth(sizes, 300, 12000, zipf=True)
    conf, preds = ada.run_experiment(Xi, Xv, Y)
    want = []
    for i in range(300):
        with torch.no_grad():
            want.append(bool(torch.sigmoid(m.forward_fm(Xi[i:i + 1], Xv[i:i + 1]))[0] > 0.5))
        m.step(opt, Xi[i:i + 1], Xv[i:i + 1], Y[i:i + 1], True)
    assert np.array_equal(preds, np.asarray(want))
    tp = int(np.sum(preds & (Y == 1)))
    assert conf["tp"] == tp and sum(conf.values()) == 300
    _assert_same(ada.o, ada, m, opt, "end")


def test_rows_no_batch_hits_keep_weights_and_sums():
    kind, sizes, B, zipf, L, H, lr, cfg = _case("frappe_zipf")
    ada = _oracle("FMAdam", sizes, 0, 0, lr, cfg, 0.1, 1e-10, 0.25)
    V0, w10 = ada.o.V.copy(), ada.o.w1.copy()
    off = ada.o.offsets
    hit = np.zeros(ada.o.R, bool)
    for s in range(20):
        Xi, Xv, Y = synth(sizes, 64, 13000 + s, zipf=True)
        ada.update_embedding(Xi, Xv, Y)
        hit[(Xi + off[:-1][None, :]).reshape(-1)] = True
    assert hit.sum() < ada.o.R // 2
    cold = ~hit
    assert np.array_equal(_bits(ada.o.V[cold]), _bits(V0[cold])) and np.array_equal(_bits(ada.o.w1[cold]), _bits(w10[cold]))
    assert (ada.sV[cold] == np.float32(0.25)).all() and (ada.sw1[cold] == np.float32(0.25)).all()
    assert (ada.sV[hit] > np.float32(0.25)).any()
