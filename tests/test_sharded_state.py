"""Update modes 3 (Adagrad) and 4 (SparseAdam) of the row-sharded step on the CPU: the reference the GPU tests use.

The sharded step folds each sample's forward sums owner by owner (OracleDeep.set_shard_order); its backward sums a row's
entries in global sample order, as the oracle does.  With two fields the owner fold is the reference's own order, so the
oracle in sharded order must step exactly like one torch.optim.Adagrad, or SparseAdam + Adam, for any number of ranks:
every loss, the tables, the bias, the sums or moments, and the step counters.  With more fields the order is really in
effect: more than one rank gives another trajectory than one."""
import numpy as np
import pytest
import torch

from _util import synth
from adagrad_ref import OracleAdagrad, TorchFM, adagrad
from sparse_adam_ref import OracleSparseAdam, TorchSparseAdam
from test_sharded import K, SIZES

avx512 = pytest.mark.skipif(torch.backends.cpu.get_cpu_capability() != "AVX512",
                            reason="the oracle restates torch's AVX-512 dispatch")

SIZES2 = [37, 300]     # F = 2: the owner fold is the reference order
ADA_HP = {2: (1e-10, 0.0), 8: (1e-6, 0.1)}   # (eps, initial_accumulator_value) per G


@pytest.fixture(autouse=True)
def _one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def oracle_in_shard_order(mode, sizes, k, G, lr, seed=0, eps=1e-10, init=0.0):
    """(update-mode oracle on an OracleDeep in G-way sharded order, its initial (V, w1, bias))"""
    from oracle.deep import OracleDeep
    orc = OracleDeep("FMAdam", sizes, k, lr=lr, seed=seed)
    orc.V *= np.float32(0.3)
    init_params = (orc.V.copy(), orc.w1.copy(), orc.bias.copy())
    orc.set_shard_order(G)
    st = OracleAdagrad(orc, eps=eps, init=init) if mode == 3 else OracleSparseAdam(orc)
    return st, init_params


def state_arrays(st):
    """the oracle's state in the order of ShardedFM.local_state(), over the full tables"""
    if isinstance(st, OracleAdagrad):
        return st.sV, st.sw1, st.sbias
    return st.mV, st.vV, st.mw1, st.vw1, st.mbias, st.vbias


def batches(sizes, n, steps, seed0):
    """uniform ids on even steps, Zipf ids on odd ones"""
    return [synth(sizes, n, seed0 + s, zipf=(s % 2 == 1)) for s in range(steps)]


@avx512
@pytest.mark.parametrize("G", [2, 8])
@pytest.mark.parametrize("mode", [3, 4])
def test_two_field_shard_order_is_torch(mode, G):
    lr, B, steps = 0.05, 24 * G, 60
    eps, init = ADA_HP[G]
    st, (V0, w0, b0) = oracle_in_shard_order(mode, SIZES2, 5, G, lr, seed=G, eps=eps, init=init)
    if mode == 3:
        m = TorchFM(SIZES2, w0, V0, b0[0])
        opt = adagrad(m, lr, eps, init)
        step = lambda Xi, Xv, Y: m.step(opt, Xi, Xv, Y, False)
    else:
        h = TorchSparseAdam(SIZES2, w0, V0, b0[0], lr)
        m = h.m
        step = lambda Xi, Xv, Y: h.step(Xi, Xv, Y, False)
    for s, (Xi, Xv, Y) in enumerate(batches(SIZES2, B, steps, 300 + G)):
        want = step(Xi, Xv, Y)
        got = np.float32(st.update_embedding(Xi, Xv, Y))
        assert _bits(got) == _bits(want), (s, got, want)
    V, w1, bias = m.tables()
    o = st.o
    for got, want, name in ((o.V, V, "V"), (o.w1, w1, "w1"), (o.bias, bias, "bias")):
        assert np.array_equal(_bits(got), _bits(want)), (name, int((got != want).sum()))
    if mode == 3:
        ref = m.adagrad_sums(opt)
    else:
        ref = h.moments()
        steps_e, steps_b = h.counters()
        assert steps_e == {st.step} and steps_b == st.step == steps
    for got, want in zip(state_arrays(st), ref):
        assert np.array_equal(_bits(got), _bits(want)), int((got != want).sum())


@pytest.mark.parametrize("mode", [3, 4])
def test_more_fields_make_the_shard_order_matter(mode):
    """premise of the GPU tests at test_sharded.SIZES: G > 1 is not the G = 1 trajectory"""
    out = []
    for G in (1, 8):
        st, _ = oracle_in_shard_order(mode, SIZES, K, G, 0.01)
        losses = [st.update_embedding(Xi, Xv, Y) for Xi, Xv, Y in batches(SIZES, 64, 6, 50)]
        out.append((np.float32(losses), st.o.V.copy()))
    assert not np.array_equal(out[0][1], out[1][1])
