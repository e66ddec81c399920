"""Update mode 4 (torch.optim.SparseAdam on the tables, torch.optim.Adam on the bias and the tower) on the GPU, bit for bit
against the C oracle of tests/sparse_adam_oracle.c after every step: the loss, V, w1, the bias, the tower, both moments of
each and both step counters.  The padding columns of the table and of its moments hold a sentinel no kernel may write."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from _util import synth
from sparse_adam_ref import OracleSparseAdam
from test_gpu_fm import _pair
from test_gpu_fm_shapes import B39, PAD, SIZES39, _push_padded, _run_batch, _same, _sizes_f

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _model(kind, sizes, k, L=0, H=0, lr=0.05, **kw):
    m, orc = _pair(kind, sizes, k, L, H, lr=lr, scale=0.1, **kw)
    orc.bias[:] = np.float32(0.1)
    _push_padded(m, orc)
    m.enable_sparse_adam()
    with torch.no_grad():
        m._sa_mv[:, :, k + 1:] = float(PAD)
    return m, orc, OracleSparseAdam(orc)


def _same_sa(m, orc, sa, step=None):
    _same(m, orc, step)
    k = orc.k
    mv = m._sa_mv.cpu().numpy()
    for j, (tV, tw1) in enumerate(((sa.mV, sa.mw1), (sa.vV, sa.vw1))):
        assert np.array_equal(_bits(mv[:, j, :k]), _bits(tV)), (step, "mv", j, int((mv[:, j, :k] != tV).sum()))
        assert np.array_equal(_bits(mv[:, j, k]), _bits(tw1)), (step, "mv w1", j)
    assert (mv[:, :, k + 1:] == PAD).all(), (step, "padding of the moments written")
    assert np.array_equal(_bits(m._sa_bias.cpu().numpy()), _bits(np.concatenate([sa.mbias, sa.vbias]))), (step, "bias m/v")
    if orc.L and m._sa_mlp is not None:
        n = m._sa_mlp.shape[1]
        t = m._sa_mlp.cpu().numpy()
        assert np.array_equal(_bits(t[0]), _bits(sa.mmlp[:n])) and np.array_equal(_bits(t[1]), _bits(sa.vmlp[:n])), \
            (step, "tower m/v")
    assert (m._sa.step, m._sa.mlp_step) == (sa.step, sa.mlp_step), step


def _ue(m, orc, sa, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        got = m.update_embedding(Xi, Xv, Y).item()
        want = sa.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), (i, got, want)
        _same_sa(m, orc, sa, i)


def _fit(m, orc, sa, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        m.fit(Xi, Xv, Y)
        sa.fit(Xi, Xv, Y)
        _same_sa(m, orc, sa, i)


def _sweep(sizes, B, seed, n=6):
    """all-ones then real-valued steps (eager, captured, re-pointed replays), Zipf ids every other step"""
    return [synth(sizes, B, seed + i, real_xv=(i >= n // 2), zipf=(i % 2 == 0)) for i in range(n)]


@pytest.mark.parametrize("F", [1, 39])
@pytest.mark.parametrize("k", [1, 3, 10, 33, 124])
def test_update_embedding(k, F):
    sizes, B = (SIZES39, B39) if F == 39 else (_sizes_f(1), 99)
    m, orc, sa = _model("FMAdam", sizes, k)
    _ue(m, orc, sa, _sweep(sizes, B, 100 + k))


@pytest.mark.parametrize("n", [2, 129, 1025])
def test_hot_row_runs(n):
    """one row hit n times in three fields: direct part, ring, and (from 128 entries) the long-run CTAs of the run kernel"""
    Xi, Xv, Y, _ = _run_batch(n, 0, 3 + n)
    sizes = [int(v) for v in [5, Xi.shape[0] + 4, 16 * Xi.shape[0], 3, Xi.shape[0] + 4]]
    batches = [(Xi, Xv, Y)] + [_run_batch(n, 1, 50 + n + i, real_xv=(i == 1))[:3] for i in range(2)]
    m, orc, sa = _model("FMAdam", sizes, 10)
    _ue(m, orc, sa, batches)
    m2, orc2, sa2 = _model("DeepFMAdam", sizes, 10, 2, 16)
    _fit(m2, orc2, sa2, batches)


def test_next_batch_pipeline_replays_one_graph():
    """device-resident steps announcing the next batch: eager first step, capture, then re-pointed replays of ONE graph
    whose scalars change every step; a few hundred steps keep the graph count constant"""
    m, orc, sa = _model("FMAdam", SIZES39, 10, lr=0.01)
    host = [synth(SIZES39, B39, 200 + i, zipf=(i % 2 == 0)) for i in range(6)]
    enc = [m.encode(*b) for b in host]
    for i, (Xi, Xv, Y) in enumerate(host):
        got = m.update_embedding(enc[i], None, None, next_batch=enc[(i + 1) % 6]).item()
        want = sa.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), i
        _same_sa(m, orc, sa, i)
    ng = m._lib.fmb_session_graph_count(m._session)
    for i in range(300):
        j = (6 + i) % 6
        m.update_embedding(enc[j], None, None, next_batch=enc[(j + 1) % 6])
        sa.update_embedding(*host[j])
    assert m._lib.fmb_session_graph_count(m._session) == ng
    _same_sa(m, orc, sa, "after 306 steps")


@pytest.mark.parametrize("nslot", [2, 4])
def test_host_pipeline(nslot):
    """fmb_session_fm_step_host_async over nslot slots (the host submits up to nslot - 1 steps ahead, every one with its own
    scalars), then blocking host steps, against the oracle"""
    m, orc, sa = _model("FMAdam", SIZES39, 10, lr=0.01)
    lib, B = m._lib, B39
    s = m._get_session(B)
    tp, bp = C.c_void_p(m._table.data_ptr()), C.c_void_p(m.bias.data_ptr())
    loss = C.c_float()
    batches = [synth(SIZES39, B, 40 + i, zipf=(i % 2 == 0)) for i in range(10)]
    want = [sa.update_embedding(*b) for b in batches] + [sa.update_embedding(*b) for b in batches[:2]]
    got = []
    for i, (Xi, Xv, Y) in enumerate(batches):
        ids = np.ascontiguousarray((Xi + m._offsets_np[:-1][None, :]).astype(np.int32))
        y = np.ascontiguousarray(Y, np.float32)
        assert lib.fmb_session_fm_step_host_async(s, i % nslot, ids.ctypes.data_as(C.c_void_p), None,
                                                  y.ctypes.data_as(C.c_void_p), B, tp, bp, m._key_bits, 0, m._lr, 4,
                                                  None) == 0, lib.fmb_last_error()
        if i >= nslot - 1:
            assert lib.fmb_session_wait_loss(s, (i - nslot + 1) % nslot, C.byref(loss)) == 0
            got.append(loss.value)
    for i in range(len(batches) - nslot + 1, len(batches)):
        assert lib.fmb_session_wait_loss(s, i % nslot, C.byref(loss)) == 0
        got.append(loss.value)
    for Xi, Xv, Y in batches[:2]:
        ids = np.ascontiguousarray((Xi + m._offsets_np[:-1][None, :]).astype(np.int32))
        y = np.ascontiguousarray(Y, np.float32)
        assert lib.fmb_session_fm_step_host(s, ids.ctypes.data_as(C.c_void_p), None, y.ctypes.data_as(C.c_void_p), B, tp,
                                            bp, m._key_bits, 0, m._lr, 4, C.byref(loss), None) == 0, lib.fmb_last_error()
        got.append(loss.value)
    assert np.array_equal(_bits(np.array(got, np.float32)), _bits(np.array(want, np.float32)))
    _same_sa(m, orc, sa, "end")


@pytest.mark.parametrize("k", [3, 10, 33])
@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 16), ("NFMAdam", 2, 24)])
def test_fit(kind, L, H, k):
    m, orc, sa = _model(kind, SIZES39, k, L, H)
    _fit(m, orc, sa, _sweep(SIZES39, B39, 300 + k))


@pytest.mark.parametrize("kind,L,H", [("DeepFMAdam", 2, 16), ("NFMAdam", 1, 12)])
def test_interleaved_update_embedding_and_fit(kind, L, H):
    """the tables and the bias count every step, the tower only fits"""
    m, orc, sa = _model(kind, SIZES39, 10, L, H)
    for i, b in enumerate(_sweep(SIZES39, B39, 800, n=7)):
        if i % 3 == 1:
            m.fit(*b)
            sa.fit(*b)
        else:
            assert np.float32(m.update_embedding(*b).item()) == np.float32(sa.update_embedding(*b)), i
        _same_sa(m, orc, sa, i)
    assert sa.mlp_step == 2 and sa.step == 7


def test_cfg4_tower_fit_tensor_cores_vs_exact_simt():
    """cfg4's tower (B = 8192, 400-400-400) on the tcgen05 tensor cores (3xTF32, not bit-exact) against the exact SIMT
    tower, both in mode 4, over two fits"""
    import fm_for_online_recommendation_b200 as pkg
    from test_gpu_fm import CRITEO
    lib = pkg.require_cuda()
    outs = []
    try:
        for tc in (1, 0):
            lib.fmb_set_tensor_cores(tc)
            torch.manual_seed(5)
            m = pkg.DeepFMAdam(CRITEO, embedding_size=10, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-4)
            m.enable_sparse_adam()
            with torch.no_grad():
                m._table[:, :11].mul_(0.1)
            for s in range(2):
                m.fit(*synth(CRITEO, 8192, 7 + s))
            outs.append((m._table.cpu().numpy().copy(), m._mlp.cpu().numpy().copy()))
    finally:
        lib.fmb_set_tensor_cores(1)
    assert (outs[0][0] == outs[1][0]).mean() > 0.99
    assert np.abs(outs[0][0] - outs[1][0]).max() <= 4.2e-4
    assert np.abs(outs[0][1] - outs[1][1]).max() <= 4.2e-4


@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 8), ("NFMAdam", 1, 12)])
@pytest.mark.parametrize("F", [1, 39])
def test_run_experiment(kind, L, H, F):
    sizes = SIZES39 if F == 39 else _sizes_f(1)
    m, orc, sa = _model(kind, sizes, 10, L, H, lr=0.01)
    m.update_embedding(*synth(sizes, 40, 399))     # the counters of the tables and the tower differ from here on
    sa.update_embedding(*synth(sizes, 40, 399))
    Xi, Xv, Y = synth(sizes, 300, 400 + F, zipf=True, real_xv=True)
    _, _, _, conf = m.run_experiment(Xi, Xv, Y)
    want, preds = sa.run_experiment(Xi, Xv, Y)
    assert conf == want
    assert np.array_equal(m._last_online_preds, preds)
    _same_sa(m, orc, sa, "end")


@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 16)])
def test_pickle_mid_run(kind, L, H):
    """a model pickled after three steps and unpickled continues bit-identical to the uninterrupted one"""
    m, orc, sa = _model(kind, SIZES39, 10, L, H)
    batches = _sweep(SIZES39, B39, 500, n=6)
    step = (lambda mm, b: mm.update_embedding(*b)) if kind == "FMAdam" else (lambda mm, b: mm.fit(*b))
    for b in batches[:3]:
        step(m, b)
    m2 = pickle.loads(pickle.dumps(m))
    assert m2.update_mode == 4 and (m2._sa.step, m2._sa.mlp_step) == (m._sa.step, m._sa.mlp_step)
    for b in batches[3:]:
        step(m, b)
        step(m2, b)
    for a, b in ((m._table, m2._table), (m.bias, m2.bias), (m._sa_mv, m2._sa_mv), (m._sa_bias, m2._sa_bias)):
        assert torch.equal(a, b)
    if L:
        assert torch.equal(m._mlp, m2._mlp) and torch.equal(m._sa_mlp, m2._sa_mlp)


def test_enable_again_resets_moments_and_counters():
    m, orc, sa = _model("DeepFMAdam", SIZES39, 10, 2, 16)
    m.fit(*synth(SIZES39, B39, 600))
    assert float(m._sa_mv[:, :, :11].abs().max()) > 0 and m._sa.step == 1 and m._sa.mlp_step == 1
    m.enable_sparse_adam(betas=(0.8, 0.99))
    assert not bool(m._sa_mv.any()) and not bool(m._sa_bias.any()) and not bool(m._sa_mlp.any())
    assert (m._sa.step, m._sa.mlp_step) == (0, 0)


def test_sharded_and_afm_refuse_mode_4():
    """the sharded step and AFM have no SparseAdam state: they refuse mode 4 with an error naming it, table unchanged"""
    import fm_for_online_recommendation_b200 as pkg
    from fm_for_online_recommendation_b200 import sharded as sh
    sizes, k, B = [50, 200, 3000], 4, 64
    Xi, _, Y = synth(sizes, B, 700)
    m = sh.ShardedFM(sizes, k, n=0.01, update_mode=4, world=1, rank=0)
    t0 = m.table.clone()

    def step():
        ids, y = m.encode(Xi, Y)
        idsT = m.phase_ids(ids)
        partial = m.phase_owner_forward(idsT.view(1, len(sizes), B))
        ctx = m.phase_combine(partial.view(1, B, m.PW), y)
        return m.phase_backward(ctx)

    with pytest.raises(pkg.FmbError, match="mode 4"):
        step()
    torch.cuda.synchronize()
    assert torch.equal(m.table, t0)
    m.update_mode = 0
    assert np.isfinite(float(step()))

    lib = pkg.require_cuda()
    a = pkg.AFMAdam(sizes, embedding_size=k, attention_size=4)
    t1 = a._table.clone()
    PD = int(lib.fmb_afm_dense_floats(k, 4))
    dg = torch.zeros(B, PD, device="cuda")
    assert lib.fmb_afm_dense_update(C.c_void_p(dg.data_ptr()), B, k, 4, *a._att_ptrs(), 0.01, 4, None, None) != 0
    assert b"mode 4" in lib.fmb_last_error()
    ws = torch.zeros(lib.fmb_bwd_workspace_bytes(B * 3, k), dtype=torch.uint8, device="cuda")
    sk = torch.zeros(B * 3, dtype=torch.int32, device="cuda")
    assert lib.fmb_fm_backward_runs_all(C.c_void_p(sk.data_ptr()), B * 3, C.c_void_p(a._table.data_ptr()), 3, k, 0.01, 4,
                                        C.c_void_p(ws.data_ptr()), ws.numel(), None) != 0
    assert b"mode 4" in lib.fmb_last_error()
    torch.cuda.synchronize()
    assert torch.equal(a._table, t1)
