"""Update mode 3 (torch.optim.Adagrad) on the GPU, bit for bit against the C oracle of tests/adagrad_oracle.c after every
step: the loss, V, w1, the bias, the tower, and the sums of the table, the bias and the tower.  The padding columns of the
table and of its sums hold a sentinel that no kernel may write.  The five traj_sgd cases are also stepped against the torch
harness (tests/adagrad_ref.py: the reference's forward pass, autograd and torch.optim.Adagrad) directly."""
import pickle

import numpy as np
import pytest
import torch

from _util import GOLDEN, synth
from adagrad_ref import OracleAdagrad, TorchFM, adagrad
from test_gpu_fm import _pair
from test_gpu_fm_shapes import B39, PAD, SIZES39, _push_padded, _run_batch, _same, _sizes_f
from traj_common import digest, init_tables

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _model(kind, sizes, k, L=0, H=0, lr=0.05, eps=1e-10, init=0.0, **kw):
    m, orc = _pair(kind, sizes, k, L, H, lr=lr, scale=0.1, **kw)
    orc.bias[:] = np.float32(0.1)
    _push_padded(m, orc)
    m.enable_adagrad(eps, init)
    with torch.no_grad():
        m._ada_sums[:, k + 1:] = float(PAD)
    return m, orc, OracleAdagrad(orc, eps, init)


def _same_ada(m, orc, ada, step=None):
    _same(m, orc, step)
    k = orc.k
    s = m._ada_sums.cpu().numpy()
    assert np.array_equal(_bits(s[:, :k]), _bits(ada.sV)), (step, "sums of V", int((s[:, :k] != ada.sV).sum()))
    assert np.array_equal(_bits(s[:, k]), _bits(ada.sw1)), (step, "sums of w1")
    assert (s[:, k + 1:] == PAD).all(), (step, "padding of the sums written")
    assert np.array_equal(_bits(m._ada_bias.cpu().numpy()), _bits(ada.sbias)), (step, "bias sum")
    if orc.L and m._ada_mlp is not None:
        assert np.array_equal(_bits(m._ada_mlp.cpu().numpy()), _bits(ada.smlp[:m._ada_mlp.numel()])), (step, "tower sums")


def _ue(m, orc, ada, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        got = m.update_embedding(Xi, Xv, Y).item()
        want = ada.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), (i, got, want)
        _same_ada(m, orc, ada, i)


def _fit(m, orc, ada, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        m.fit(Xi, Xv, Y)
        ada.fit(Xi, Xv, Y)
        _same_ada(m, orc, ada, i)


def _sweep(sizes, B, seed, n=6):
    """all-ones then real-valued steps (eager, captured, re-pointed replay of each), Zipf ids every other step"""
    return [synth(sizes, B, seed + i, real_xv=(i >= n // 2), zipf=(i % 2 == 0)) for i in range(n)]


@pytest.mark.parametrize("F", [1, 39])
@pytest.mark.parametrize("k", [1, 3, 10, 33, 124])
def test_update_embedding(k, F):
    sizes, B = (SIZES39, B39) if F == 39 else (_sizes_f(1), 99)
    m, orc, ada = _model("FMAdam", sizes, k, init=0.1 if k == 10 else 0.0)
    _ue(m, orc, ada, _sweep(sizes, B, 100 + k))


def test_update_embedding_f511_k32():
    sizes = _sizes_f(511)
    m, orc, ada = _model("FMAdam", sizes, 32, eps=1e-6)
    _ue(m, orc, ada, _sweep(sizes, 24, 7))


@pytest.mark.parametrize("n", [2, 129, 1025])
def test_hot_row_runs(n):
    """one row hit n times in three fields: direct part, ring, and (from 128 entries) the long-run CTAs of the run kernel"""
    Xi, Xv, Y, _ = _run_batch(n, 0, 3 + n)
    sizes = [int(v) for v in [5, Xi.shape[0] + 4, 16 * Xi.shape[0], 3, Xi.shape[0] + 4]]
    m, orc, ada = _model("FMAdam", sizes, 10)
    batches = [(Xi, Xv, Y)] + [_run_batch(n, 1, 50 + n + i, real_xv=(i == 1))[:3] for i in range(2)]
    _ue(m, orc, ada, batches)
    m2, orc2, ada2 = _model("FMAdam", sizes, 10)
    _fit(m2, orc2, ada2, batches)


def test_batch_above_per_field_sort_limit():
    sizes, k, B = [70, 9, 40000, 3000, 150000], 33, 70001
    m, orc, ada = _model("FMAdam", sizes, k)
    assert B > m._lib.fmb_sort_fields_max_batch()
    _ue(m, orc, ada, [synth(sizes, B, 60 + i, zipf=True, real_xv=(i == 1)) for i in range(2)])


def test_next_batch_pipeline():
    """update_embedding with next_batch: eager first step, graph capture, re-pointed replays with the pre-sort"""
    m, orc, ada = _model("FMAdam", SIZES39, 10)
    host = [synth(SIZES39, B39, 200 + i, zipf=(i % 2 == 0)) for i in range(6)]
    enc = [m.encode(*b) for b in host]
    for i, (Xi, Xv, Y) in enumerate(host):
        nxt = enc[i + 1] if i + 1 < len(enc) else None
        got = m.update_embedding(enc[i], None, None, next_batch=nxt).item()
        want = ada.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), i
        _same_ada(m, orc, ada, i)
    assert m._lib.fmb_session_graph_count(m._session) >= 1


@pytest.mark.parametrize("k", [3, 10, 33])
@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 16), ("NFMAdam", 2, 24)])
def test_fit(kind, L, H, k):
    """tower fit at SIMT shapes (bit-exact): two gradient chains per row for DeepFM, the tower chain alone for NFM, the
    tower's and the bias's sums; the third and later calls replay the captured fit"""
    m, orc, ada = _model(kind, SIZES39, k, L, H, init=0.1 if k == 10 else 0.0)
    _fit(m, orc, ada, _sweep(SIZES39, B39, 300 + k))


def test_cfg4_tower_fit_tensor_cores_vs_exact_simt():
    """cfg4's tower (B = 8192, 400-400-400) on the tcgen05 tensor cores against the exact SIMT tower, both in mode 3:
    the first Adagrad step of a coordinate is lr * g / (|g| + eps), a sign step like the reference's, so the tolerances of
    tests/test_gpu_deep.py's mode-0 comparison apply"""
    import fm_for_online_recommendation_b200 as pkg
    from test_gpu_fm import CRITEO
    lib = pkg.require_cuda()
    Xi, Xv, Y = synth(CRITEO, 8192, 7)
    outs = []
    try:
        for tc in (1, 0):
            lib.fmb_set_tensor_cores(tc)
            torch.manual_seed(5)
            m = pkg.DeepFMAdam(CRITEO, embedding_size=10, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-4)
            m.enable_adagrad()
            with torch.no_grad():
                m._table[:, :11].mul_(0.1)
            e = m.encode(Xi, Xv, Y)
            z0 = m.forward(e, None).clone()
            m.fit(e, None, None)
            outs.append((z0.cpu().numpy(), m._table.cpu().numpy().copy(), m._mlp.cpu().numpy().copy()))
    finally:
        lib.fmb_set_tensor_cores(1)
    np.testing.assert_allclose(outs[0][0], outs[1][0], rtol=1e-5, atol=1e-5)
    same = (outs[0][1] == outs[1][1]).mean()
    assert same > 0.99, same
    assert np.abs(outs[0][1] - outs[1][1]).max() <= 2.1e-4
    assert np.abs(outs[0][2] - outs[1][2]).max() <= 2.1e-4


@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 8), ("NFMAdam", 1, 12)])
@pytest.mark.parametrize("F", [1, 39])
def test_run_experiment(kind, L, H, F):
    sizes = SIZES39 if F == 39 else _sizes_f(1)
    m, orc, ada = _model(kind, sizes, 10, L, H, lr=0.01)
    Xi, Xv, Y = synth(sizes, 300, 400 + F, zipf=True, real_xv=True)
    _, _, _, conf = m.run_experiment(Xi, Xv, Y)
    want, preds = ada.run_experiment(Xi, Xv, Y)
    assert conf == want
    assert np.array_equal(m._last_online_preds, preds)
    _same_ada(m, orc, ada, "end")


@pytest.mark.parametrize("name", ["cfg1", "frappe_zipf", "deepfm_fm_part", "nfm_loss_of_sigmoid", "frappe_zipf_xv"])
def test_traj_cases_against_torch_adagrad(name):
    """300 steps of update_embedding against the torch harness with torch.optim.Adagrad (CPU): every loss, the whole
    table, the bias and the sums"""
    import fm_for_online_recommendation_b200 as pkg
    from golden.make_trajectory_sgd import CASES, cfg_of
    kind, sizes, B, zipf, (L, H), lr, steps = CASES[name]
    g = dict(np.load(GOLDEN + "/traj_sgd.npz"))
    w1, V = init_tables(cfg_of(name))
    bias = g[name + "_init_bias"][0]
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        h = TorchFM(sizes, w1, V, bias)
        opt = adagrad(h, lr)
        kw = dict(num_hidden_layers=L, neuron_per_hidden_layer=H) if L else {}
        m = getattr(pkg, kind)(sizes, embedding_size=10, n=lr, **kw)
        with torch.no_grad():
            m._table[:, :10] = torch.from_numpy(V)
            m._table[:, 10] = torch.from_numpy(w1)
            m.bias.fill_(float(bias))
        m.enable_adagrad()
        for s in range(300):
            Xi, Xv, Y = synth(sizes, B, 9000 + s, real_xv=name.endswith("_xv"), zipf=zipf)
            want = h.step(opt, Xi, Xv, Y, kind == "NFMAdam")
            got = np.float32(m.update_embedding(Xi, Xv, Y).item())
            assert _bits(got) == _bits(want), (s, got, want)
            if s + 1 in (1, 100, 300):
                t = m._table.cpu().numpy()
                hV, hw1, hb = h.tables()
                assert digest(np.ascontiguousarray(t[:, :10]), np.ascontiguousarray(t[:, 10]),
                              m.bias.detach().cpu().numpy().reshape(1)) == digest(hV, hw1, hb), s + 1
                sV, sw1, sb = h.adagrad_sums(opt)
                su = m._ada_sums.cpu().numpy()
                assert np.array_equal(_bits(su[:, :10]), _bits(sV)) and np.array_equal(_bits(su[:, 10]), _bits(sw1)), s + 1
                assert np.array_equal(_bits(m._ada_bias.cpu().numpy()), _bits(sb)), s + 1
    finally:
        torch.set_num_threads(n)


@pytest.mark.parametrize("kind,L,H", [("FMAdam", 0, 0), ("DeepFMAdam", 2, 16)])
def test_pickle_mid_run(kind, L, H):
    """a model pickled after three steps and unpickled continues bit-identical to the uninterrupted one"""
    m, orc, ada = _model(kind, SIZES39, 10, L, H)
    batches = _sweep(SIZES39, B39, 500, n=6)
    step = (lambda mm, b: mm.update_embedding(*b)) if kind == "FMAdam" else (lambda mm, b: mm.fit(*b))
    for b in batches[:3]:
        step(m, b)
    m2 = pickle.loads(pickle.dumps(m))
    assert m2.update_mode == 3
    for b in batches[3:]:
        step(m, b)
        step(m2, b)
    for a, b in ((m._table, m2._table), (m.bias, m2.bias), (m._ada_sums, m2._ada_sums), (m._ada_bias, m2._ada_bias)):
        assert torch.equal(a, b)
    if L:
        assert torch.equal(m._mlp, m2._mlp) and torch.equal(m._ada_mlp, m2._ada_mlp)


def test_enable_adagrad_again_resets_the_sums():
    m, orc, ada = _model("FMAdam", SIZES39, 10)
    m.update_embedding(*synth(SIZES39, B39, 600))
    assert float(m._ada_sums[:, :11].max()) > 0
    m.enable_adagrad(initial_accumulator_value=0.5)
    assert bool((m._ada_sums == 0.5).all()) and float(m._ada_bias) == 0.5


def test_sharded_and_afm_refuse_mode_3():
    """the sharded step and AFM have no Adagrad state: they refuse mode 3 with an error naming it and stay usable"""
    import ctypes as C
    import fm_for_online_recommendation_b200 as pkg
    from fm_for_online_recommendation_b200 import sharded as sh
    sizes, k, B = [50, 200, 3000], 4, 64
    Xi, _, Y = synth(sizes, B, 700)
    m = sh.ShardedFM(sizes, k, n=0.01, update_mode=3, world=1, rank=0)
    t0 = m.table.clone()

    def step():
        ids, y = m.encode(Xi, Y)
        idsT = m.phase_ids(ids)
        partial = m.phase_owner_forward(idsT.view(1, len(sizes), B))
        ctx = m.phase_combine(partial.view(1, B, m.PW), y)
        return m.phase_backward(ctx)

    with pytest.raises(pkg.FmbError, match="mode 3"):
        step()
    torch.cuda.synchronize()
    assert torch.equal(m.table, t0)
    m.update_mode = 0
    assert np.isfinite(float(step()))

    lib = pkg.require_cuda()
    a = pkg.AFMAdam(sizes, embedding_size=k, attention_size=4)
    PD = int(lib.fmb_afm_dense_floats(k, 4))
    dg = torch.zeros(B, PD, device="cuda")
    ptrs = a._att_ptrs()
    assert lib.fmb_afm_dense_update(C.c_void_p(dg.data_ptr()), B, k, 4, *ptrs, 0.01, 3, None, None) != 0
    assert b"mode 3" in lib.fmb_last_error()
    ws = torch.zeros(lib.fmb_bwd_workspace_bytes(B * 3, k), dtype=torch.uint8, device="cuda")
    sk = torch.zeros(B * 3, dtype=torch.int32, device="cuda")
    assert lib.fmb_fm_backward_runs_all(C.c_void_p(sk.data_ptr()), B * 3, C.c_void_p(a._table.data_ptr()), 3, k, 0.01, 3,
                                        C.c_void_p(ws.data_ptr()), ws.numel(), None) != 0
    assert b"mode 3" in lib.fmb_last_error()
    loss = a.update_embedding(Xi, np.ones(Xi.shape, np.float32), Y)
    assert np.isfinite(float(loss))
