"""Update modes 3 (Adagrad) and 4 (SparseAdam) of the row-sharded step on one B200, ranks emulated in one process (as in
test_sharded.py and test_sharded3.py), bit for bit against the oracle in sharded order (test_sharded_state.py pins that
oracle on torch) after every step: every rank's loss, its table shard, its state shard, the bias, the bias state and the
SparseAdam counter.  The padding columns and the extra row of the table and of the state hold a sentinel no kernel may
write."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from fm_for_online_recommendation_b200 import sharded as sh
from test_sharded import K, SIZES
from test_sharded3 import _attach
from test_sharded_state import batches, oracle_in_shard_order, state_arrays

pytestmark = pytest.mark.gpu

PAD = np.float32(-7.25)
LR = 0.01


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _enable(m, mode):
    if mode == 3:
        m.enable_adagrad(eps=1e-6, initial_accumulator_value=0.05)
    else:
        m.enable_sparse_adam()


def _ranks(mode, sizes, k, G, init_params, pad=True):
    ranks = [sh.ShardedFM(sizes, k, n=LR, init="zeros", world=G, rank=r) for r in range(G)]
    for m in ranks:
        m.load_full(*init_params)
        _enable(m, mode)
        if pad:
            with torch.no_grad():
                m.table[:, k + 1:] = float(PAD)
                m.table[m.R_local] = float(PAD)
                st = m._ada_sums if mode == 3 else m._sa_mv
                st[..., k + 1:] = float(PAD)
                st[m.R_local] = float(PAD)
    return ranks


def _same(ranks, st, what, pad=True):
    o = st.o
    G = len(ranks)
    want_state = state_arrays(st)
    for r, m in enumerate(ranks):
        V, w1 = m.local_params()
        assert np.array_equal(_bits(V), _bits(sh.shard_from_full(o.V, G, r))), (what, r, "V")
        assert np.array_equal(_bits(w1), _bits(sh.shard_from_full(o.w1, G, r))), (what, r, "w1")
        assert _bits(np.float32(m.bias.item())) == _bits(o.bias[0]), (what, r, "bias")
        got = m.local_state()
        n_rows = 2 if m.update_mode == 3 else 4      # per-row arrays, then the bias state
        for i, (g, w) in enumerate(zip(got, want_state)):
            w = sh.shard_from_full(w, G, r) if i < n_rows else w
            assert np.array_equal(_bits(g), _bits(w)), (what, r, "state", i, int((g != w).sum()))
        if m.update_mode == 4:
            assert got[-1] == st.step, (what, r, got[-1], st.step)
        if pad:
            t = m.table
            st_t = m._ada_sums if m.update_mode == 3 else m._sa_mv
            for name, x in (("table padding", t[:, ranks[0].k + 1:]), ("table extra row", t[m.R_local]),
                            ("state padding", st_t[..., ranks[0].k + 1:]), ("state extra row", st_t[m.R_local])):
                assert bool((x == float(PAD)).all()), (what, r, name, "written")


def _three_kernel_step(ranks, Xi, Y):
    G = len(ranks)
    B = Xi.shape[0] // G
    enc = [m.encode(Xi[r * B:(r + 1) * B], Y[r * B:(r + 1) * B]) for r, m in enumerate(ranks)]
    idsT_all = torch.stack([m.phase_ids(e[0]).clone() for m, e in zip(ranks, enc)]).contiguous()
    partials = [m.phase_owner_forward(idsT_all).clone() for m in ranks]
    ctxs = []
    for r, m in enumerate(ranks):
        recv = torch.stack([partials[o][r] for o in range(G)]).contiguous()
        ctxs.append(m.phase_combine(recv, enc[r][1]).clone())
    ctx_all = torch.cat(ctxs).contiguous()
    losses = [float(m.phase_backward(ctx_all).item()) for m in ranks]
    for m in ranks:
        m.check_overflow()
    return losses, ctx_all


def _fused_step(ranks, Xi, Y, streams):
    G = len(ranks)
    B = Xi.shape[0] // G
    enc = [m.encode(Xi[r * B:(r + 1) * B], Y[r * B:(r + 1) * B]) for r, m in enumerate(ranks)]
    for m, e in zip(ranks, enc):
        sh.check(m._lib.fmb_shard_transpose_ids_peers(sh.ptr(e[0]), B, m.F, G, m.rank, m._peer["ptrs"]["ids0"],
                                                      *m._sync_args(), -1, sh._stream()), "transpose")
    torch.cuda.synchronize()
    for m in ranks:
        m._sort_owned(m._peer["ids"][0], 0, m._peer["posflag"][0])
    torch.cuda.synchronize()
    held = []
    for m, e, s in zip(ranks, enc, streams):
        with torch.cuda.stream(s):
            held.append(m._fused_launch(e[1], 0, 0))
    torch.cuda.synchronize()
    for m in ranks:
        m.check_exchange()
        m.check_overflow()
    losses = [float(m._fused_finish(ws, wsb, 0).item()) for m, (ws, wsb) in zip(ranks, held)]
    return losses, ranks[0]._peer["ctx"]


def _check_losses(losses, want, what):
    assert all(_bits(np.float32(l)) == _bits(np.float32(want)) for l in losses), (what, losses, want)


@pytest.mark.parametrize("G,B", [(1, 64), (2, 48), (4, 33), (8, 16), (3, 20), (8, 128)])
@pytest.mark.parametrize("mode", [3, 4])
def test_three_kernel_step(mode, G, B):
    st, init_params = oracle_in_shard_order(mode, SIZES, K, G, LR, eps=1e-6, init=0.05)
    ranks = _ranks(mode, SIZES, K, G, init_params)
    for s, (Xi, Xv, Y) in enumerate(batches(SIZES, G * B, 5, 50)):
        want = st.update_embedding(Xi, Xv, Y)
        losses, _ = _three_kernel_step(ranks, Xi, Y)
        _check_losses(losses, want, s)
        _same(ranks, st, s)


@pytest.mark.parametrize("G", [1, 2, 4, 8])
@pytest.mark.parametrize("mode", [3, 4])
def test_fused_step(mode, G):
    B = 64
    st, init_params = oracle_in_shard_order(mode, SIZES, K, G, LR, eps=1e-6, init=0.05)
    ranks = _ranks(mode, SIZES, K, G, init_params)
    _attach(ranks, B)
    streams = [torch.cuda.Stream() for _ in range(G)]
    for s, (Xi, Xv, Y) in enumerate(batches(SIZES, G * B, 5, 80)):
        want = st.update_embedding(Xi, Xv, Y)
        losses, _ = _fused_step(ranks, Xi, Y, streams)
        _check_losses(losses, want, s)
        _same(ranks, st, s)


@pytest.mark.parametrize("G,B", [(2, 256), (8, 128)])
@pytest.mark.parametrize("mode", [3, 4])
def test_fused_step_hash_pass(mode, G, B):
    """test_sharded3's hash-pass batches (rows hit once, twice and many times in two sparse fields)"""
    sizes, k = [9, 300007, 5, 50021, 64, 3], 6
    st, init_params = oracle_in_shard_order(mode, sizes, k, G, LR, seed=1, eps=1e-6, init=0.05)
    ranks = _ranks(mode, sizes, k, G, init_params)
    _attach(ranks, B)
    streams = [torch.cuda.Stream() for _ in range(G)]
    rs = np.random.RandomState(5)
    for s in range(4):
        n = G * B
        Xi = np.stack([rs.randint(0, 9, n), (rs.randint(0, 700, n) * 428) % 300007, rs.randint(0, 5, n),
                       (rs.randint(0, 2000, n) * 25) % 50021, rs.randint(0, 64, n), rs.randint(0, 3, n)], 1)
        Y = (rs.uniform(size=n) < 0.4).astype(np.float32)
        want = st.update_embedding(Xi, np.ones(Xi.shape, np.float32), Y)
        losses, _ = _fused_step(ranks, Xi, Y, streams)
        cnts = ranks[0]._ws["counts0"].cpu().numpy()
        assert cnts[1] < B and cnts[3] < B, cnts          # the hash pass listed only the multi-hit entries
        _check_losses(losses, want, s)
        _same(ranks, st, s)


@pytest.mark.parametrize("path", ["three_kernel", "fused"])
@pytest.mark.parametrize("mode", [3, 4])
def test_zero_gradient_rows_hit_once(mode, path):
    """samples whose logit saturates (sigmoid(z) rounds to y = 1) have delta = +0, so their rows hit once get a zero
    gradient: SparseAdam still steps them (m and v decay, p moves), Adagrad leaves them bit-unchanged"""
    sizes, k, G, B = [64, 100, 128], 4, 2, 32
    n, F = G * B, 3
    st, init_params = oracle_in_shard_order(mode, sizes, k, G, LR, seed=7, eps=1e-6, init=0.05)
    rs = np.random.RandomState(11)
    Xi = np.stack([rs.permutation(fs)[:n] for fs in sizes], 1)     # every row hit at most once
    sat = np.arange(n) < n // 2                                     # these samples saturate
    V0, w0, b0 = init_params
    off = np.concatenate([[0], np.cumsum(sizes)])[:-1]
    for f in range(F):
        w0[off[f] + Xi[sat, f]] = np.float32(30.0)                 # z ~ 90
    st.o.w1[:] = w0
    ranks = _ranks(mode, sizes, k, G, (V0, w0, b0))
    if path == "fused":
        _attach(ranks, B)
        streams = [torch.cuda.Stream() for _ in range(G)]
        step = lambda Xi, Y: _fused_step(ranks, Xi, Y, streams)
    else:
        step = lambda Xi, Y: _three_kernel_step(ranks, Xi, Y)
    Y0 = np.where(sat, 0.0, (rs.uniform(size=n) < 0.4)).astype(np.float32)   # step 1: every row gets a gradient
    Y1 = np.where(sat, 1.0, (rs.uniform(size=n) < 0.4)).astype(np.float32)   # step 2: the saturated ones get +0
    ones = np.ones(Xi.shape, np.float32)
    for s, Y in enumerate((Y0, Y1)):
        before = [(m.table.clone(), (m._ada_sums if mode == 3 else m._sa_mv).clone()) for m in ranks]
        want = st.update_embedding(Xi, ones, Y)
        losses, ctx = step(Xi, Y)
        _check_losses(losses, want, s)
        _same(ranks, st, s)
    # premise: delta is +0 exactly on the saturated samples of step 2, nonzero on the others
    kp4 = ranks[0].kp4
    d = ctx[:, kp4].cpu().numpy()
    assert (_bits(d[sat]) == 0).all(), d[sat]
    assert (d[~sat] != 0).all()
    # the rows the saturated samples hit, on their owners
    for r, m in enumerate(ranks):
        t0, s0 = before[r]
        t1, s1 = m.table, (m._ada_sums if mode == 3 else m._sa_mv)
        gids = (Xi[sat] + off[None, :]).reshape(-1)
        lrows = torch.from_numpy(gids[gids % G == r] // G).to(m.device)
        assert lrows.numel() > 0
        moved_p = (t1[lrows, :k + 1] != t0[lrows, :k + 1]).any(1)
        moved_s = (s1[lrows] != s0[lrows]).reshape(lrows.numel(), -1).any(1)
        if mode == 4:
            assert bool(moved_p.all()) and bool(moved_s.all()), (r, "SparseAdam must step every row hit")
        else:
            assert not bool(moved_p.any()) and not bool(moved_s.any()), (r, "Adagrad must leave zero-gradient rows")


@pytest.mark.parametrize("G,mode", [(1, 3), (1, 4), (2, 3), (2, 4), (8, 3), (8, 4)])
def test_same_as_single_gpu_fm(mode, G):
    """G = 1 at test_sharded.SIZES, and two fields at G = 2 and 8 (where the owner fold is the reference order), step
    exactly like FMAdam.update_embedding with the same update mode"""
    from test_gpu_fm import _pair
    sizes, k = (SIZES, K) if G == 1 else ([37, 300], 5)
    fm, orc = _pair("FMAdam", sizes, k, lr=LR, scale=0.3)
    _enable(fm, mode)
    ranks = _ranks(mode, sizes, k, G, (orc.V, orc.w1, orc.bias), pad=False)
    R = sum(sizes)
    for s, (Xi, Xv, Y) in enumerate(batches(sizes, 24 * G, 6, 900)):
        want = float(fm.update_embedding(Xi, Xv, Y).item())
        losses, _ = _three_kernel_step(ranks, Xi, Y)
        _check_losses(losses, want, s)
    full = lambda f: sh.full_from_shards([f(m) for m in ranks])
    t = fm._table[:R].cpu().numpy()
    assert np.array_equal(_bits(full(lambda m: m.table[:m.R_local].cpu().numpy())[:, :k + 1]), _bits(t[:, :k + 1]))
    assert _bits(np.float32(ranks[0].bias.item())) == _bits(np.float32(fm.bias.item()))
    if mode == 3:
        got = full(lambda m: m._ada_sums[:m.R_local].cpu().numpy())[:, :k + 1]
        want_s = fm._ada_sums[:R, :k + 1].cpu().numpy()
        got_b, want_b = ranks[0]._ada_bias, fm._ada_bias
    else:
        got = full(lambda m: m._sa_mv[:m.R_local].cpu().numpy())[:, :, :k + 1]
        want_s = fm._sa_mv[:R, :, :k + 1].cpu().numpy()
        got_b, want_b = ranks[0]._sa_bias, fm._sa_bias
        assert all(m._sa.step == fm._sa.step for m in ranks)
    assert np.array_equal(_bits(got), _bits(want_s))
    assert torch.equal(got_b, want_b)


def test_refusals():
    """mode 4 cannot be captured: every capture entry point names the mode and leaves table and state as they were;
    a mode 3 or 4 fused step without its state is refused by the library, naming the mode"""
    import fm_for_online_recommendation_b200 as pkg
    sizes, k, B = [50, 200, 3000], 4, 64
    Xi, _, Y = batches(sizes, B, 1, 700)[0]
    m = sh.ShardedFM(sizes, k, n=LR, world=1, rank=0)
    m.enable_sparse_adam()
    t0, s0 = m.table.clone(), m._sa_mv.clone()
    ids, y = m.encode(Xi, Y)
    for name in ("capture", "capture_pipelined", "capture_peers", "capture_fused"):
        with pytest.raises(RuntimeError, match="mode 4"):
            getattr(m, name)(ids, y)
    torch.cuda.synchronize()
    assert torch.equal(m.table, t0) and torch.equal(m._sa_mv, s0) and m._sa.step == 0
    for mode in (3, 4):
        f = sh.ShardedFM(sizes, k, n=LR, update_mode=mode, world=1, rank=0, init="zeros")
        _attach([f], B)
        f._sort_owned(f._peer["ids"][0], 0, f._peer["posflag"][0])
        with pytest.raises(pkg.FmbError, match=f"mode {mode}"):
            f._fused_launch(y, 0, 0)
        torch.cuda.synchronize()
        assert not bool(f.table.any())


@pytest.mark.parametrize("mode,graph", [(3, False), (3, True), (4, False)])
def test_pipelined_peer_fused_equal_eager_world1_nccl(mode, graph):
    """the pipelined, peer-memory and fused steps against update_embedding over a real NCCL group (world 1), state
    included; run as a child process with a timeout (tests/sharded_state_pipeline_check.py)"""
    here = os.path.dirname(os.path.abspath(__file__))
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="1", RANK="0", LOCAL_RANK="0")
    cmd = [sys.executable, os.path.join(here, "sharded_state_pipeline_check.py"), "--mode", str(mode)] + (["--graph"] if graph else [])
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "STATE_PIPELINE_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
