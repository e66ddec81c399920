"""The FM step session's bookkeeping (csrc/session.cu): how many step graphs it keeps and how many kernels it launches, step
by step, for fixed call sequences of its device-input, pipelined host-input and blocking host-input entry points.  The
counts follow from which graph each step replays, captures or re-points, and from whether a batch's sort runs in the step,
rides along the step before or runs ahead on the side stream.  The results of these steps are pinned bit for bit by
test_gpu_fm.py; this pins the decisions."""
import ctypes as C

import numpy as np
import pytest
import torch

from _util import synth

pytestmark = pytest.mark.gpu

SIZES, K = [300, 40, 7, 2000, 3], 10

# per step: (graphs cached, kernels launched by the step); an entry (n, 0) is a point between steps
EXPECTED = {
    "device_next": [(0, 7), (1, 5)] + [(2, 5)] * 9 + [(3, 3), (4, 7)] + [(4, 5)] * 10 + [(4, 3)],
    "host_async_2": [(0, 5), (1, 5)] + [(2, 5)] * 8 + [(3, 5), (4, 5)],
    "host_async_4": [(0, 5), (1, 5), (2, 5), (3, 5)] + [(4, 5)] * 6 + [(5, 5), (6, 5)],
    "host_blocking": [(0, 5), (1, 5), (2, 5), (2, 5), (2, 5)],
    "adagrad_drops_graphs": [(0, 7), (1, 5), (2, 5), (2, 5), (0, 0), (1, 5), (2, 5), (2, 5), (3, 3)],
}


def _model():
    import fm_for_online_recommendation_b200 as pkg
    torch.manual_seed(0)
    return pkg.FMAdam(SIZES, embedding_size=K, n=1e-3)


class _Trace:
    def __init__(self, lib, session):
        self.lib, self.s, self.out = lib, session, []
        self.last = lib.fmb_session_launches(session)

    def mark(self):
        torch.cuda.synchronize()
        n = self.lib.fmb_session_launches(self.s)
        self.out.append((self.lib.fmb_session_graph_count(self.s), n - self.last))
        self.last = n


def _host_args(m, B, seed):
    Xi, _, Y = synth(SIZES, B, seed, zipf=(seed % 2 == 0))
    ids = np.ascontiguousarray((Xi + m._offsets_np[:-1][None, :]).astype(np.int32))
    return ids, np.ascontiguousarray(Y, dtype=np.float32)


def device_next(B=2048):
    """12 device-resident batches, each step announcing the next one, twice over"""
    import fm_for_online_recommendation_b200 as pkg
    m = _model()
    enc = [m.encode(*synth(SIZES, B, 10 + i, zipf=(i % 3 == 0))) for i in range(12)]
    tr = _Trace(pkg.require_cuda(), m._get_session(B))
    for _ in range(2):
        for i in range(12):
            m._fm_step(enc[i], 0, enc[i + 1] if i + 1 < 12 else None)
            tr.mark()
    return tr.out


def host_async(nslot, B=4100, nsteps=10):
    """fmb_session_fm_step_host_async over nslot slots (even steps pinned, odd steps pageable), losses collected nslot - 1
    steps later, then two blocking host steps on the same session"""
    import fm_for_online_recommendation_b200 as pkg
    lib = pkg.require_cuda()
    m = _model()
    s = m._get_session(B)
    tr = _Trace(lib, s)
    tp, bp = C.c_void_p(m._table.data_ptr()), C.c_void_p(m.bias.data_ptr())
    args = [_host_args(m, B, 40 + i) for i in range(nsteps)]
    pinned = [torch.from_numpy(a[0]).pin_memory() for a in args]
    loss = C.c_float()
    for i, (ids, y) in enumerate(args):
        src = C.c_void_p(pinned[i].data_ptr()) if i % 2 == 0 else ids.ctypes.data_as(C.c_void_p)
        rc = lib.fmb_session_fm_step_host_async(s, i % nslot, src, None, y.ctypes.data_as(C.c_void_p), B, tp, bp,
                                                m._key_bits, 0, m._lr, 0, None)
        assert rc == 0, lib.fmb_last_error()
        if i >= nslot - 1:
            assert lib.fmb_session_wait_loss(s, (i - nslot + 1) % nslot, C.byref(loss)) == 0
        tr.mark()
    for i in range(nsteps - nslot + 1, nsteps):
        assert lib.fmb_session_wait_loss(s, i % nslot, C.byref(loss)) == 0
    for ids, y in args[:2]:
        rc = lib.fmb_session_fm_step_host(s, ids.ctypes.data_as(C.c_void_p), None, y.ctypes.data_as(C.c_void_p), B, tp, bp,
                                          m._key_bits, 0, m._lr, 0, C.byref(loss), None)
        assert rc == 0, lib.fmb_last_error()
        tr.mark()
    return tr.out


def host_blocking(B=1000, nsteps=5):
    """fmb_session_fm_step_host: copies in, step, loss copied back, synchronised"""
    import fm_for_online_recommendation_b200 as pkg
    lib = pkg.require_cuda()
    m = _model()
    s = m._get_session(B)
    tr = _Trace(lib, s)
    tp, bp = C.c_void_p(m._table.data_ptr()), C.c_void_p(m.bias.data_ptr())
    loss = C.c_float()
    for i in range(nsteps):
        ids, y = _host_args(m, B, 70 + i)
        rc = lib.fmb_session_fm_step_host(s, ids.ctypes.data_as(C.c_void_p), None, y.ctypes.data_as(C.c_void_p), B, tp, bp,
                                          m._key_bits, 0, m._lr, 0, C.byref(loss), None)
        assert rc == 0, lib.fmb_last_error()
        tr.mark()
    return tr.out


def adagrad_drops_graphs(B=2048):
    """device steps in mode 0, enable_adagrad (the cached graphs are dropped), device steps in mode 3"""
    import fm_for_online_recommendation_b200 as pkg
    m = _model()
    enc = [m.encode(*synth(SIZES, B, 90 + i)) for i in range(8)]
    tr = _Trace(pkg.require_cuda(), m._get_session(B))
    for i in range(4):
        m._fm_step(enc[i], 0, enc[i + 1])
        tr.mark()
    m.enable_adagrad()
    tr.mark()
    for i in range(4, 8):
        m._fm_step(enc[i], 0, enc[i + 1] if i + 1 < 8 else None)
        tr.mark()
    return tr.out


SEQUENCES = {
    "device_next": device_next,
    "host_async_2": lambda: host_async(2),
    "host_async_4": lambda: host_async(4),
    "host_blocking": host_blocking,
    "adagrad_drops_graphs": adagrad_drops_graphs,
}


@pytest.mark.parametrize("name", sorted(SEQUENCES))
def test_session_graphs_and_launches(name):
    assert [tuple(x) for x in SEQUENCES[name]()] == [tuple(x) for x in EXPECTED[name]]
