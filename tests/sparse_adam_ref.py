"""References for update mode 4 (torch.optim.SparseAdam on the tables, torch.optim.Adam on the bias and the tower): the C
oracle of tests/sparse_adam_oracle.c and the torch harness of tests/adagrad_ref.py stepped by the two optimizers.

The harness is not nn.Embedding(sparse=True): SparseAdam coalesces that gradient, and CPU coalesce sums a row's repeated
entries in the order of an unstable sort, not in sample order.  The target takes the reference's dense gradient from
autograd (rows summed in sample order, as every kernel here does) and hands SparseAdam the rows the batch hits, as a sparse
tensor with unique indices (coalesce then adds nothing).  DESIGN.md section 4 has the difference.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch

from adagrad_ref import TorchFM

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_f = C.POINTER(C.c_float)
_lib = None


class _Sa(C.Structure):
    _fields_ = [("mV", _f), ("vV", _f), ("mw1", _f), ("vw1", _f), ("mbias", _f), ("vbias", _f), ("mmlp", _f), ("vmlp", _f),
                ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_float), ("step", C.c_int64),
                ("mlp_step", C.c_int64)]


def lib():
    """tests/sparse_adam_oracle.c compiled into a temporary directory (the source tree may be read-only)."""
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "sparse_adam_oracle.c")] + [os.path.join(ROOT, "oracle", f) for f in
                                                               ("fm_oracle.c", "oracle_math.h", "rsqrt14_table.inc")]
        h = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "fmb_sparse_adam_oracle_%d_%s.so" % (os.getuid(), h))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math",
                                   "-fvisibility=hidden", "-I", os.path.join(ROOT, "oracle"), "-o", tmp, srcs[0], "-lm",
                                   "-lpthread"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_adam_scalars.restype = None
        L.orc_adam_scalars.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int64, _f]
        L.orc_sparse_adam_update.restype = C.c_float
        L.orc_sparse_adam_update.argtypes = [C.c_float, C.c_float, _f, _f] + [C.c_float] * 4
        L.orc_vec_adam.restype = None
        L.orc_vec_adam.argtypes = [_f, _f, _f, _f, C.c_int64] + [C.c_float] * 6
        for n in ("orc_sa_update_embedding", "orc_sa_fit"):
            getattr(L, n).argtypes = [C.c_void_p] * 5 + [C.c_int]
        L.orc_sa_update_embedding.restype = C.c_float
        L.orc_sa_fit.restype = None
        L.orc_sa_run_experiment.restype = None
        L.orc_sa_run_experiment.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def scalars(lr, t, betas=(0.9, 0.999)):
    """the oracle's float scalars of step t: SparseAdam's -step_size, Adam's -step_size, Adam's sqrt(bias_correction2)"""
    out = (C.c_float * 3)()
    lib().orc_adam_scalars(float(lr), betas[0], betas[1], t, out)
    return np.array(out, np.float32)


def vec_sparse_adam(p, g, m, v, step, betas=(0.9, 0.999), eps=1e-8):
    """one SparseAdam step of the oracle on float32 arrays p, m, v (in place) with gradient g and scalar `step`"""
    b1c, b2c = np.float32(1.0 - betas[0]), np.float32(1.0 - betas[1])
    for i in range(p.size):
        mi, vi = C.c_float(m[i]), C.c_float(v[i])
        p[i] = lib().orc_sparse_adam_update(p[i], g[i], C.byref(mi), C.byref(vi), b1c, b2c, np.float32(eps), step)
        m[i], v[i] = mi.value, vi.value


def vec_adam(p, g, m, v, step, bc2s, betas=(0.9, 0.999), eps=1e-8):
    fp = lambda a: a.ctypes.data_as(_f)
    lib().orc_vec_adam(fp(p), fp(np.ascontiguousarray(g, np.float32)), fp(m), fp(v), p.size, np.float32(1.0 - betas[0]),
                       np.float32(betas[1]), np.float32(1.0 - betas[1]), np.float32(eps), step, bc2s)


class OracleSparseAdam:
    """Update mode 4 on an OracleDeep: m and v of V [R,k], w1 [R], the bias [1] and the tower [n_mlp], both counters."""

    def __init__(self, orc, betas=(0.9, 0.999), eps=1e-8):
        self.o = orc
        z = lambda a: np.zeros(a.shape, np.float32)
        self.mV, self.vV, self.mw1, self.vw1 = z(orc.V), z(orc.V), z(orc.w1), z(orc.w1)
        self.mbias, self.vbias = np.zeros(1, np.float32), np.zeros(1, np.float32)
        self.mmlp, self.vmlp = z(orc.mlp), z(orc.mlp)
        fp = lambda a: a.ctypes.data_as(_f)
        self.a = _Sa(fp(self.mV), fp(self.vV), fp(self.mw1), fp(self.vw1), fp(self.mbias), fp(self.vbias), fp(self.mmlp),
                     fp(self.vmlp), betas[0], betas[1], float(np.float32(eps)), 0, 0)
        orc.m.update_mode = 4

    @property
    def step(self):
        return self.a.step

    @property
    def mlp_step(self):
        return self.a.mlp_step

    def _args(self, Xi, Xv, Y):
        ids, xv, B = self.o._prep(Xi, Xv)
        y = np.ascontiguousarray(np.asarray(Y, dtype=np.float32).reshape(-1))
        return ids, xv, y, B

    def update_embedding(self, Xi, Xv, Y):
        ids, xv, y, B = self._args(Xi, Xv, Y)
        return float(lib().orc_sa_update_embedding(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data,
                                                   y.ctypes.data, B))

    def fit(self, Xi, Xv, Y):
        ids, xv, y, B = self._args(Xi, Xv, Y)
        lib().orc_sa_fit(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data, y.ctypes.data, B)

    def run_experiment(self, Xi, Xv, Y):
        ids, xv, y, N = self._args(Xi, Xv, Y)
        conf = (C.c_int64 * 4)()
        preds = np.empty(N, np.uint8)
        lib().orc_sa_run_experiment(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data, y.ctypes.data,
                                    N, conf, preds.ctypes.data)
        tp, fp, tn, fn = (int(c) for c in conf)
        return dict(tp=tp, fp=fp, tn=tn, fn=fn), preds.astype(bool)


class TorchSparseAdam:
    """TorchFM stepped by torch.optim.SparseAdam (tables: the unique rows each batch hits) and torch.optim.Adam (bias)."""

    def __init__(self, sizes, w1, V, bias, lr, betas=(0.9, 0.999), eps=1e-8):
        self.m = TorchFM(sizes, w1, V, bias)
        lr = float(np.float32(lr))
        self.tables = list(self.m.first_order_embeddings.parameters()) + list(self.m.second_order_embeddings.parameters())
        self.opt_e = torch.optim.SparseAdam(self.tables, lr=lr, betas=betas, eps=eps)
        self.opt_d = torch.optim.Adam([self.m.bias], lr=lr, betas=betas, eps=eps, foreach=False)

    def step(self, Xi, Xv, Y, loss_of_sigmoid):
        m = self.m
        self.opt_e.zero_grad()
        self.opt_d.zero_grad()
        z = m.forward_fm(Xi, Xv)
        loss = torch.nn.functional.binary_cross_entropy_with_logits(torch.sigmoid(z) if loss_of_sigmoid else z,
                                                                    torch.from_numpy(np.asarray(Y, np.float32)))
        loss.backward()
        Xi = np.asarray(Xi, np.int64).reshape(len(Y), -1)
        for f in range(Xi.shape[1]):
            rows = torch.from_numpy(np.unique(Xi[:, f]))
            for emb in (m.first_order_embeddings[f], m.second_order_embeddings[f]):
                w = emb.weight
                w.grad = torch.sparse_coo_tensor(rows[None], w.grad[rows], w.shape)
        self.opt_e.step()
        self.opt_d.step()
        return np.float32(loss.detach().item())

    def moments(self):
        """(mV, vV, mw1, vw1, m_bias, v_bias) in the layout of TorchFM.tables()"""
        m = self.m
        st = lambda p, key: self.opt_e.state[p][key] if p in self.opt_e.state else torch.zeros_like(p)
        cat = lambda mods, key: torch.cat([st(e.weight, key).detach() for e in mods]).numpy()
        mV, vV = cat(m.second_order_embeddings, "exp_avg"), cat(m.second_order_embeddings, "exp_avg_sq")
        mw1, vw1 = cat(m.first_order_embeddings, "exp_avg")[:, 0], cat(m.first_order_embeddings, "exp_avg_sq")[:, 0]
        sb = self.opt_d.state[m.bias]
        return (np.ascontiguousarray(mV), np.ascontiguousarray(vV), np.ascontiguousarray(mw1), np.ascontiguousarray(vw1),
                sb["exp_avg"].numpy().reshape(1), sb["exp_avg_sq"].numpy().reshape(1))

    def counters(self):
        steps = {int(self.opt_e.state[p]["step"]) for p in self.tables}
        return steps, int(self.opt_d.state[self.m.bias]["step"])
