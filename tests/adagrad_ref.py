"""References for update mode 3 (torch.optim.Adagrad): the C oracle of tests/adagrad_oracle.c and a torch harness.

``OracleAdagrad`` wraps an ``oracle.deep.OracleDeep`` (its parameters, forward pass and gradient sums) and adds Adagrad's
sums.  ``TorchFM`` restates the reference's forward_fm (models/models_online_deep/fm_adam.py:34-54) with per-field
nn.Embedding tables, so that torch autograd and a real ``torch.optim`` optimizer can step it; tests/test_adagrad.py first
checks that it reproduces the live reference's SGD trajectories (tests/golden/traj_sgd.npz) bit for bit.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_f = C.POINTER(C.c_float)
_lib = None


class _Ada(C.Structure):
    _fields_ = [("sV", _f), ("sw1", _f), ("sbias", _f), ("smlp", _f), ("eps", C.c_float)]


def lib():
    """tests/adagrad_oracle.c compiled into a temporary directory (the source tree may be read-only)."""
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "adagrad_oracle.c")] + [os.path.join(ROOT, "oracle", f) for f in
                                                           ("fm_oracle.c", "oracle_math.h", "rsqrt14_table.inc")]
        h = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "fmb_adagrad_oracle_%d_%s.so" % (os.getuid(), h))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math",
                                   "-fvisibility=hidden", "-I", os.path.join(ROOT, "oracle"), "-o", tmp, srcs[0], "-lm",
                                   "-lpthread"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_adagrad_update.restype = C.c_float
        L.orc_adagrad_update.argtypes = [C.c_float, C.c_float, _f, C.c_float, C.c_float]
        L.orc_vec_adagrad.restype = None
        L.orc_vec_adagrad.argtypes = [_f, _f, _f, C.c_int64, C.c_float, C.c_float]
        L.orc_ada_update_embedding.restype = C.c_float
        L.orc_ada_update_embedding.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_ada_fit.restype = None
        L.orc_ada_fit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_ada_run_experiment.restype = None
        L.orc_ada_run_experiment.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                             C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def vec_adagrad(p, g, s, lr, eps):
    """one Adagrad step of the oracle on float32 arrays p, s (in place) with gradient g"""
    fp = lambda a: a.ctypes.data_as(_f)
    lib().orc_vec_adagrad(fp(p), fp(np.ascontiguousarray(g, np.float32)), fp(s), p.size, lr, eps)


class OracleAdagrad:
    """Update mode 3 on an OracleDeep: sums sV [R,k], sw1 [R], sbias [1], smlp [n_mlp], all starting at `init`."""

    def __init__(self, orc, eps=1e-10, init=0.0):
        self.o = orc
        v = np.float32(init)
        self.sV = np.full(orc.V.shape, v, np.float32)
        self.sw1 = np.full(orc.w1.shape, v, np.float32)
        self.sbias = np.full(1, v, np.float32)
        self.smlp = np.full(orc.mlp.shape, v, np.float32)
        fp = lambda a: a.ctypes.data_as(_f)
        self.a = _Ada(fp(self.sV), fp(self.sw1), fp(self.sbias), fp(self.smlp), float(np.float32(eps)))
        orc.m.update_mode = 3

    def _args(self, Xi, Xv, Y):
        ids, xv, B = self.o._prep(Xi, Xv)
        y = np.ascontiguousarray(np.asarray(Y, dtype=np.float32).reshape(-1))
        return ids, xv, y, B

    def update_embedding(self, Xi, Xv, Y):
        ids, xv, y, B = self._args(Xi, Xv, Y)
        return float(lib().orc_ada_update_embedding(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data,
                                                    y.ctypes.data, B))

    def fit(self, Xi, Xv, Y):
        ids, xv, y, B = self._args(Xi, Xv, Y)
        lib().orc_ada_fit(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data, y.ctypes.data, B)

    def run_experiment(self, Xi, Xv, Y):
        ids, xv, y, N = self._args(Xi, Xv, Y)
        conf = (C.c_int64 * 4)()
        preds = np.empty(N, np.uint8)
        lib().orc_ada_run_experiment(C.byref(self.o.m), C.byref(self.a), ids.ctypes.data, xv.ctypes.data, y.ctypes.data,
                                     N, conf, preds.ctypes.data)
        tp, fp, tn, fn = (int(c) for c in conf)
        return dict(tp=tp, fp=fp, tn=tn, fn=fn), preds.astype(bool)


class TorchFM(nn.Module):
    """forward_fm of the reference with per-field nn.Embedding tables (fm_adam.py:34-54, deepfm_adam.py:46-77)."""

    def __init__(self, sizes, w1, V, bias):
        super().__init__()
        off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self.off, k = off, V.shape[1]
        self.first_order_embeddings = nn.ModuleList([nn.Embedding(int(fs), 1) for fs in sizes])
        self.second_order_embeddings = nn.ModuleList([nn.Embedding(int(fs), k) for fs in sizes])
        with torch.no_grad():
            for f in range(len(sizes)):
                self.first_order_embeddings[f].weight.copy_(torch.from_numpy(w1[off[f]:off[f + 1]].reshape(-1, 1)))
                self.second_order_embeddings[f].weight.copy_(torch.from_numpy(V[off[f]:off[f + 1]]))
        self.bias = nn.Parameter(torch.tensor(float(np.float32(bias))))

    def forward_fm(self, Xi, Xv):
        Xi = torch.from_numpy(np.asarray(Xi, np.int64)).reshape(Xv.shape[0], -1, 1)
        Xv = torch.from_numpy(np.asarray(Xv, np.float32))
        first = torch.cat([(emb(Xi[:, f, :]).sum(1).t() * Xv[:, f]).t()
                           for f, emb in enumerate(self.first_order_embeddings)], 1)
        e = [emb(Xi[:, f, :]).sum(1).t() * Xv[:, f] for f, emb in enumerate(self.second_order_embeddings)]
        S = sum(e)
        Q = sum([x * x for x in e])
        bi = ((S * S - Q) * 0.5).t()
        return torch.sum(first, 1) + torch.sum(bi, 1) + self.bias

    def step(self, opt, Xi, Xv, Y, loss_of_sigmoid):
        opt.zero_grad()
        z = self.forward_fm(Xi, Xv)
        loss = F.binary_cross_entropy_with_logits(torch.sigmoid(z) if loss_of_sigmoid else z, torch.from_numpy(Y))
        loss.backward()
        opt.step()
        return np.float32(loss.detach().item())

    def tables(self):
        """(V [R,k], w1 [R], bias [1]) as float32 arrays"""
        V = torch.cat([e.weight.detach() for e in self.second_order_embeddings]).numpy()
        w1 = torch.cat([e.weight.detach() for e in self.first_order_embeddings])[:, 0].numpy()
        return np.ascontiguousarray(V), np.ascontiguousarray(w1), self.bias.detach().numpy().reshape(1)

    def adagrad_sums(self, opt):
        """Adagrad's state_sum of the tables and the bias, in the layout of tables()"""
        st = lambda p: opt.state[p]["sum"].detach()
        sV = torch.cat([st(e.weight) for e in self.second_order_embeddings]).numpy()
        sw1 = torch.cat([st(e.weight) for e in self.first_order_embeddings])[:, 0].numpy()
        return np.ascontiguousarray(sV), np.ascontiguousarray(sw1), st(self.bias).numpy().reshape(1)


def adagrad(model, lr, eps=1e-10, init=0.0):
    return torch.optim.Adagrad(model.parameters(), lr=float(np.float32(lr)), eps=eps, initial_accumulator_value=init,
                               foreach=False)
