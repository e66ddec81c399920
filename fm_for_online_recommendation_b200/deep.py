"""Drop-in replacements for the reference's deep FM family (models/models_online_deep/*.py).

Same class names, constructor kwargs, method names, argument meaning and return types as
`FMAdam` (fm_adam.py), `DeepFMAdam` (deepfm_adam.py), `NFMAdam` (nfm_adam.py), `DeepFMOnn`
(deepfm_onn.py) and `NFMOnn` (nfm_onn.py); every method body is a call sequence into
lib/libfmb200.so (include/fmb200.h).  There is no CPU path: constructing a model without a visible
CUDA device raises `FmbError`.

Layout: one packed device table [R, rowp] (rowp = round_up(k+1, 16): 64-byte aligned rows) holds, per global row, the
second-order embedding (k floats), the first-order weight and padding.
`second_order_embeddings[f].weight` / `first_order_embeddings[f].weight` are strided Parameter
views into it, `hidden_layers[l].weight/.bias` are views into one flat MLP buffer, so
`parameters()`, `state_dict()`, `str()` and `pickle` keep working (SURVEY.md section 8b).

Semantics follow the reference's CPU path (`use_cuda=False`): the bias IS trained (SURVEY.md
fact 6); "Adam" is the per-call fresh-state sign step (fact 1).
"""
import ctypes as C
from time import time

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import AdagradState, FmbError, RunList, SparseAdamState, check, ptr

UPDATE_ADAM1, UPDATE_SGD, UPDATE_FTRL = 0, 1, 2   # 2: per-coordinate FTRL-Proximal (enable_ftrl), FM-only steps
UPDATE_ADAGRAD = 3   # torch.optim.Adagrad with state kept across calls (enable_adagrad): FM steps, tower fit, run_experiment
UPDATE_SPARSE_ADAM = 4   # torch.optim.SparseAdam on the tables + torch.optim.Adam on the bias and the tower, state kept
                         # across calls (enable_sparse_adam): FM steps, tower fit, run_experiment
LOSS_LOGITS, LOSS_LOGITS_OF_SIG = 0, 1


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class EncodedBatch:
    """Device-resident inputs (SURVEY.md 8f.1): ids int32 [B,F] global row ids, xv fp32 [B,F] or None
    (all ones), y fp32 [B] or None."""

    __slots__ = ("ids", "xv", "y", "B", "feature_sizes")

    def __init__(self, ids, xv, y, feature_sizes=None):
        self.ids, self.xv, self.y, self.B = ids, xv, y, ids.shape[0]
        self.feature_sizes = feature_sizes   # set by data.DeviceDataset: the table layout the global ids were built for


class _ViewEmbedding(nn.Embedding):
    """nn.Embedding whose weight is a strided view into the packed table (no separate storage)."""

    def __init__(self, view):
        nn.Module.__init__(self)
        self.num_embeddings, self.embedding_dim = view.shape
        self.padding_idx = None
        self.max_norm = None
        self.norm_type = 2.0
        self.scale_grad_by_freq = False
        self.sparse = False
        self.weight = nn.Parameter(view, requires_grad=True)


class _ViewLinear(nn.Linear):
    def __init__(self, wview, bview):
        nn.Module.__init__(self)
        self.out_features, self.in_features = wview.shape
        self.weight = nn.Parameter(wview, requires_grad=True)
        self.bias = nn.Parameter(bview, requires_grad=True)


def _rebuild(cls, kwargs, state):
    m = cls(**kwargs)
    m._load_packed_state(state)
    return m


def _f32(t):
    return None if t is None else t.detach().cpu()


class _DeepBase(nn.Module):
    _NAME = ""
    _HAS_MLP = True
    _IS_ONN = False
    _IS_NFM = False

    # ------------------------------------------------------------------ construction
    def _setup(self, feature_sizes, embedding_size, num_hidden_layers, neuron_per_hidden_layer, batch_size,
               num_classes, b, n, s, use_cuda, update_mode):
        self._lib = _lib.require_cuda()  # raises: no CPU fallback
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.field_size = len(feature_sizes)
        self.feature_sizes = feature_sizes
        self.embedding_size = embedding_size
        self.num_classes = num_classes
        self.dtype = torch.long
        self.update_mode = update_mode
        F, k = self.field_size, embedding_size
        if self._HAS_MLP:
            self.num_hidden_layers = num_hidden_layers
            self.neuron_per_hidden_layer = neuron_per_hidden_layer
        self._L = num_hidden_layers if self._HAS_MLP else 0
        self._H = neuron_per_hidden_layer if self._HAS_MLP else 0
        if self._HAS_MLP and not (self._IS_NFM and not self._IS_ONN):
            self.batch_size = batch_size  # NFMAdam has no batch_size attribute (nfm_adam.py:13-27)
        self._batch_size = batch_size
        self._rowp = self._lib.fmb_rowp(k)
        self._kp4 = self._lib.fmb_kp4(k)
        sizes = np.asarray(list(feature_sizes), dtype=np.int64)
        self._feature_sizes_t = tuple(int(v) for v in sizes)
        self._offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self._R = int(self._offsets_np[-1])
        if self._R >= 2 ** 31:
            raise ValueError("total rows must fit int32")
        self._key_bits = max(1, int(self._R - 1).bit_length())
        self._offsets_dev = torch.from_numpy(self._offsets_np[:-1].copy()).to(self.device)
        self._sizes_dev = torch.from_numpy(sizes.copy()).to(self.device)
        self._field_off_dev = torch.from_numpy(self._offsets_np.astype(np.int32)).to(self.device)

        # parameters are drawn on the CPU in the reference's order so torch.manual_seed(s) gives the
        # same initial model as the reference (fm_adam.py:26-32, deepfm_onn.py:30-53)
        if self._IS_ONN:
            bias0 = torch.rand(1)                       # deepfm_onn.py:30
        else:
            bias0 = torch.tensor(b)                     # fm_adam.py:26
        self.bias = nn.Parameter(bias0.to(self.device))
        if self._IS_ONN:
            self.b = nn.Parameter(torch.tensor(b).to(self.device))
        self.n = nn.Parameter(torch.tensor(n).to(self.device), requires_grad=False)
        if self._IS_ONN:
            self.s = nn.Parameter(torch.tensor(s).to(self.device), requires_grad=False)
        self._lr = float(np.float32(n))
        self._hb = float(np.float32(b))
        self._hs = float(np.float32(s))

        table = torch.zeros(self._R, self._rowp, dtype=torch.float32)
        fo = [nn.Embedding(int(fs), 1) for fs in sizes]
        so = [nn.Embedding(int(fs), k) for fs in sizes]
        with torch.no_grad():
            for f in range(F):
                lo, hi = int(self._offsets_np[f]), int(self._offsets_np[f + 1])
                table[lo:hi, :k] = so[f].weight
                table[lo:hi, k] = fo[f].weight[:, 0]
        del fo, so
        self._table = table.to(self.device)
        self._bind_embeddings()

        if self._HAS_MLP:
            lins = [nn.Linear(k, self._H)] + [nn.Linear(self._H, self._H) for _ in range(self._L - 1)]
            flat = torch.cat([torch.cat([l.weight.detach().reshape(-1), l.bias.detach()]) for l in lins])
            self._mlp = flat.to(self.device).contiguous()
            self._bind_mlp()
        else:
            self._mlp = None
        if self._IS_ONN:
            self.alpha = nn.Parameter(torch.full((self._L,), 1.0 / (self._L + 1), device=self.device),
                                      requires_grad=False)
        self._session = None
        self._session_cap = 0
        self._presorted = None   # the EncodedBatch whose sorted form the session holds (kept alive: its ids pointer is the key)
        self._ws = {}
        self._ada = None
        self._sa = None
        if update_mode == UPDATE_ADAGRAD:
            self.enable_adagrad()
        elif update_mode == UPDATE_SPARSE_ADAM:
            self.enable_sparse_adam()

    def _bind_embeddings(self):
        k = self.embedding_size
        fo, so = [], []
        for f in range(self.field_size):
            lo, hi = int(self._offsets_np[f]), int(self._offsets_np[f + 1])
            so.append(_ViewEmbedding(self._table[lo:hi, :k]))
            fo.append(_ViewEmbedding(self._table[lo:hi, k:k + 1]))
        self.first_order_embeddings = nn.ModuleList(fo)
        self.second_order_embeddings = nn.ModuleList(so)

    def _bind_mlp(self):
        k, H = self.embedding_size, self._H
        mods, o = [], 0
        for l in range(self._L):
            nin = k if l == 0 else H
            w = self._mlp[o:o + H * nin].view(H, nin)
            o += H * nin
            c = self._mlp[o:o + H]
            o += H
            mods.append(_ViewLinear(w, c))
        self.hidden_layers = nn.ModuleList(mods)

    def _apply(self, fn, recurse=True):
        """nn.Module.to()/.cpu()/.double()/.half() would re-create the Parameters away from the packed table the kernels
        train (the views would silently stop being the model): the classes live on the device they were built on."""
        raise RuntimeError("fm_for_online_recommendation_b200 models are bound to their CUDA device and to fp32: "
                           ".to()/.cpu()/.cuda()/.double() are not supported (pickle the model to move it)")

    # ------------------------------------------------------------------ persistence
    def _ctor_kwargs(self):
        raise NotImplementedError

    def _export_state(self):
        st = {"table": self._table.detach().cpu(), "bias": self.bias.detach().cpu()}
        if self._mlp is not None:
            st["mlp"] = self._mlp.detach().cpu()
        if self._IS_ONN:
            st["alpha"] = self.alpha.detach().cpu()
        if self.update_mode == UPDATE_ADAGRAD:
            st["adagrad"] = {"eps": self._ada_eps, "sums": _f32(self._ada_sums), "bias_sum": _f32(self._ada_bias),
                             "mlp_sums": _f32(self._ada_mlp)}
        if self.update_mode == UPDATE_SPARSE_ADAM:
            a = self._sa
            st["sparse_adam"] = {"betas": (a.beta1, a.beta2), "eps": a.eps, "step": a.step, "mlp_step": a.mlp_step,
                                 "mv": _f32(self._sa_mv), "bias_mv": _f32(self._sa_bias), "mlp_mv": _f32(self._sa_mlp)}
        return st

    def _load_packed_state(self, st):
        with torch.no_grad():
            self._table.copy_(st["table"])
            self.bias.copy_(st["bias"])
            if self._mlp is not None:
                self._mlp.copy_(st["mlp"])
            if self._IS_ONN:
                self.alpha.copy_(st["alpha"])
        ada = st.get("adagrad")
        if ada is not None:
            self.enable_adagrad(eps=ada["eps"])
            with torch.no_grad():
                self._ada_sums.copy_(ada["sums"])
                self._ada_bias.copy_(ada["bias_sum"])
                if self._ada_mlp is not None:
                    self._ada_mlp.copy_(ada["mlp_sums"])
        sa = st.get("sparse_adam")
        if sa is not None:
            self.enable_sparse_adam(betas=sa["betas"], eps=sa["eps"])
            self._sa.step, self._sa.mlp_step = sa["step"], sa["mlp_step"]
            with torch.no_grad():
                self._sa_mv.copy_(sa["mv"])
                self._sa_bias.copy_(sa["bias_mv"])
                if self._sa_mlp is not None:
                    self._sa_mlp.copy_(sa["mlp_mv"])

    def __reduce__(self):  # pickle.dump(model) (main_experiment.py:160-162): one copy of the table, no handles
        return (_rebuild, (type(self), self._ctor_kwargs(), self._export_state()))

    def __del__(self):
        try:
            if getattr(self, "_session", None):
                self._lib.fmb_session_destroy(self._session)
                self._session = None
        except Exception:
            pass

    # ------------------------------------------------------------------ inputs
    def encode(self, Xi, Xv=None, Y=None):
        """lists / ndarrays / tensors -> EncodedBatch on the device. Xi holds per-field local ids."""
        if isinstance(Xi, EncodedBatch):
            if Xi.feature_sizes is not None and tuple(Xi.feature_sizes) != self._feature_sizes_t:
                raise IndexError("index out of range in self: the batch was encoded for other feature_sizes")
            return Xi
        F = self.field_size
        if torch.is_tensor(Xi):
            loc = Xi.to(self.device).reshape(-1, F).to(torch.int64)
            # same failure as nn.Embedding in the reference: an out-of-range id must raise, never gather out of bounds
            if loc.numel() and bool(((loc < 0) | (loc >= self._sizes_dev)).any()):
                raise IndexError("index out of range in self")
            ids = (loc + self._offsets_dev).to(torch.int32)
        else:
            a = np.asarray(Xi, dtype=np.int64).reshape(-1, F)
            if a.size and (a.min() < 0 or (a >= (self._offsets_np[1:] - self._offsets_np[:-1])[None, :]).any()):
                raise IndexError("index out of range in self")  # what nn.Embedding raises in the reference
            ids = torch.from_numpy((a + self._offsets_np[:-1][None, :]).astype(np.int32)).to(self.device)
        ids = ids.contiguous()
        xv = None
        if Xv is not None:
            if torch.is_tensor(Xv):
                xv = Xv.to(self.device, torch.float32).reshape(-1, F).contiguous()
            else:
                v = np.asarray(Xv, dtype=np.float32).reshape(-1, F)
                if not np.all(v == 1.0):  # all-ones values (Criteo, data_preprocess.py:41) need no upload
                    xv = torch.from_numpy(np.ascontiguousarray(v)).to(self.device)
        y = None
        if Y is not None:
            if torch.is_tensor(Y):
                y = Y.to(self.device, torch.float32).reshape(-1).contiguous()
            else:
                y = torch.from_numpy(np.asarray(Y, dtype=np.float32).reshape(-1)).to(self.device)
        return EncodedBatch(ids, xv, y)

    def enable_ftrl(self, beta=1.0, l1=0.0, l2=0.0):
        """Switch update_embedding / FMAdam.fit to per-coordinate FTRL-Proximal (z, n, w; SURVEY.md 8f.4): alpha is the
        learning rate `n`.  The state starts at n = 0 with z chosen so that the closed form reproduces the current
        weights (warm start).  The reference's own FM_FTRL is the unregularised linearised form
        (models/models_online/FM_FTRL.py:76-80) and lives in classical.py; this mode is the McMahan update the
        north_star names, off by default."""
        k, rp = self.embedding_size, self._rowp
        self.update_mode = UPDATE_FTRL
        self._ftrl = (float(np.float32(beta)), float(np.float32(l1)), float(np.float32(l2)))
        c = np.float32(np.float32(beta) / np.float32(self._lr) + np.float32(l2))
        z0 = lambda w: (-(w * c) - np.sign(w) * np.float32(l1)).astype(np.float32)
        w = self._table.detach().cpu().numpy()
        zn = np.zeros((self._R, 2, rp), np.float32)
        zn[:, 0, :k + 1] = z0(w[:, :k + 1])
        self._ftrl_zn = torch.from_numpy(zn).to(self.device)
        self._ftrl_bias = torch.from_numpy(np.array([z0(self.bias.detach().cpu().numpy().reshape(1))[0], 0.0],
                                                    np.float32)).to(self.device)
        if self._session is not None:
            self._bind_ftrl()

    def _bind_ftrl(self):
        check(self._lib.fmb_session_set_ftrl(self._session, ptr(self._ftrl_zn), ptr(self._ftrl_bias), *self._ftrl),
              "fmb_session_set_ftrl")

    def enable_adagrad(self, eps=1e-10, initial_accumulator_value=0.0):
        """Switch update_embedding, fit (FMAdam / DeepFMAdam / NFMAdam) and run_experiment to torch.optim.Adagrad: the
        same trajectory as ONE `torch.optim.Adagrad(model.parameters(), lr=n, eps=eps,
        initial_accumulator_value=initial_accumulator_value)` kept across calls in place of the reference's per-call
        Adam.  Only the rows a batch hits are updated: a zero gradient leaves Adagrad's weight and sum as they are, so this
        is the dense optimizer exactly.  The sums (one per coordinate of the table, the bias and the tower) start at
        `initial_accumulator_value`; calling this again resets them.  The ONN classes' hedge fit uses no optimizer and
        stays as it is."""
        v = float(np.float32(initial_accumulator_value))
        if v < 0:
            raise ValueError("initial_accumulator_value must be >= 0")
        self.update_mode = UPDATE_ADAGRAD
        self._ada_eps = float(np.float32(eps))
        self._ada_sums = torch.full((self._R, self._rowp), v, dtype=torch.float32, device=self.device)
        self._ada_bias = torch.full((1,), v, dtype=torch.float32, device=self.device)
        self._ada_mlp = None if self._mlp is None else torch.full_like(self._mlp, v)
        self._ada = AdagradState(self._ada_sums.data_ptr(), self._ada_bias.data_ptr(),
                                 None if self._ada_mlp is None else self._ada_mlp.data_ptr(), self._ada_eps)
        self.__dict__.pop("_fit_graphs", None)   # captured fits hold the previous state's pointers
        if self._session is not None:
            self._bind_adagrad()

    def enable_sparse_adam(self, betas=(0.9, 0.999), eps=1e-8):
        """Switch update_embedding, fit (FMAdam / DeepFMAdam / NFMAdam) and run_experiment to Adam with its moments kept
        across calls: the same trajectory as ONE `torch.optim.SparseAdam(<embedding tables>, lr=n, betas, eps)` stepped on
        the sparse gradient of the rows each batch hits (nn.Embedding(sparse=True)'s, summed in sample order) and ONE
        `torch.optim.Adam([bias] + <tower>, lr=n, betas, eps)`.  Every row a batch hits steps, also when its gradient is
        zero; the other rows keep their weights and moments.  The tables and the bias count every step, the tower only
        the steps that give it a gradient (fit, run_experiment), as torch does.  Calling this again resets the moments and
        both counters.  The ONN classes' hedge fit uses no optimizer and stays as it is."""
        b1, b2 = (float(b) for b in betas)
        if not (0.0 <= b1 < 1.0 and 0.0 <= b2 < 1.0) or eps < 0:
            raise ValueError("need 0 <= beta1, beta2 < 1 and eps >= 0")
        self.update_mode = UPDATE_SPARSE_ADAM
        self._sa_mv = torch.zeros((self._R, 2, self._rowp), dtype=torch.float32, device=self.device)
        self._sa_bias = torch.zeros((2,), dtype=torch.float32, device=self.device)
        self._sa_mlp = None if self._mlp is None else torch.zeros((2, self._mlp.numel()), dtype=torch.float32,
                                                                  device=self.device)
        self._sa = SparseAdamState(self._sa_mv.data_ptr(), self._sa_bias.data_ptr(),
                                   None if self._sa_mlp is None else self._sa_mlp.data_ptr(), b1, b2, float(np.float32(eps)),
                                   0, 0)
        self.__dict__.pop("_fit_graphs", None)
        if self._session is not None:
            self._bind_sparse_adam()

    def _bind_sparse_adam(self):
        check(self._lib.fmb_session_set_sparse_adam(self._session, C.byref(self._sa)), "fmb_session_set_sparse_adam")

    def _ada_arg(self):
        """the state slot of the C entry points: fmb_adagrad_t in mode 3, fmb_sparse_adam_t in mode 4, else NULL"""
        if self.update_mode == UPDATE_ADAGRAD and self._ada is not None:
            return C.byref(self._ada)
        if self.update_mode == UPDATE_SPARSE_ADAM and self._sa is not None:
            return C.byref(self._sa)
        return None

    def _bind_adagrad(self):
        check(self._lib.fmb_session_set_adagrad(self._session, ptr(self._ada_sums), ptr(self._ada_bias), self._ada_eps),
              "fmb_session_set_adagrad")

    def _get_session(self, B):
        if self._session is None or B > self._session_cap:
            if self._session is not None:
                torch.cuda.synchronize()
                self._lib.fmb_session_destroy(self._session)
            cap = max(B, 1)
            h = C.c_void_p()
            off32 = np.ascontiguousarray(self._offsets_np.astype(np.int32))
            check(self._lib.fmb_session_create(C.byref(h), self.field_size, self.embedding_size, cap,
                                               off32.ctypes.data_as(C.c_void_p)), "fmb_session_create")
            self._session, self._session_cap = h, cap
            self._presorted = None
            if self.update_mode == UPDATE_FTRL:
                self._bind_ftrl()
            elif self.update_mode == UPDATE_ADAGRAD:
                self._bind_adagrad()
            elif self.update_mode == UPDATE_SPARSE_ADAM:
                self._bind_sparse_adam()
        return self._session

    def _buf(self, name, shape, dtype=torch.float32):
        t = self._ws.get(name)
        n = int(np.prod(shape))
        if t is None or t.numel() < n or t.dtype != dtype:
            if t is not None:
                # the fit graphs captured so far point into the buffer this one replaces, which goes back to torch's
                # allocator: drop them, the next calls capture again.  A capture re-runs a configuration whose eager
                # call already sized every buffer, so it never gets here.
                if torch.cuda.is_current_stream_capturing():
                    raise RuntimeError(f"workspace '{name}' would grow inside a CUDA graph capture")
                self.__dict__.pop("_fit_graphs", None)
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._ws[name] = t
        return t[:n].view(*shape)

    # ------------------------------------------------------------------ forward pieces (A1-A5)
    def _fm_forward(self, e, first=False, S=False, bi=False, sum_first=False, z=True):
        B, F, k = e.B, self.field_size, self.embedding_size
        out = {}
        if first:
            out["first"] = torch.empty(B, F, device=self.device)
        if S:
            out["S"] = self._buf("S", (B, self._kp4))
        if bi:
            out["bi"] = torch.empty(B, k, device=self.device)
        if sum_first:
            out["sum_first"] = self._buf("sum_first", (B,))
        if z:
            out["z"] = torch.empty(B, device=self.device)
        check(self._lib.fmb_fm_forward(ptr(e.ids), ptr(e.xv), ptr(self._table), ptr(self.bias), B, F, k,
                                       ptr(out.get("first")), ptr(out.get("S")), ptr(out.get("bi")),
                                       ptr(out.get("sum_first")), ptr(out.get("z")), None, 0, None, None, _stream()),
              "fmb_fm_forward")
        return out

    def first_order(self, Xi, Xv):
        return self._fm_forward(self.encode(Xi, Xv), first=True, z=False)["first"]

    def second_order(self, Xi, Xv):
        return self._fm_forward(self.encode(Xi, Xv), bi=True, z=False)["bi"]

    def forward_fm(self, Xi, Xv):
        return self._fm_forward(self.encode(Xi, Xv))["z"]

    def _mlp_forward(self, bi, B):
        L, H, k = self._L, self._H, self.embedding_size
        act = self._buf("act", (L, B, H))
        head = self._buf("head", (L, B))
        check(self._lib.fmb_mlp_forward(ptr(bi), k, ptr(self._mlp), B, k, L, H, ptr(act), ptr(head), _stream()),
              "fmb_mlp_forward")
        return act, head

    def _full_forward(self, e, need_S=False):
        """returns dict with z (logit, or last-head probability for ONN) and the intermediates."""
        if not self._HAS_MLP:
            o = self._fm_forward(e, S=need_S)
            return o
        o = self._fm_forward(e, S=need_S, bi=True, sum_first=True)
        B = e.B
        act, head = self._mlp_forward(o["bi"], B)
        o["act"], o["head"] = act, head
        nfm = 1 if self._IS_NFM else 0
        if self._IS_ONN:
            p = torch.empty(self._L, B, device=self.device)
            check(self._lib.fmb_onn_heads(nfm, ptr(o["z"]), ptr(o["sum_first"]), ptr(self.bias), ptr(head), self._L,
                                          B, ptr(p), _stream()), "fmb_onn_heads")
            o["players"] = p
            o["z_fm"], o["z"] = o["z"], p[self._L - 1]
        else:
            z = torch.empty(B, device=self.device)
            check(self._lib.fmb_combine_logit(nfm, ptr(o["z"]), ptr(o["sum_first"]), ptr(self.bias),
                                              ptr(head[self._L - 1]), B, ptr(z), _stream()), "fmb_combine_logit")
            o["z_fm"], o["z"] = o["z"], z
        return o

    def forward(self, Xi, Xv):
        o = self._full_forward(self.encode(Xi, Xv))
        if self._IS_ONN:
            return o["z"], o["players"]
        return o["z"]

    # ------------------------------------------------------------------ training steps (A6, A7)
    def _fm_step(self, e, loss_kind, next_batch=None):
        """One FM-only step on EncodedBatch `e`.  `next_batch` (an EncodedBatch of the same size, optional) is the
        batch the following call will step on: its sort rides along with this step (SURVEY.md 8f.1)."""
        if e.y is None:
            raise ValueError("labels required")
        s = self._get_session(e.B)
        if self._presorted is not None and self._presorted is not e:
            self._lib.fmb_session_presort_invalidate(s)   # a pre-sort is only ever honoured for the very same batch object
        nxt = next_batch if (next_batch is not None and next_batch.B == e.B) else None
        loss = torch.empty((), device=self.device)
        check(self._lib.fmb_session_fm_step_next(s, ptr(e.ids), ptr(e.xv), ptr(e.y), e.B, ptr(self._table),
                                                 ptr(self.bias), self._key_bits, loss_kind, self._lr, self.update_mode,
                                                 ptr(nxt.ids) if nxt is not None else None, ptr(loss), _stream()),
              "fmb_session_fm_step_next")
        self._presorted = nxt
        return loss

    _UE_LOSS = LOSS_LOGITS
    _FIT_LOSS = LOSS_LOGITS_OF_SIG

    def presort(self, batch):
        """Start sorting the ids of `batch` (an EncodedBatch that will be passed to the NEXT update_embedding /
        FMAdam.fit) on a side stream, overlapping the step in flight (the sort depends on the ids only)."""
        s = self._get_session(batch.B)
        check(self._lib.fmb_session_presort(s, ptr(batch.ids), batch.B, self._key_bits), "fmb_session_presort")
        self._presorted = batch

    def update_embedding(self, Xi, Xv, Y, next_batch=None):
        """fm_adam.py:56-69 and the same method of the other four classes: loss on forward_fm only.
        `next_batch` (extension, optional): the EncodedBatch the next call will be given."""
        self.train()
        return self._fm_step(self.encode(Xi, Xv, Y), self._UE_LOSS, next_batch)

    def _sort(self, e, with_runlist=False):
        """Stable sort of the batch's row ids -> (sorted keys, permutation[, run list]).  with_runlist (per-field sort only):
        also the run list the run kernel consumes (one warp per run, long runs first)."""
        N = e.B * self.field_size
        sk = self._buf("skeys", (N,), torch.int32)
        pm = self._buf("perm", (N,), torch.int32)
        if e.B <= self._lib.fmb_sort_fields_max_batch():
            if with_runlist:
                nseg, cap = C.c_int(), C.c_int()
                self._lib.fmb_runlist_shape(e.B, self.field_size, C.byref(nseg), C.byref(cap))
                ent = self._buf("rl_entries", (nseg.value * cap.value, 4), torch.int32)
                cnt = self._buf("rl_counts", (2 * nseg.value,), torch.int32)
                self._rl = RunList(ent.data_ptr(), cnt.data_ptr(), nseg.value, cap.value)
                check(self._lib.fmb_sort_fields_ex(ptr(e.ids), e.B, self.field_size, ptr(self._field_off_dev), ptr(sk),
                                                   ptr(pm), None, C.byref(self._rl), 0, _stream()), "fmb_sort_fields_ex")
                return sk, pm, self._rl
            check(self._lib.fmb_sort_fields(ptr(e.ids), e.B, self.field_size, ptr(self._field_off_dev), ptr(sk),
                                            ptr(pm), _stream()), "fmb_sort_fields")
            return (sk, pm, None) if with_runlist else (sk, pm)
        wsb = self._lib.fmb_sort_workspace_bytes(N)
        ws = self._buf("sort_ws", (wsb,), torch.uint8)
        check(self._lib.fmb_sort_segment(ptr(e.ids), N, self._key_bits, ptr(ws), wsb, ptr(sk), ptr(pm), None, None,
                                         _stream()), "fmb_sort_segment")
        return (sk, pm, None) if with_runlist else (sk, pm)

    def _deep_fit(self, e):
        """DeepFMAdam.fit / NFMAdam.fit (deepfm_adam.py:106-117, nfm_adam.py:105-116)."""
        B, F, k, L, H = e.B, self.field_size, self.embedding_size, self._L, self._H
        lib, st = self._lib, _stream()
        # the sort depends on the ids only: side stream, beside the forward pass and the tower's backward
        main = torch.cuda.current_stream()
        if getattr(self, "_sort_stream", None) is None:
            self._sort_stream = torch.cuda.Stream(device=self.device)
        self._sort_stream.wait_stream(main)
        with torch.cuda.stream(self._sort_stream):
            sk, pm, rl = self._sort(e, with_runlist=True)
        o = self._full_forward(e, need_S=True)
        delta = self._buf("delta", (B,))
        check(lib.fmb_loss_delta(self._FIT_LOSS, ptr(o["z"]), ptr(e.y), B, ptr(delta), None, st), "fmb_loss_delta")
        gmlp = self._buf("gmlp", (self._mlp.numel(),))
        gbi = self._buf("gbi", (B, self._kp4))
        wsb = lib.fmb_mlp_bwd_workspace_bytes(B, H)
        ws = self._buf("mlp_ws", (wsb,), torch.uint8)
        check(lib.fmb_mlp_backward(ptr(o["bi"]), k, ptr(self._mlp), ptr(o["act"]), ptr(delta), L - 1, B, k, L, H,
                                   ptr(gmlp), ptr(gbi), self._kp4, ptr(ws), wsb, st), "fmb_mlp_backward")
        main.wait_stream(self._sort_stream)
        N = B * F
        bwsb = lib.fmb_bwd_workspace_bytes(N, k)
        bws = self._buf("bwd_ws", (bwsb,), torch.uint8)
        ada = self._ada_arg()   # the _ex forms are the plain ones outside modes 3 and 4
        sa = self.update_mode == UPDATE_SPARSE_ADAM
        if sa:
            check(lib.fmb_sparse_adam_advance(ada, self._lr, 1), "fmb_sparse_adam_advance")
        check(lib.fmb_fm_backward_update_rl_ex(ptr(sk), ptr(pm), N, N, ptr(e.xv), ptr(self._table), F, k, ptr(o["S"]),
                                               self._kp4, ptr(delta), 1, 0 if self._IS_NFM else 1, ptr(gbi), 0x7FFFFFFF,
                                               self._lr, self.update_mode, ada, C.byref(rl) if rl is not None else None,
                                               ptr(bws), bwsb, st), "fmb_fm_backward_update")
        if sa:
            check(lib.fmb_update_dense_adam(ptr(self._mlp), ptr(gmlp), self._mlp.numel(), ada, st), "fmb_update_dense_adam")
        else:
            check(lib.fmb_update_dense_ex(ptr(self._mlp), ptr(gmlp), self._mlp.numel(), self._lr, self.update_mode,
                                          ptr(self._ada_mlp) if ada else None, self._ada_eps if ada else 0.0, st),
                  "fmb_update_dense")
        check(lib.fmb_finish_step_ex(ptr(delta), None, B, ptr(self.bias), self._lr, self.update_mode, ada, None, st),
              "fmb_finish_step")

    def _deep_fit_graphed(self, e):
        """_deep_fit as ONE CUDA graph per configuration: the step is ~25 kernel launches through ctypes, which the host
        submits more slowly than the GPU runs them at cfg4's shapes.  First call of a configuration: eager (allocations,
        function attributes); second: captured on static input buffers; afterwards: copy the batch in, replay."""
        # mode 4: every step has scalars of its own (taken by value at launch), so it is not replayed from a graph
        if torch.cuda.is_current_stream_capturing() or self.update_mode == UPDATE_SPARSE_ADAM:
            return self._deep_fit(e)
        key = (e.B, e.xv is not None, self._lr, self.update_mode, int(self._lib.fmb_tensor_cores_enabled()))
        ent = self.__dict__.get("_fit_graphs", {}).get(key)
        if ent is None:
            self._deep_fit(e)   # may grow a workspace, which drops every graph captured so far (_buf)
            self.__dict__.setdefault("_fit_graphs", {})[key] = "warm"
            return
        if ent == "warm":
            se = EncodedBatch(torch.empty_like(e.ids), None if e.xv is None else torch.empty_like(e.xv), torch.empty_like(e.y))
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                self._deep_fit(se)
            ent = self._fit_graphs[key] = (g, se)
        g, se = ent
        se.ids.copy_(e.ids, non_blocking=True)
        if se.xv is not None:
            se.xv.copy_(e.xv, non_blocking=True)
        se.y.copy_(e.y, non_blocking=True)
        g.replay()

    def _hedge_fit(self, e):
        """DeepFMOnn.fit / NFMOnn.fit (deepfm_onn.py:109-154): hedge backpropagation; only the tower and
        alpha change."""
        B, k, L, H = e.B, self.embedding_size, self._L, self._H
        if B != self._batch_size:
            raise RuntimeError(f"shape '[{self._batch_size}]' is invalid for input of size {B}")  # out.view(batch_size)
        lib, st = self._lib, _stream()
        o = self._full_forward(e)
        lossv = self._buf("lossv", (B,))
        loss_sum = self._buf("loss_sum", (L,))
        acc = self._buf("hedge_acc", (self._mlp.numel(),))
        wsb = lib.fmb_mlp_bwd_workspace_bytes(B, H)
        ws = self._buf("mlp_ws", (wsb,), torch.uint8)
        if self._hedge_single_pass(B):
            # towers on the tensor cores (cfg4: B = 8 192, H = 400): ONE backward pass with alpha_i * dL_i/d(head_i) injected at
            # every head instead of L passes of growing depth (SURVEY.md A7; half the products at L = 3)
            gtop_all = self._buf("gtop_all", (L, B))
            for i in range(L):
                check(lib.fmb_hedge_head_grad(ptr(o["players"][i]), ptr(e.y), B, ptr(gtop_all[i]), ptr(lossv), st),
                      "fmb_hedge_head_grad")
                check(lib.fmb_sum_aten(ptr(lossv), B, ptr(loss_sum[i:]), st), "fmb_sum_aten")
            check(lib.fmb_mlp_backward_hedge(ptr(o["bi"]), k, ptr(self._mlp), ptr(o["act"]), ptr(gtop_all), ptr(self.alpha),
                                             B, k, L, H, ptr(acc), ptr(ws), wsb, st), "fmb_mlp_backward_hedge")
        else:
            gtop = self._buf("delta", (B,))
            gmlp = self._buf("gmlp", (self._mlp.numel(),))
            for i in range(L):
                check(lib.fmb_hedge_head_grad(ptr(o["players"][i]), ptr(e.y), B, ptr(gtop), ptr(lossv), st),
                      "fmb_hedge_head_grad")
                check(lib.fmb_sum_aten(ptr(lossv), B, ptr(loss_sum[i:]), st), "fmb_sum_aten")
                check(lib.fmb_mlp_backward(ptr(o["bi"]), k, ptr(self._mlp), ptr(o["act"]), ptr(gtop), i, B, k, L, H,
                                           ptr(gmlp), None, 0, ptr(ws), wsb, st), "fmb_mlp_backward")
                check(lib.fmb_hedge_accumulate(ptr(acc), ptr(gmlp), ptr(self.alpha), i, k, L, H, st),
                      "fmb_hedge_accumulate")
        check(lib.fmb_hedge_apply(ptr(self._mlp), ptr(acc), self._lr, ptr(self.alpha), ptr(loss_sum), B, k, L, H,
                                  self._hb, self._hs, st), "fmb_hedge_apply")

    def _hedge_single_pass(self, B):
        """single-pass hedge backward only where the tower's H x H products are on the tensor cores (already within
        tolerance rather than bit-exact); FMB_HEDGE_SINGLE=0/1 forces it off/on (tests)."""
        env = __import__("os").environ.get("FMB_HEDGE_SINGLE")
        if env is not None:
            return env == "1"
        return bool(self._lib.fmb_tensor_cores_enabled()) and self._L > 1 and \
            B * self._H * self._H >= (1 << self._lib.fmb_tensor_core_threshold_log2())

    def _hedge_fit_graphed(self, e):
        """_hedge_fit as one CUDA graph per configuration when it takes the single-pass route (large towers: ~40 launches
        through ctypes otherwise); same scheme as _deep_fit_graphed."""
        if torch.cuda.is_current_stream_capturing() or not self._hedge_single_pass(e.B):
            return self._hedge_fit(e)
        key = ("hedge", e.B, e.xv is not None, self._lr)
        ent = self.__dict__.get("_fit_graphs", {}).get(key)
        if ent is None:
            self._hedge_fit(e)   # may grow a workspace, which drops every graph captured so far (_buf)
            self.__dict__.setdefault("_fit_graphs", {})[key] = "warm"
            return
        if ent == "warm":
            se = EncodedBatch(torch.empty_like(e.ids), None if e.xv is None else torch.empty_like(e.xv), torch.empty_like(e.y))
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                self._hedge_fit(se)
            ent = self._fit_graphs[key] = (g, se)
        g, se = ent
        se.ids.copy_(e.ids, non_blocking=True)
        if se.xv is not None:
            se.xv.copy_(e.xv, non_blocking=True)
        se.y.copy_(e.y, non_blocking=True)
        g.replay()

    def fit(self, Xi, Xv, Y):
        self.train()
        e = self.encode(Xi, Xv, Y)
        if e.y is None:
            raise ValueError("labels required")
        if not self._HAS_MLP:
            self._fm_step(e, self._FIT_LOSS)
        elif self._IS_ONN:
            self._hedge_fit_graphed(e)
        else:
            self._deep_fit_graphed(e)

    # ------------------------------------------------------------------ predict / online loop (A8)
    def _predict_dev(self, e):
        z = self._full_forward(e)["z"].contiguous()
        out = torch.empty(e.B, dtype=torch.uint8, device=self.device)
        check(self._lib.fmb_predict(ptr(z), e.B, ptr(out), _stream()), "fmb_predict")
        return out

    def predict(self, Xi, Xv):
        self.eval()
        return self._predict_dev(self.encode(Xi, Xv)).cpu().numpy().astype(bool)

    def predict_proba(self, Xi, Xv):
        """torch.sigmoid(forward(...)) as a device tensor (extension, SURVEY.md 8f.2: scores for AUC / RMSE checks; the
        ONN classes return sigmoid of the last head's probability, exactly what their predict thresholds)."""
        self.eval()
        o = self._full_forward(self.encode(Xi, Xv))
        z = o["z"].contiguous()
        p = torch.empty_like(z)
        check(self._lib.fmb_sigmoid(ptr(z), z.numel(), ptr(p), _stream()), "fmb_sigmoid")
        return p

    _KIND_ID = 0

    def run_experiment(self, data_Xi, data_Xv, data_Y):
        """fm_adam.py:90-119: strictly sequential predict-then-fit per example, as one persistent kernel
        (csrc/online.cu); the bookkeeping below is the reference's, evaluated on the returned predictions."""
        data_size = len(data_Y)
        confusion_matrix = {"tp": 0, "fp": 0, "tn": 0, "fn": 0}
        accuracy = []
        roc = []
        start = time()
        enc = self.encode(data_Xi, data_Xv, data_Y)
        if self._IS_ONN and self._batch_size != 1:
            raise RuntimeError(f"shape '[{self._batch_size}]' is invalid for input of size 1")
        preds_dev = torch.empty(data_size, dtype=torch.uint8, device=self.device)
        conf_dev = torch.zeros(4, dtype=torch.int64, device=self.device)
        acc = self._buf("hedge_acc", (self._mlp.numel(),)) if self._IS_ONN else None
        if self.update_mode == UPDATE_SPARSE_ADAM and not self._IS_ONN:
            # the scalars of the data_size single-example steps, filled on the host (one row per example)
            tab = torch.empty(4 + 5 * data_size, dtype=torch.float32)
            check(self._lib.fmb_sparse_adam_online_steps(C.byref(self._sa), self._lr, int(self._HAS_MLP), data_size,
                                                         tab.data_ptr()), "fmb_sparse_adam_online_steps")
            steps_dev = tab.to(self.device)
            self._sa.steps_dev = steps_dev.data_ptr()
        check(self._lib.fmb_online_deep_run_ex(self._KIND_ID, ptr(enc.ids), ptr(enc.xv), ptr(enc.y), data_size,
                                               self.field_size, self.embedding_size, self._L, self._H, ptr(self._table),
                                               ptr(self.bias), ptr(self._mlp), ptr(getattr(self, "alpha", None)),
                                               ptr(acc), self._lr, self._hb, self._hs, self.update_mode, self._ada_arg(),
                                               ptr(preds_dev), ptr(conf_dev), _stream()), "fmb_online_deep_run")
        # bookkeeping of fm_adam.py:101-116: the kernel counted tp/fp/tn/fn as it went; the reference returns only the
        # LAST accuracy / roc entry, which are functions of the final counts (one 32-byte read, no per-sample host loop)
        tp, fp, tn, fn = (int(v) for v in conf_dev.cpu())
        confusion_matrix = {"tp": tp, "fp": fp, "tn": tn, "fn": fn}
        tpr = tp / (tp + fn + 1e-16)
        fpr = fp / (fp + tn + 1e-16)
        roc = [{'tpr': tpr, 'fpr': fpr}]
        accuracy = [(tp + tn) / data_size * 100]
        preds = preds_dev.cpu().numpy().astype(bool)
        time_elapsed = time() - start
        self._last_online_preds = preds
        return time_elapsed, accuracy[-1], roc[-1], confusion_matrix


class FMAdam(_DeepBase):
    """fm_adam.py:12-123."""
    _HAS_MLP = False

    def __init__(self, feature_sizes, embedding_size=4, num_classes=1, b=0.99, n=0.01, use_cuda=True,
                 update_mode=UPDATE_ADAM1):
        super().__init__()
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size, num_classes=num_classes, b=b,
                        n=n, use_cuda=use_cuda, update_mode=update_mode)
        self._setup(feature_sizes, embedding_size, 0, 0, 1, num_classes, b, n, 0.2, use_cuda, update_mode)

    def _ctor_kwargs(self):
        return self._kw

    def __str__(self):
        return f"FMAdam-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Classes{self.num_classes}"


class DeepFMAdam(_DeepBase):
    """deepfm_adam.py:12-159."""
    _KIND_ID = 1

    def __init__(self, feature_sizes, embedding_size=4, num_hidden_layers=2, neuron_per_hidden_layer=32,
                 batch_size=1, num_classes=1, b=0.99, n=0.01, use_cuda=True, update_mode=UPDATE_ADAM1):
        super().__init__()
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size,
                        num_hidden_layers=num_hidden_layers, neuron_per_hidden_layer=neuron_per_hidden_layer,
                        batch_size=batch_size, num_classes=num_classes, b=b, n=n, use_cuda=use_cuda,
                        update_mode=update_mode)
        self._setup(feature_sizes, embedding_size, num_hidden_layers, neuron_per_hidden_layer, batch_size,
                    num_classes, b, n, 0.2, use_cuda, update_mode)

    def _ctor_kwargs(self):
        return self._kw

    def __str__(self):
        return f"DeepFMAdam-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Hidden_Layers{self.num_hidden_layers}-Neuron_Per_Hidden_Layer{self.neuron_per_hidden_layer}-" \
               f"Num_Classes{self.num_classes}"


class NFMAdam(_DeepBase):
    """nfm_adam.py:12-158: update_embedding uses BCEWL(sigmoid(z_fm)) (:100), fit uses BCEWL(z) (:114)."""
    _IS_NFM = True
    _KIND_ID = 2
    _UE_LOSS = LOSS_LOGITS_OF_SIG
    _FIT_LOSS = LOSS_LOGITS

    def __init__(self, feature_sizes, embedding_size=4, num_hidden_layers=2, neuron_per_hidden_layer=32,
                 num_classes=1, b=0.99, n=0.01, use_cuda=True, update_mode=UPDATE_ADAM1):
        super().__init__()
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size,
                        num_hidden_layers=num_hidden_layers, neuron_per_hidden_layer=neuron_per_hidden_layer,
                        num_classes=num_classes, b=b, n=n, use_cuda=use_cuda, update_mode=update_mode)
        self._setup(feature_sizes, embedding_size, num_hidden_layers, neuron_per_hidden_layer, 1, num_classes, b, n,
                    0.2, use_cuda, update_mode)

    def _ctor_kwargs(self):
        return self._kw

    def __str__(self):
        return f"NFMAdam-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Hidden_Layers{self.num_hidden_layers}-Neuron_Per_Hidden_Layer{self.neuron_per_hidden_layer}-" \
               f"Num_Classes{self.num_classes}"


class DeepFMOnn(_DeepBase):
    """deepfm_onn.py:12-210 (hedge backpropagation)."""
    _IS_ONN = True
    _KIND_ID = 3

    def __init__(self, feature_sizes, embedding_size=4, num_hidden_layers=2, neuron_per_hidden_layer=32,
                 batch_size=1, num_classes=1, b=0.99, n=0.01, s=0.2, use_cuda=True, update_mode=UPDATE_ADAM1):
        super().__init__()
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size,
                        num_hidden_layers=num_hidden_layers, neuron_per_hidden_layer=neuron_per_hidden_layer,
                        batch_size=batch_size, num_classes=num_classes, b=b, n=n, s=s, use_cuda=use_cuda,
                        update_mode=update_mode)
        self._setup(feature_sizes, embedding_size, num_hidden_layers, neuron_per_hidden_layer, batch_size,
                    num_classes, b, n, s, use_cuda, update_mode)

    def _ctor_kwargs(self):
        return self._kw

    def __str__(self):
        return f"DeepFMOnn-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Hidden_Layers{self.num_hidden_layers}-Neuron_Per_Hidden_Layer{self.neuron_per_hidden_layer}-" \
               f"Num_Classes{self.num_classes}-N{self.n}"


class NFMOnn(_DeepBase):
    """nfm_onn.py:13-212. Positional order is (..., num_classes, batch_size, ...) here (nfm_onn.py:14-15)."""
    _IS_ONN = True
    _IS_NFM = True
    _KIND_ID = 4
    _UE_LOSS = LOSS_LOGITS_OF_SIG

    def __init__(self, feature_sizes, embedding_size=4, num_hidden_layers=2, neuron_per_hidden_layer=32,
                 num_classes=1, batch_size=1, b=0.99, n=0.01, s=0.2, use_cuda=True, update_mode=UPDATE_ADAM1):
        super().__init__()
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size,
                        num_hidden_layers=num_hidden_layers, neuron_per_hidden_layer=neuron_per_hidden_layer,
                        num_classes=num_classes, batch_size=batch_size, b=b, n=n, s=s, use_cuda=use_cuda,
                        update_mode=update_mode)
        self._setup(feature_sizes, embedding_size, num_hidden_layers, neuron_per_hidden_layer, batch_size,
                    num_classes, b, n, s, use_cuda, update_mode)

    def _ctor_kwargs(self):
        return self._kw

    def __str__(self):
        return f"NFMOnn-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Hidden_Layers{self.num_hidden_layers}-Neuron_Per_Hidden_Layer{self.neuron_per_hidden_layer}-" \
               f"Num_Classes{self.num_classes}-N{self.n}"


class AFMAdam(nn.Module):
    """Attentional FM with the reference's constructor and parameter set (models/models_online_deep/afm_adam.py:13-41).
    The reference class cannot run (afm_adam.py:67,69 pass a float to .view; :121-123,167 use undefined attributes --
    SURVEY.md fact 7), so `forward` is the AFM paper's model (Xiao et al. 2017, eq. 8; definition: oracle/afm.py) and the
    training step is the family's per-call fresh-state Adam step on every parameter (`update_embedding`, and `fit` as the
    reference's epoch / mini-batch loop around it).  F <= 64, embedding_size <= 15, attention_size <= 8."""

    def __init__(self, feature_sizes, embedding_size=4, attention_size=4, n_epochs=64, batch_size=256, num_classes=1,
                 b=0.99, n=0.003, use_cuda=True):
        super().__init__()
        self._lib = _lib.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.field_size, self.feature_sizes = len(feature_sizes), feature_sizes
        self.embedding_size, self.attention_size = embedding_size, attention_size
        self.n_epochs, self.batch_size, self.num_classes, self.use_cuda = n_epochs, batch_size, num_classes, use_cuda
        F, k, A = self.field_size, embedding_size, attention_size
        if not (2 <= F <= 64 and k <= 15 and A <= 8):
            raise ValueError("AFMAdam: need 2 <= fields <= 64, embedding_size <= 15, attention_size <= 8")
        self._kw = dict(feature_sizes=feature_sizes, embedding_size=embedding_size, attention_size=attention_size,
                        n_epochs=n_epochs, batch_size=batch_size, num_classes=num_classes, b=b, n=n, use_cuda=use_cuda)
        self._rowp = self._lib.fmb_rowp(k)
        sizes = np.asarray(list(feature_sizes), dtype=np.int64)
        self._offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self._R = int(self._offsets_np[-1])
        self._field_off_dev = torch.from_numpy(self._offsets_np.astype(np.int32)).to(self.device)
        # parameters drawn on the CPU in the reference's order (afm_adam.py:30-41)
        self.bias = nn.Parameter(torch.tensor(b).to(self.device))
        self.n = nn.Parameter(torch.tensor(n).to(self.device), requires_grad=False)
        self._lr = float(np.float32(n))
        table = torch.zeros(self._R, self._rowp)
        fo = [nn.Embedding(int(fs), 1) for fs in sizes]
        so = [nn.Embedding(int(fs), k) for fs in sizes]
        with torch.no_grad():
            for f in range(F):
                lo, hi = int(self._offsets_np[f]), int(self._offsets_np[f + 1])
                table[lo:hi, :k] = so[f].weight
                table[lo:hi, k] = fo[f].weight[:, 0]
        self._table = table.to(self.device)
        fo_m, so_m = [], []
        for f in range(F):
            lo, hi = int(self._offsets_np[f]), int(self._offsets_np[f + 1])
            so_m.append(_ViewEmbedding(self._table[lo:hi, :k]))
            fo_m.append(_ViewEmbedding(self._table[lo:hi, k:k + 1]))
        self.first_order_embeddings, self.second_order_embeddings = nn.ModuleList(fo_m), nn.ModuleList(so_m)
        lin = nn.Linear(k, A)
        flat = torch.cat([lin.weight.detach().reshape(-1), lin.bias.detach(), torch.randn(A), torch.randn(k)])
        self._att = flat.to(self.device).contiguous()          # W [A,k] | c [A] | H [A] | P [k]
        self.attention_linear = _ViewLinear(self._att[:A * k].view(A, k), self._att[A * k:A * k + A])
        self.H = nn.Parameter(self._att[A * k + A:A * k + 2 * A])
        self.P = nn.Parameter(self._att[A * k + 2 * A:])
        pi, pj = np.triu_indices(F, 1)
        self._pair_i = torch.from_numpy(pi.astype(np.uint8)).to(self.device)
        self._pair_j = torch.from_numpy(pj.astype(np.uint8)).to(self.device)
        self._ws = {}

    def _apply(self, fn, recurse=True):
        raise RuntimeError("fm_for_online_recommendation_b200 models are bound to their CUDA device and to fp32")

    def __reduce__(self):
        return (_rebuild_afm, (self._kw, self._table.detach().cpu(), self.bias.detach().cpu(), self._att.detach().cpu()))

    def __str__(self):
        return f"AFMAdam-Feature_Sizes{self.feature_sizes}-Embedding_Sizes{self.embedding_size}-" \
               f"Num_Classes{self.num_classes}"

    def _buf(self, name, shape, dtype=torch.float32):
        n = int(np.prod(shape))
        t = self._ws.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._ws[name] = t
        return t[:n].view(*shape)

    def _encode(self, Xi, Xv, Y=None):
        F = self.field_size
        a = np.asarray(Xi.cpu() if torch.is_tensor(Xi) else Xi, dtype=np.int64).reshape(-1, F)
        if a.size and (a.min() < 0 or (a >= (self._offsets_np[1:] - self._offsets_np[:-1])[None, :]).any()):
            raise IndexError("index out of range in self")
        ids = torch.from_numpy((a + self._offsets_np[:-1][None, :]).astype(np.int32)).to(self.device).contiguous()
        xv = torch.from_numpy(np.ascontiguousarray(np.asarray(Xv.cpu() if torch.is_tensor(Xv) else Xv, dtype=np.float32)
                                                   .reshape(-1, F))).to(self.device)
        y = None if Y is None else torch.from_numpy(np.asarray(Y.cpu() if torch.is_tensor(Y) else Y, dtype=np.float32)
                                                    .reshape(-1)).to(self.device)
        return ids, xv, y

    def _att_ptrs(self):
        k, A = self.embedding_size, self.attention_size
        base = self._att.data_ptr()
        return [C.c_void_p(base + 4 * o) for o in (0, A * k, A * k + A, A * k + 2 * A)]

    def forward(self, Xi, Xv):
        ids, xv, _ = self._encode(Xi, Xv)
        B = ids.shape[0]
        z = torch.empty(B, device=self.device)
        check(self._lib.fmb_afm_step(ptr(ids), ptr(xv), None, None, ptr(self._table), ptr(self.bias), *self._att_ptrs(),
                                     ptr(self._pair_i), ptr(self._pair_j), B, self.field_size, self.embedding_size,
                                     self.attention_size, 0, ptr(z), None, None, None, None, 0, _stream()), "fmb_afm_step")
        return z

    def predict(self, Xi, Xv):
        self.eval()
        z = self.forward(Xi, Xv)
        out = torch.empty(z.numel(), dtype=torch.uint8, device=self.device)
        check(self._lib.fmb_predict(ptr(z), z.numel(), ptr(out), _stream()), "fmb_predict")
        return out.cpu().numpy().astype(bool)

    def update_embedding(self, Xi, Xv, Y, _grads_out=None):
        """one batch: BCE-with-logits on the AFM logit, fresh-state Adam step on every parameter; returns the loss"""
        self.train()
        lib, st = self._lib, _stream()
        ids, xv, y = self._encode(Xi, Xv, Y)
        B, F, k, A = ids.shape[0], self.field_size, self.embedding_size, self.attention_size
        N = B * F
        sk = self._buf("skeys", (N,), torch.int32); pm = self._buf("perm", (N,), torch.int32)
        pf = self._buf("posflag", (N,), torch.int32)
        if B <= lib.fmb_sort_fields_max_batch():
            check(lib.fmb_sort_fields(ptr(ids), B, F, ptr(self._field_off_dev), ptr(sk), ptr(pm), st), "fmb_sort_fields")
        else:
            wsb = lib.fmb_sort_workspace_bytes(N)
            sws = self._buf("sort_ws", (wsb,), torch.uint8)
            kb = max(1, int(self._R - 1).bit_length())
            check(lib.fmb_sort_segment(ptr(ids), N, kb, ptr(sws), wsb, ptr(sk), ptr(pm), None, None, st), "fmb_sort_segment")
        check(lib.fmb_pos_flags(ptr(sk), ptr(pm), N, ptr(pf), st), "fmb_pos_flags")
        delta = self._buf("delta", (B,)); lossv = self._buf("lossv", (B,))
        PD = int(lib.fmb_afm_dense_floats(k, A))
        dg = self._buf("dense_g", (B, PD))
        wsb = lib.fmb_bwd_workspace_bytes(N, k)
        ws = self._buf("bwd_ws", (wsb,), torch.uint8)
        check(lib.fmb_afm_step(ptr(ids), ptr(xv), ptr(y), ptr(pf), ptr(self._table), ptr(self.bias), *self._att_ptrs(),
                               ptr(self._pair_i), ptr(self._pair_j), B, F, k, A, 0, None, ptr(delta), ptr(lossv), ptr(dg),
                               ptr(ws), wsb, st), "fmb_afm_step")
        check(lib.fmb_fm_backward_runs_all(ptr(sk), N, ptr(self._table), F, k, self._lr, 0, ptr(ws), wsb, st),
              "fmb_fm_backward_runs_all")
        check(lib.fmb_afm_dense_update(ptr(dg), B, k, A, *self._att_ptrs(), self._lr, 0, ptr(_grads_out), st),
              "fmb_afm_dense_update")
        loss = torch.empty((), device=self.device)
        check(lib.fmb_finish_step(ptr(delta), ptr(lossv), B, ptr(self.bias), self._lr, 0, ptr(loss), st), "fmb_finish_step")
        return loss

    def fit(self, Xi_train, Xv_train, y_train, Xi_valid=None, Xv_valid=None, y_valid=None):
        """afm_adam.py:76-135's loop: n_epochs passes over the training set in mini-batches of batch_size"""
        Xi = np.asarray(Xi_train).reshape(-1, self.field_size)
        Xv = np.asarray(Xv_train, dtype=np.float32).reshape(-1, self.field_size)
        y = np.asarray(y_train, dtype=np.float32).reshape(-1)
        losses = []
        for _ in range(self.n_epochs):
            tot, nb = 0.0, 0
            for off in range(0, len(y), self.batch_size):
                end = min(len(y), off + self.batch_size)
                tot += float(self.update_embedding(Xi[off:end], Xv[off:end], y[off:end]).item())
                nb += 1
            losses.append(tot / max(nb, 1))
        return losses


def _rebuild_afm(kw, table, bias, att):
    m = AFMAdam(**kw)
    with torch.no_grad():
        m._table.copy_(table)
        m.bias.copy_(bias)
        m._att.copy_(att)
    return m
