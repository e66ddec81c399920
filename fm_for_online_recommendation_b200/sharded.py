"""Row-sharded multi-GPU FM training step (BASELINE.json configs[4]; SURVEY.md 8e).

One process per GPU (`torch.distributed`, backend nccl).  Global row r of the packed table lives on
rank r % G at local row r // G; every rank feeds its own batch of B samples and one call performs
the step over the global batch of G*B samples (same semantics as the single-GPU
`update_embedding` on the concatenated batch: loss is the mean over G*B, duplicate rows are summed in
global sample order).  Pipeline and reduction order: see csrc/sharded.cu.

The reference has no distributed code; this module is the B200-native design for its Criteo-scale
configuration.  `ShardedFM` is not a reference class, it is the engine `bench.py --gpus N` drives.
"""
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import AdagradState, RunList, SparseAdamState, check, ptr
from .deep import UPDATE_ADAGRAD, UPDATE_SPARSE_ADAM

INT_MAX = 0x7FFFFFFF
_USE_RUNLIST = os.environ.get("FMB_SHARD_RL", "1") != "0"   # experiment knob: 0 = one warp per 32 sorted positions (round 1)


# ------------------------------------------------------------------ host-side shard map (CPU-testable)
def owner_of(gid, G):
    return gid % G


def local_row(gid, G):
    return gid // G


def local_rows_count(R, G, rank):
    """rows r in [0, R) with r % G == rank."""
    return (R - rank + G - 1) // G if R > rank else 0


def shard_from_full(full, G, rank):
    """rows of a full [R, ...] array owned by `rank`, in local-row order."""
    return full[rank::G]


def full_from_shards(shards):
    """inverse of shard_from_full for a list of per-rank arrays."""
    G = len(shards)
    R = sum(s.shape[0] for s in shards)
    out = np.empty((R,) + tuple(shards[0].shape[1:]), dtype=shards[0].dtype)
    for r, s in enumerate(shards):
        out[r::G] = s
    return out


_DMA_IDS = os.environ.get("FMB_SHARD_DMA_IDS", "1") != "0"   # fused path: ids exchanged by copy-engine copies


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class ShardedFM:
    """FM (first + second order, bias) with the embedding tables row-sharded over the process group."""

    def __init__(self, feature_sizes, embedding_size, n=1e-4, b=0.99, update_mode=0, group=None, seed=0,
                 init="normal", world=None, rank=None):
        self._lib = _lib.require_cuda()
        self.group = group
        # world/rank given explicitly: no process group is touched (single-process emulation of the
        # ranks in tests: the phases below are called rank by rank and the exchanges done by hand)
        self.G = world if world is not None else dist.get_world_size(group)
        self.rank = rank if rank is not None else dist.get_rank(group)
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.feature_sizes = list(feature_sizes)
        self.F, self.k = len(feature_sizes), embedding_size
        self.rowp = self._lib.fmb_rowp(self.k)
        self.kp4 = self._lib.fmb_kp4(self.k)
        self.PW = self._lib.fmb_shard_pw(self.k)
        self.CW = self._lib.fmb_shard_cw(self.k)
        self.offsets_np = np.concatenate([[0], np.cumsum(feature_sizes)]).astype(np.int64)
        self.R = int(self.offsets_np[-1])
        self.R_local = local_rows_count(self.R, self.G, self.rank)
        self.field_off_dev = torch.from_numpy(self.offsets_np.astype(np.int32)).to(self.device)
        self.offsets_dev = torch.from_numpy(self.offsets_np[:-1].copy()).to(self.device)
        self.lr = float(np.float32(n))
        self.update_mode = update_mode
        self.table = torch.zeros(self.R_local + 1, self.rowp, device=self.device)
        if init == "normal":  # N(0,1) like nn.Embedding; drawn on the device (synthetic weights)
            g = torch.Generator(device=self.device)
            g.manual_seed(seed * 1000 + self.rank)
            self.table[:self.R_local, :self.k + 1].normal_(generator=g)
        self.bias = torch.full((1,), float(np.float32(b)), device=self.device)
        self._ws = {}
        self._rl = {}
        self._side = torch.cuda.Stream()   # owner-side sort and bias/loss epilogue run beside the main chain
        self._pre = torch.cuda.Stream()    # pipelined mode: the NEXT batch's owner-side sort
        self._slot = 0                     # pipelined mode: which buffer set holds the current batch
        self.launches = 0
        self.overflow = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._ada = None                   # update mode 3's state (enable_adagrad)
        self._sa = None                    # update mode 4's state (enable_sparse_adam)

    # ---------------------------------------------------------------- parameters (tests)
    def load_full(self, V, w1, bias):
        V = np.asarray(V, np.float32)
        w1 = np.asarray(w1, np.float32)
        t = np.zeros((self.R_local + 1, self.rowp), np.float32)
        t[:self.R_local, :self.k] = shard_from_full(V, self.G, self.rank)
        t[:self.R_local, self.k] = shard_from_full(w1, self.G, self.rank)
        self.table.copy_(torch.from_numpy(t))
        self.bias.fill_(float(np.asarray(bias).reshape(-1)[0]))

    def local_params(self):
        t = self.table[:self.R_local].cpu().numpy()
        return t[:, :self.k].copy(), t[:, self.k].copy()

    # ---------------------------------------------------------------- update modes 3 and 4 (state kept across steps)
    # Row r's state lives beside row r: on rank r % G at local row r // G, in a table with the local table's shape (Adagrad)
    # or FTRL's [rows][2][rowp] layout (SparseAdam).  Only the owner updates a row, so the state never crosses a link.  The
    # bias is replicated and every rank runs the same bias step over the global batch, so its state is replicated too.
    def enable_adagrad(self, eps=1e-10, initial_accumulator_value=0.0):
        """Switch the step to torch.optim.Adagrad(lr=n, eps=eps, initial_accumulator_value=...) kept across steps: the
        trajectory of ONE such optimizer over the full tables stepped on the global batch.  Every rank calls it.  Calling it
        again resets the sums; captured step graphs are dropped (they hold the previous sums' addresses)."""
        v = float(np.float32(initial_accumulator_value))
        if v < 0:
            raise ValueError("initial_accumulator_value must be >= 0")
        self.update_mode = UPDATE_ADAGRAD
        self._ada_eps = float(np.float32(eps))
        self._ada_sums = torch.full((self.R_local + 1, self.rowp), v, dtype=torch.float32, device=self.device)
        self._ada_bias = torch.full((1,), v, dtype=torch.float32, device=self.device)
        self._ada = AdagradState(self._ada_sums.data_ptr(), self._ada_bias.data_ptr(), None, self._ada_eps)
        self._drop_graphs()

    def enable_sparse_adam(self, betas=(0.9, 0.999), eps=1e-8):
        """Switch the step to torch.optim.SparseAdam(<tables>, lr=n, betas, eps) on the rows each global batch hits and
        torch.optim.Adam([bias], lr=n, betas, eps), both kept across steps.  Every row hit steps, also with a zero
        gradient.  Every rank calls it and counts every step.  Calling it again resets the moments and the counter;
        captured step graphs are dropped, and the step cannot be captured in this mode (a replay would repeat the
        captured step's bias corrections)."""
        b1, b2 = (float(b) for b in betas)
        if not (0.0 <= b1 < 1.0 and 0.0 <= b2 < 1.0) or eps < 0:
            raise ValueError("need 0 <= beta1, beta2 < 1 and eps >= 0")
        self.update_mode = UPDATE_SPARSE_ADAM
        self._sa_mv = torch.zeros((self.R_local + 1, 2, self.rowp), dtype=torch.float32, device=self.device)
        self._sa_bias = torch.zeros((2,), dtype=torch.float32, device=self.device)
        self._sa = SparseAdamState(self._sa_mv.data_ptr(), self._sa_bias.data_ptr(), None, b1, b2, float(np.float32(eps)),
                                   0, 0)
        self._drop_graphs()

    def local_state(self):
        """this rank's shard of the update rule's state, in local-row order, and the (replicated) bias state:
        mode 3 (sums_V [R_local, k], sums_w1 [R_local], bias_sum [1]);
        mode 4 (m_V, v_V [R_local, k], m_w1, v_w1 [R_local], bias_m, bias_v [1], steps taken)."""
        k, n = self.k, self.R_local
        if self.update_mode == UPDATE_ADAGRAD and self._ada is not None:
            s = self._ada_sums[:n].cpu().numpy()
            return s[:, :k].copy(), s[:, k].copy(), self._ada_bias.cpu().numpy().copy()
        if self.update_mode == UPDATE_SPARSE_ADAM and self._sa is not None:
            mv = self._sa_mv[:n].cpu().numpy()
            b = self._sa_bias.cpu().numpy()
            return (mv[:, 0, :k].copy(), mv[:, 1, :k].copy(), mv[:, 0, k].copy(), mv[:, 1, k].copy(), b[:1].copy(),
                    b[1:].copy(), int(self._sa.step))
        raise RuntimeError(f"update mode {self.update_mode} keeps no state (enable_adagrad / enable_sparse_adam)")

    def _state_arg(self):
        """the state slot of the C entry points: fmb_adagrad_t in mode 3, fmb_sparse_adam_t in mode 4, else NULL (a mode
        3 or 4 step without its state is refused by the library, naming the mode, before any kernel runs)"""
        if self.update_mode == UPDATE_ADAGRAD and self._ada is not None:
            return C.byref(self._ada)
        if self.update_mode == UPDATE_SPARSE_ADAM and self._sa is not None:
            return C.byref(self._sa)
        return None

    def _advance(self):
        """mode 4: one more step on this rank's counter when the step is submitted (the scalars go by value into the
        launches), so that every rank has the same scalars and host pipelining stays exact"""
        if self.update_mode == UPDATE_SPARSE_ADAM and self._sa is not None:
            check(self._lib.fmb_sparse_adam_advance(C.byref(self._sa), self.lr, 0), "fmb_sparse_adam_advance")

    def _drop_graphs(self):
        for name in ("_graph", "_g_loss", "_pgraphs", "_pg_loss"):
            self.__dict__.pop(name, None)

    def _refuse_capture(self):
        if self.update_mode == UPDATE_SPARSE_ADAM:
            raise RuntimeError("update mode 4 (SparseAdam) cannot be captured into a step graph: a replay would repeat the "
                               "captured step's bias corrections; run the step eagerly")

    # ---------------------------------------------------------------- the step
    def _buf(self, name, shape, dtype=torch.float32):
        n = int(np.prod(shape))
        t = self._ws.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._ws[name] = t
        return t[:n].view(*shape)

    def encode(self, Xi_local, Y_local):
        """per-field ids [B,F] (lists / ndarray) + labels -> device (global row ids int32, labels fp32)."""
        a = np.asarray(Xi_local, dtype=np.int64).reshape(-1, self.F)
        ids = torch.from_numpy((a + self.offsets_np[:-1][None, :]).astype(np.int32)).to(self.device)
        y = torch.from_numpy(np.asarray(Y_local, dtype=np.float32).reshape(-1)).to(self.device)
        return ids.contiguous(), y

    # the step, split at the three exchanges so tests can emulate several ranks in one process
    def phase_ids(self, ids, slot=0):
        """-> idsT [F,B] (to be all-gathered into [G,F,B])."""
        B = ids.shape[0]
        idsT = self._buf(f"idsT{slot}", (self.F, B), torch.int32)
        check(self._lib.fmb_transpose_ids(ptr(ids), B, self.F, ptr(idsT), _stream()), "fmb_transpose_ids")
        return idsT

    def phase_partial(self, idsT_all):
        """idsT_all [G,F,B] -> partial [G,B,PW] (block r goes to rank r): per sample, the rows this rank owns."""
        lib, st = self._lib, _stream()
        G, F, k = self.G, self.F, self.k
        B = idsT_all.shape[2]
        partial = self._buf("partial", (G, B, self.PW))
        check(lib.fmb_shard_partial_forward(ptr(idsT_all), ptr(self.table), G, self.rank, B, F, k, ptr(partial), st),
              "fmb_shard_partial_forward")
        return partial

    def _sort_owned(self, idsT_all, slot, posflag=None):
        """stable per-field sort of the entries this rank owns, on the CURRENT stream, into buffer set `slot`
        (posflag: also every owned entry's sorted position | multi-hit flag, for the fused step)."""
        lib = self._lib
        G, F = self.G, self.F
        B = idsT_all.shape[2]
        Btot = G * B
        cap = min(lib.fmb_shard_sort_max_cap(), ((2 * Btot // G + Btot // 4 + 1023) // 1024) * 1024)
        self._cap = cap
        skeys = self._buf(f"skeys{slot}", (F, cap), torch.int32)
        perm = self._buf(f"perm{slot}", (F, cap), torch.int32)
        counts = self._buf(f"counts{slot}", (F,), torch.int32)
        # run list of the sorted owned entries (one segment per field), consumed by the backward's run kernel: one warp
        # per run, the long runs (the hot rows' G*B/rows-entry chains) first and with the deeper ring
        rl = None
        if _USE_RUNLIST:
            rcap = cap // 2 + 32
            ent = self._buf(f"rl_entries{slot}", (F * rcap, 4), torch.int32)
            cnt = self._buf(f"rl_counts{slot}", (2 * F,), torch.int32)
            self._rl[slot] = RunList(ent.data_ptr(), cnt.data_ptr(), F, rcap)
            rl = C.byref(self._rl[slot])
        check(lib.fmb_shard_sort_fields_pf(ptr(idsT_all), G, self.rank, B, F, ptr(self.field_off_dev), cap,
                                           ptr(skeys), ptr(perm), ptr(counts), ptr(self.overflow), rl, ptr(posflag),
                                           _stream()), "fmb_shard_sort_fields")

    def phase_owner_forward(self, idsT_all):
        """idsT_all [G,F,B] -> partial [G,B,PW] (block r goes to rank r); also sorts the owned entries."""
        partial = self.phase_partial(idsT_all)
        # the sort needs the ids only: it runs on the side stream, next to the partial forward, the all-to-all,
        # the combine and the context all-gather; phase_backward joins it
        main = torch.cuda.current_stream()
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self._sort_owned(idsT_all, 0)
        return partial

    def phase_combine(self, recv, y, loss_kind=0):
        """recv [G,B,PW] (block o = owner o's partials for MY samples) -> ctx [B,CW]."""
        B = recv.shape[1]
        ctx = self._buf("ctx", (B, self.CW))
        check(self._lib.fmb_shard_combine(ptr(recv), ptr(self.bias), ptr(y), self.G, self.rank, B, self.k, loss_kind, ptr(ctx),
                                          None, _stream()), "fmb_shard_combine")
        return ctx

    def phase_backward(self, ctx_all, slot=0, join_sort=True):
        """ctx_all [G*B,CW] -> row updates of the owned rows (sorted entries of buffer set `slot`), bias step;
        returns the mean loss."""
        lib, st = self._lib, _stream()
        F, k, cap = self.F, self.k, self._cap
        Btot = ctx_all.shape[0]
        N = F * cap
        main = torch.cuda.current_stream()
        self._advance()
        state = self._state_arg()
        if join_sort:
            main.wait_stream(self._side)  # sorted keys / permutation are ready (phase_owner_forward put them there)
        wsb = lib.fmb_bwd_workspace_bytes(N, k)
        ws = self._buf("bwd_ws", (wsb,), torch.uint8)
        gs = ctx_all.view(-1)[self.kp4:]
        # bias step + mean loss depend on ctx_all only: side stream, beside the row updates
        delta_all = self._buf("delta_all", (Btot,))
        lossv_all = self._buf("lossv_all", (Btot,))
        loss = torch.empty((), device=self.device)
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            check(lib.fmb_shard_unpack_ctx(ptr(ctx_all), Btot, k, ptr(delta_all), ptr(lossv_all), _stream()),
                  "fmb_shard_unpack_ctx")
            check(lib.fmb_finish_step_ex(ptr(delta_all), ptr(lossv_all), Btot, ptr(self.bias), self.lr,
                                         self.update_mode, state, ptr(loss), _stream()), "fmb_finish_step")
        self.launches += 9
        rl = C.byref(self._rl[slot]) if (_USE_RUNLIST and slot in self._rl) else None
        check(lib.fmb_fm_backward_update_rl_ex(ptr(self._ws[f"skeys{slot}"]), ptr(self._ws[f"perm{slot}"]), N, Btot * F,
                                               None, ptr(self.table), F, k, ptr(ctx_all), self.CW, ptr(gs), self.CW, 1, None,
                                               INT_MAX, self.lr, self.update_mode, state, rl, ptr(ws), wsb, st),
              "fmb_fm_backward_update_rl")
        main.wait_stream(self._side)      # join: the step is complete when both branches are
        return loss

    def update_embedding(self, ids, y, loss_kind=0):
        """ids int32 [B,F] global row ids of THIS rank's batch (device), y fp32 [B] (device).
        Returns the mean loss over the global batch (0-dim device tensor, identical on every rank)."""
        G, B, F = self.G, ids.shape[0], self.F
        idsT = self.phase_ids(ids)
        idsT_all = self._buf("idsT_all", (G, F, B), torch.int32)
        dist.all_gather_into_tensor(idsT_all.view(-1), idsT.view(-1), group=self.group)
        partial = self.phase_owner_forward(idsT_all)
        recv = self._buf("recv", (G, B, self.PW))
        dist.all_to_all_single(recv.view(-1), partial.view(-1), group=self.group)
        ctx = self.phase_combine(recv, y, loss_kind)
        ctx_all = self._buf("ctx_all", (G * B, self.CW))
        dist.all_gather_into_tensor(ctx_all.view(-1), ctx.view(-1), group=self.group)
        return self.phase_backward(ctx_all)

    # ---------------------------------------------------------------- pipelined steps
    # The exchange of the ids and the owner-side sort depend on the ids only, so they can be done one step ahead:
    # step t runs while the ids of batch t+1 are all-gathered (NCCL stream, under step t's partial forward) and
    # sorted (stream _pre, under step t's exchanges and backward).  Same kernels, same arithmetic, same results.
    def _prepare(self, ids, slot):
        G, B, F = self.G, ids.shape[0], self.F
        main = torch.cuda.current_stream()
        idsT = self.phase_ids(ids, slot)
        idsT_all = self._buf(f"idsT_all{slot}", (G, F, B), torch.int32)
        work = dist.all_gather_into_tensor(idsT_all.view(-1), idsT.view(-1), group=self.group, async_op=True)
        self._pre.wait_stream(main)   # every earlier reader of this buffer set was enqueued on main before now
        with torch.cuda.stream(self._pre):
            work.wait()               # _pre (not main) waits for the collective
            self._sort_owned(idsT_all, slot)

    def prepare(self, ids):
        """start the pipeline: exchange and sort the FIRST batch's ids (the batch the next step trains on)."""
        self._slot = 0
        self._prepare(ids, 0)
        torch.cuda.current_stream().wait_stream(self._pre)

    def update_embedding_pipelined(self, y, ids_next, loss_kind=0):
        """train on the batch whose ids were given to the previous call (or to prepare()), labels `y`; meanwhile
        exchange and sort `ids_next` (None at the end of the stream).  Returns the mean loss of the trained batch."""
        G, F = self.G, self.F
        p = self._slot
        main = torch.cuda.current_stream()
        if ids_next is not None:
            self._prepare(ids_next, 1 - p)
        idsT_all = self._ws[f"idsT_all{p}"]
        B = idsT_all.numel() // (G * F)
        partial = self.phase_partial(idsT_all.view(G, F, B))
        recv = self._buf("recv", (G, B, self.PW))
        dist.all_to_all_single(recv.view(-1), partial.view(-1), group=self.group)
        ctx = self.phase_combine(recv, y, loss_kind)
        ctx_all = self._buf("ctx_all", (G * B, self.CW))
        dist.all_gather_into_tensor(ctx_all.view(-1), ctx.view(-1), group=self.group)
        loss = self.phase_backward(ctx_all, p, join_sort=False)   # sorted one call earlier
        main.wait_stream(self._pre)   # the call is complete when the next batch is sorted too
        self._slot = 1 - p
        return loss

    # ---------------------------------------------------------------- pipelined steps over peer memory (no NCCL)
    # Same step, but the three exchanges are plain stores into the peers' buffers (symmetric memory over NVLink)
    # followed by epoch flags: csrc/sharded.cu "Peer-memory exchange".  Channels of the flag block:
    CH_IDS, CH_A2A, CH_CTX = 0, 1, 2

    def _peer_layout(self, B):
        """sub-buffers of the exchange arena (int32 words, 256-byte aligned): name -> (offset, words)"""
        G, F = self.G, self.F
        T = self._lib.fmb_shard3_tiles(G, B, F, self.k)
        words = {"ids0": G * F * B, "ids1": G * F * B, "recv": G * B * self.PW, "ctx": G * B * self.CW, "flags": 64,
                 "tflags": max(2 * T, 64)}
        off, total = {}, 0
        for name, n in words.items():
            off[name] = (total, n)
            total += (n + 63) // 64 * 64
        return off, total, T

    def _peer_bind(self, B, arena, base_ptrs, hdl=None):
        """arena: MY zero-initialised exchange buffer; base_ptrs[r]: the address at which this device sees rank r's"""
        G, F = self.G, self.F
        off, total, T = self._peer_layout(B)
        ptrs = {name: (C.c_void_p * G)(*[int(base_ptrs[r]) + 4 * o for r in range(G)]) for name, (o, _) in off.items()}
        view = {name: arena[o:o + n] for name, (o, n) in off.items()}
        self._peer = {"B": B, "arena": arena, "hdl": hdl, "ptrs": ptrs, "tiles": T,
                      "ids": [view["ids0"].view(G, F, B), view["ids1"].view(G, F, B)],
                      "recv": view["recv"].view(torch.float32).view(G, B, self.PW),
                      "ctx": view["ctx"].view(torch.float32).view(G * B, self.CW),
                      "flags": view["flags"], "tflags": view["tflags"],
                      "posflag": [torch.zeros((F, G * B), dtype=torch.int32, device=self.device) for _ in range(2)] if T else None,
                      "epoch": torch.zeros(16, dtype=torch.int32, device=self.device),   # epoch[8] | block counters[8]
                      "error": torch.zeros(1, dtype=torch.int32, device=self.device)}

    def _peer_setup(self, B):
        """allocate idsT_all (two slots), recv, ctx_all and the flag blocks in symmetric memory and map the peers'
        copies (collective: every rank calls it with the same B)."""
        import torch.distributed._symmetric_memory as symm
        group = self.group if self.group is not None else dist.group.WORLD
        _, total, _ = self._peer_layout(B)
        arena = symm.empty(total, dtype=torch.int32, device=self.device)
        arena.zero_()
        hdl = symm.rendezvous(arena, group)
        torch.cuda.synchronize()
        dist.barrier(group=group)                  # every flag block is zero before anyone publishes
        self._peer_bind(B, arena, [int(hdl.buffer_ptrs[r]) for r in range(self.G)], hdl)
        # tensor views of the peers' id slabs (copy-engine exchange of the fused path)
        try:
            off, total, _ = self._peer_layout(B)
            G, F = self.G, self.F
            views = []
            for r in range(G):
                whole = hdl.get_buffer(r, (total,), torch.int32, 0)
                views.append([whole[off[f"ids{sl}"][0]:off[f"ids{sl}"][0] + G * F * B].view(G, F, B) for sl in (0, 1)])
            self._peer["peer_ids"] = views
        except Exception as exc:  # noqa: BLE001 -- the store-based exchange needs only the raw pointers
            print(f"[rank {self.rank}] no tensor views of the peers' buffers ({type(exc).__name__}: {exc}); "
                  "ids are exchanged by the store kernel", file=sys.stderr, flush=True)
            self._peer["peer_ids"] = None

    def _sync_args(self):
        pr = self._peer
        return pr["ptrs"]["flags"], ptr(pr["flags"]), ptr(pr["epoch"]), ptr(pr["error"])

    def _signal(self, channel, mode):
        pr = self._peer
        check(self._lib.fmb_shard_signal(pr["ptrs"]["flags"], ptr(pr["flags"]), ptr(pr["epoch"]), channel, self.G,
                                         self.rank, mode, ptr(pr["error"]), _stream()), "fmb_shard_signal")

    def _prepare_peers(self, ids, slot):
        """everything about the next batch's ids happens on the _pre stream, beside the current step."""
        pr, B = self._peer, ids.shape[0]
        main = torch.cuda.current_stream()
        self._pre.wait_stream(main)               # `ids` is ready; every earlier reader of this slot is behind us
        with torch.cuda.stream(self._pre):
            check(self._lib.fmb_shard_transpose_ids_peers(ptr(ids), B, self.F, self.G, self.rank,
                                                          pr["ptrs"][f"ids{slot}"], *self._sync_args(), self.CH_IDS,
                                                          _stream()), "fmb_shard_transpose_ids_peers")
            self._signal(self.CH_IDS, 2)          # every rank's slab has landed in MY idsT_all
            self._sort_owned(pr["ids"][slot], slot)

    def prepare_peers(self, ids):
        """start the peer-memory pipeline with the first batch's ids (collective on first use: maps the buffers)."""
        if getattr(self, "_peer", None) is None or self._peer["B"] != ids.shape[0]:
            self._peer_setup(ids.shape[0])
        self._slot = 0
        self._prepare_peers(ids, 0)
        torch.cuda.current_stream().wait_stream(self._pre)

    def update_embedding_peers(self, y, ids_next, loss_kind=0):
        """update_embedding_pipelined with every exchange done by stores into peer memory + epoch flags."""
        pr, lib, G, F, k = self._peer, self._lib, self.G, self.F, self.k
        p, B = self._slot, self._peer["B"]
        main = torch.cuda.current_stream()
        if ids_next is not None:
            self._prepare_peers(ids_next, 1 - p)
        # partial forward: stores block r into rank r's recv, its last block publishes the A2A epoch
        check(lib.fmb_shard_partial_forward_peers(ptr(pr["ids"][p]), ptr(self.table), G, self.rank, B, F, k,
                                                  pr["ptrs"]["recv"], *self._sync_args(), self.CH_A2A, _stream()),
              "fmb_shard_partial_forward_peers")
        # combine: waits for the G owners' A2A epochs, folds, stores ctx into every rank's ctx_all, publishes CTX
        check(lib.fmb_shard_combine_peers(ptr(pr["recv"]), ptr(self.bias), ptr(y), G, self.rank, B, k, loss_kind,
                                          pr["ptrs"]["ctx"], None, *self._sync_args(), self.CH_A2A, self.CH_CTX,
                                          _stream()), "fmb_shard_combine_peers")
        self._signal(self.CH_CTX, 2)              # every rank's ctx rows have landed in MY ctx_all
        loss = self.phase_backward(pr["ctx"], p, join_sort=False)
        self.launches += 1                        # the two wait kernels (phase_backward counts 9 for the rest)
        main.wait_stream(self._pre)
        self._slot = 1 - p
        if not torch.cuda.is_current_stream_capturing():
            self._poll()
        return loss

    # ---------------------------------------------------------------- the step as ONE kernel (csrc/shard3.cu)
    CH_TILE = 3     # word of the sync block that counts the fused steps (the per-tile flags carry this epoch)

    def fused_supported(self, B):
        return self._lib.fmb_shard3_tiles(self.G, B, self.F, self.k) > 0

    def _prepare_fused(self, ids, slot):
        """ids of the NEXT batch: exchange, owner sort with the per-entry position words, on the _pre stream.
        With a symmetric-memory handle the exchange is a local transpose + one copy-engine copy of my [F][B] slab into every
        peer's idsT_all (DMA over NVLink: no SM time, no store fences beside the step's kernels -- the store-based transpose
        took 49 us next to the fused kernel), then the epoch flag; emulated ranks (no handle) keep the store kernel."""
        pr, B = self._peer, ids.shape[0]
        main = torch.cuda.current_stream()
        self._pre.wait_stream(main)
        with torch.cuda.stream(self._pre):
            if pr.get("peer_ids") is not None and _DMA_IDS:
                mine = pr["ids"][slot][self.rank]
                check(self._lib.fmb_transpose_ids(ptr(ids), B, self.F, ptr(mine), _stream()), "fmb_transpose_ids")
                for r in range(self.G):
                    if r != self.rank:
                        pr["peer_ids"][r][slot][self.rank].copy_(mine, non_blocking=True)
                self._signal(self.CH_IDS, 3)      # publish my epoch (the copies are complete: stream order), wait for the peers'
            else:
                check(self._lib.fmb_shard_transpose_ids_peers(ptr(ids), B, self.F, self.G, self.rank,
                                                              pr["ptrs"][f"ids{slot}"], *self._sync_args(), self.CH_IDS,
                                                              _stream()), "fmb_shard_transpose_ids_peers")
                self._signal(self.CH_IDS, 2)
            self._sort_owned(pr["ids"][slot], slot, pr["posflag"][slot])

    def prepare_fused(self, ids):
        if getattr(self, "_peer", None) is None or self._peer["B"] != ids.shape[0]:
            self._peer_setup(ids.shape[0])
        if not self._peer["tiles"]:
            raise RuntimeError("fused sharded step: shape not supported (G power of two, B % (8 G) == 0, k <= 15)")
        self._slot = 0
        self._prepare_fused(ids, 0)
        torch.cuda.current_stream().wait_stream(self._pre)

    def _fused_launch(self, y, p, loss_kind):
        """the fused kernel + step-counter bump on the current stream (emulated ranks launch these on their own streams)"""
        pr, lib, G, F, k = self._peer, self._lib, self.G, self.F, self.k
        B, cap = pr["B"], self._cap
        wsb = lib.fmb_bwd_workspace_bytes(F * cap, k)
        ws = self._buf("bwd_ws", (wsb,), torch.uint8)
        ep = C.c_void_p(pr["epoch"].data_ptr() + 4 * self.CH_TILE)
        self._advance()   # _fused_finish steps the multi-hit rows and the bias with the same scalars
        check(lib.fmb_shard3_step_ex(ptr(pr["ids"][p]), ptr(self.table), ptr(self.bias), ptr(y), ptr(pr["posflag"][p]), G,
                                     self.rank, B, F, k, cap, loss_kind, self.lr, self.update_mode, self._state_arg(), ptr(ws),
                                     wsb, pr["ptrs"]["recv"], pr["ptrs"]["ctx"], pr["ptrs"]["tflags"], ptr(pr["recv"]),
                                     ptr(pr["ctx"]), ptr(pr["tflags"]), ep, ptr(pr["error"]), _stream()), "fmb_shard3_step")
        check(lib.fmb_shard3_bump(ep, _stream()), "fmb_shard3_bump")
        return ws, wsb

    def _fused_finish(self, ws, wsb, p):
        """behind the fused kernel: run kernel over the staged multi-hit contributions (main) beside the bias step (side)"""
        pr, lib, F, k, cap = self._peer, self._lib, self.F, self.k, self._cap
        Btot = self.G * pr["B"]
        main = torch.cuda.current_stream()
        delta_all = self._buf("delta_all", (Btot,))
        lossv_all = self._buf("lossv_all", (Btot,))
        loss = torch.empty((), device=self.device)
        state = self._state_arg()
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            check(lib.fmb_shard_unpack_ctx(ptr(pr["ctx"]), Btot, k, ptr(delta_all), ptr(lossv_all), _stream()),
                  "fmb_shard_unpack_ctx")
            check(lib.fmb_finish_step_ex(ptr(delta_all), ptr(lossv_all), Btot, ptr(self.bias), self.lr,
                                         self.update_mode, state, ptr(loss), _stream()), "fmb_finish_step")
        rl = C.byref(self._rl[p]) if (_USE_RUNLIST and p in self._rl) else None
        check(lib.fmb_fm_backward_runs_list(ptr(self._ws[f"skeys{p}"]), F * cap, ptr(self.table), F, k, self.lr,
                                            self.update_mode, state, rl, ptr(ws), wsb, _stream()),
              "fmb_fm_backward_runs_list")
        self.launches += 6
        main.wait_stream(self._side)
        return loss

    def update_embedding_fused(self, y, ids_next, loss_kind=0):
        """update_embedding_peers with partial forward, both exchanges, combine and the row updates in ONE kernel whose
        tiles keep their rows in shared memory (rows read once; per-tile flags instead of per-kernel epochs)."""
        p = self._slot
        main = torch.cuda.current_stream()
        if ids_next is not None:
            self._prepare_fused(ids_next, 1 - p)
        ws, wsb = self._fused_launch(y, p, loss_kind)
        loss = self._fused_finish(ws, wsb, p)
        main.wait_stream(self._pre)
        self._slot = 1 - p
        if not torch.cuda.is_current_stream_capturing():
            self._poll()
        return loss

    def capture_fused(self, ids, y, loss_kind=0):
        """capture_peers for the fused step"""
        self._refuse_capture()
        self._g_ids = ids.clone()
        self._g_y = y.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.prepare_fused(self._g_ids)
            for _ in range(2):
                self.update_embedding_fused(self._g_y, self._g_ids, loss_kind)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._pgraphs, self._pg_loss = [], []
        for parity in (0, 1):
            self._slot = parity
            g = torch.cuda.CUDAGraph()
            l0 = self.launches
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                loss = self.update_embedding_fused(self._g_y, self._g_ids, loss_kind)
            self._graph_launches = self.launches - l0
            self.launches = l0
            self._pgraphs.append(g)
            self._pg_loss.append(loss)
        self._slot = 0
        return self

    def check_exchange(self):
        v = int(self._peer["error"].item()) if getattr(self, "_peer", None) else 0
        if v == 32:
            raise RuntimeError("fused sharded step: a tile owned more entries than its shared-memory capacity (skewed ids)")
        if v >= 16:
            raise RuntimeError(f"fused sharded step: phase {v - 16} timed out waiting for a peer's tile flag")
        if v:
            raise RuntimeError(f"peer-memory exchange: channel {v - 1} timed out waiting for a peer's epoch flag")

    def capture_peers(self, ids, y, loss_kind=0):
        """capture_pipelined for the peer-memory step (no collective inside the graphs)."""
        self._refuse_capture()
        self._g_ids = ids.clone()
        self._g_y = y.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.prepare_peers(self._g_ids)
            for _ in range(2):
                self.update_embedding_peers(self._g_y, self._g_ids, loss_kind)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._pgraphs, self._pg_loss = [], []
        for parity in (0, 1):
            self._slot = parity
            g = torch.cuda.CUDAGraph()
            l0 = self.launches
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                loss = self.update_embedding_peers(self._g_y, self._g_ids, loss_kind)
            self._graph_launches = self.launches - l0   # kernels of one replay (capturing launches nothing)
            self.launches = l0
            self._pgraphs.append(g)
            self._pg_loss.append(loss)
        self._slot = 0
        return self

    # ---------------------------------------------------------------- CUDA-graph replay of the whole step
    def capture(self, ids, y, loss_kind=0):
        """Capture one step (kernels + the three NCCL collectives) into a CUDA graph over static input
        buffers.  `ids`/`y` seed the buffers; two eager warm-up steps run first (they do train)."""
        self._refuse_capture()
        self._g_ids = ids.clone()
        self._g_y = y.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.update_embedding(self._g_ids, self._g_y, loss_kind)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        l0 = self.launches
        with torch.cuda.graph(self._graph, capture_error_mode="thread_local"):
            self._g_loss = self.update_embedding(self._g_ids, self._g_y, loss_kind)
        self._graph_launches = self.launches - l0   # kernels of one replay (capturing launches nothing)
        self.launches = l0
        return self

    def step_graphed(self, ids, y):
        """same as update_embedding(ids, y) through the captured graph (ids/y copied into its buffers)."""
        self._g_ids.copy_(ids, non_blocking=True)
        self._g_y.copy_(y, non_blocking=True)
        self._graph.replay()
        self.launches += self._graph_launches
        return self._g_loss

    def capture_pipelined(self, ids, y, loss_kind=0):
        """Capture the pipelined step for both buffer-set parities.  `ids`/`y` seed the static buffers; two eager
        warm-up steps run first (they do train).  Afterwards call prepare(first ids), then step_graphed_pipelined."""
        self._refuse_capture()
        self._g_ids = ids.clone()
        self._g_y = y.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.prepare(self._g_ids)
            for _ in range(2):
                self.update_embedding_pipelined(self._g_y, self._g_ids, loss_kind)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._pgraphs, self._pg_loss = [], []
        for parity in (0, 1):
            self._slot = parity
            g = torch.cuda.CUDAGraph()
            l0 = self.launches
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                loss = self.update_embedding_pipelined(self._g_y, self._g_ids, loss_kind)
            self._graph_launches = self.launches - l0   # kernels of one replay (capturing launches nothing)
            self.launches = l0
            self._pgraphs.append(g)
            self._pg_loss.append(loss)
        self._slot = 0
        return self

    _POLL_EVERY = 256      # steps between two reads of the device error words (a read synchronises the stream)

    def _poll(self):
        """A field that overflowed its per-field sort capacity loses gradient contributions, an exchange that timed out
        leaves stale partials: neither may train on silently.  Both error words are read every _POLL_EVERY steps (and by
        bench_main at the end) and raise."""
        self._steps_since_poll = getattr(self, "_steps_since_poll", 0) + 1
        if self._steps_since_poll >= self._POLL_EVERY:
            self._steps_since_poll = 0
            self.check_overflow()
            self.check_exchange()

    def step_graphed_pipelined(self, y, ids_next):
        """update_embedding_pipelined(y, ids_next) through the captured graphs."""
        self._poll()
        self._g_y.copy_(y, non_blocking=True)
        self._g_ids.copy_(ids_next, non_blocking=True)
        p = self._slot
        self._pgraphs[p].replay()
        self.launches += self._graph_launches
        self._slot = 1 - p
        return self._pg_loss[p]

    def check_overflow(self):
        v = int(self.overflow.item())
        if v:
            raise RuntimeError(f"a field had {v} owned entries on one rank, more than the per-field sort capacity")


# ------------------------------------------------------------------ bench.py --gpus N (N > 1)
def bench_main(args, sizes, config):
    """weak scaling: every rank trains on its own batch of args.batch samples per step."""
    from bench import ClockSampler, measured_peaks, synth_batches  # noqa: WPS433 (bench.py is the caller)
    world, rank = dist.get_world_size(), dist.get_rank()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    B, F, k = args.batch, len(sizes), 10
    K, W = args.steps, max(args.warmup, 3)
    model = ShardedFM(sizes, k, n=1e-4, seed=0)
    NB = 8
    host = synth_batches(sizes, B, NB, 1234 + rank)
    enc = [model.encode(Xi, Y) for Xi, Y in host]
    stream = torch.cuda.current_stream()
    use_graph = os.environ.get("FMB_NO_GRAPH", "0") != "1"
    pipelined = os.environ.get("FMB_SHARD_PIPELINE", "1") != "0"
    # exchanges: "peers" = stores into peer-mapped symmetric memory + epoch flags (default), "nccl" = collectives
    # "fused" = csrc/shard3.cu, one kernel per rank per step.  Default where it measured faster: 99 us against 122 us per step
    # at 2 GPUs; at 8 GPUs it is correct (tests/sharded_pipeline_check.py --fused) but slower (228 against 213 us), see DESIGN.md 5
    default_exchange = "fused" if world == 2 else "peers"
    exchange = os.environ.get("FMB_SHARD_EXCHANGE", default_exchange) if pipelined else "nccl"
    fused = exchange == "fused"          # csrc/shard3.cu: the step as one kernel with per-tile flags (needs the peer mapping)
    if fused and not model.fused_supported(B):
        print(f"[rank {rank}] fused sharded step does not support this shape; using the three-kernel peer path", file=sys.stderr, flush=True)
        fused = False
    if exchange == "fused":
        exchange = "peers"
    if exchange == "peers":
        # mapping the peers' buffers needs symmetric-memory support on this box; every rank must take the same path,
        # so the ranks agree (all-reduce of a success flag) and fall back to the NCCL exchange together, loudly
        ok = 1
        try:
            model._peer_setup(B)
        except Exception as exc:  # noqa: BLE001 - any failure means "no peer mapping here"
            ok = 0
            print(f"[rank {rank}] symmetric-memory mapping failed ({type(exc).__name__}: {exc}); "
                  "using the NCCL exchange", file=sys.stderr, flush=True)
        flag = torch.tensor([ok], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            exchange = "nccl"
            model._peer = None
    fused = fused and exchange == "peers"
    state = {}

    def setup(fused_now):
        """(re)build the step function for the chosen exchange; returns (prepare, run, step)"""
        prepare = model.prepare_fused if fused_now else (model.prepare_peers if exchange == "peers" else model.prepare)
        if pipelined:
            # step i trains on batch i while batch i+1's ids are exchanged and sorted (update_embedding_pipelined)
            if use_graph:
                (model.capture_fused if fused_now else model.capture_peers if exchange == "peers" else model.capture_pipelined)(*enc[0])
                run = model.step_graphed_pipelined
            else:
                run = (model.update_embedding_fused if fused_now else
                       model.update_embedding_peers if exchange == "peers" else model.update_embedding_pipelined)
            prepare(enc[0][0])

            def step(i):
                return run(enc[i % NB][1], enc[(i + 1) % NB][0])
        else:
            if use_graph:
                model.capture(*enc[0])
                run = model.step_graphed
            else:
                run = model.update_embedding

            def step(i):
                return run(*enc[i % NB])
        state.update(prepare=prepare, run=run, step=step)

    setup(fused)
    if fused:
        # a trial round: a tile whose owned entries exceed its shared-memory capacity (ids whose hot rows concentrate on one
        # rank) or a flag time-out raises the error word; every rank then falls back to the three-kernel path together
        for i in range(2 * NB):
            state["step"](i)
        torch.cuda.synchronize()
        bad = torch.tensor([int(model._peer["error"].item()) != 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        if int(bad.item()):
            print(f"[rank {rank}] fused sharded step raised its error word ({int(model._peer['error'].item())}); "
                  "falling back to the three-kernel peer path", file=sys.stderr, flush=True)
            model._peer["error"].zero_()
            fused = False
            torch.cuda.synchronize()
            dist.barrier()
            setup(False)
    prepare, run, step = state["prepare"], state["run"], state["step"]
    sampler = ClockSampler(local)   # started before the warm-up: the timed region is a few ms, nvidia-smi needs ~50 ms to start
    W_run = max(W, 2 * NB + 2)      # at least two rounds over the rotating batches (reported: the requested W)
    for i in range(W_run):
        step(i)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    l0 = model.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(K):
        step(W_run + i)
    ev1.record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    launches = model.launches - l0
    # e2e: host ids/labels of this rank in, loss out, every step
    hosts = [(np.ascontiguousarray((Xi + model.offsets_np[:-1][None, :]).astype(np.int32)), Y) for Xi, Y in host]
    pin_i = torch.empty(B, F, dtype=torch.int32).pin_memory()
    pin_y = torch.empty(B, dtype=torch.float32).pin_memory()
    d_i = torch.empty(B, F, dtype=torch.int32, device="cuda")
    d_y = torch.empty(B, device="cuda")

    def host_step(i):
        # this step's labels and (pipelined) the NEXT batch's ids come from pinned host memory every step
        ids_h = hosts[(i + 1) % NB][0] if pipelined else hosts[i % NB][0]
        pin_i.numpy()[...] = ids_h
        pin_y.numpy()[...] = hosts[i % NB][1]
        d_i.copy_(pin_i, non_blocking=True)
        d_y.copy_(pin_y, non_blocking=True)
        return float((run(d_y, d_i) if pipelined else run(d_i, d_y)).item())

    if pipelined:   # the e2e sequence starts over at batch 0: restart the pipeline there
        prepare(enc[0][0])
    for i in range(W):
        host_step(i)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for i in range(K):
        host_step(W + i)
    torch.cuda.synchronize()
    dist.barrier()
    e2e = torch.tensor([time.perf_counter() - t0], device="cuda")
    dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
    clocks = sampler.stop()
    model.check_overflow()
    model.check_exchange()
    dist.barrier()
    if rank == 0:
        value = world * B * K / (ms * 1e-3)
        step_bytes = B * (8 * F * (k + 1) + 8 * F + 8)
        step_gbps = step_bytes / (ms / K * 1e-3) / 1e9
        peaks, peak_src = measured_peaks()
        line = {
            "metric": "train samples/sec (fwd+bwd+update)", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(config, parallelism=f"row-sharded tables over {world} GPUs (r % G); ids / pooled partials / "
                                               "sample contexts exchanged by " +
                                               ("stores into peer-mapped symmetric memory inside ONE fused step kernel per rank (tiles "
                                                "keep their rows in shared memory across both exchanges; per-tile flags; no NCCL "
                                                "in the step)" if fused else
                                                "stores into peer-mapped symmetric memory + epoch flags (no NCCL in the step)"
                                                if exchange == "peers" else "NCCL all-gather + all-to-all + all-gather") +
                                               ("; next batch's id exchange + owner sort overlapped" if pipelined else ""),
                          global_batch=world * B),
            "clocks": clocks,
            "e2e": {"value": world * B * K / float(e2e.item()), "unit": "samples/s",
                    "h2d_bytes_per_step": 4 * B * F + 4 * B, "d2h_bytes_per_step": 4,
                    "api": ("ShardedFM.update_embedding_fused" if fused else
                            "ShardedFM.update_embedding_peers" if exchange == "peers" else
                            "ShardedFM.update_embedding_pipelined" if pipelined else "ShardedFM.update_embedding") +
                           " (pinned host ids/y in, loss out, per rank)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "whole sharded step, per GPU (no single dominant kernel: see DESIGN.md 5)",
                         "achieved": step_gbps, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": step_gbps / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": step_bytes,
                         "note": "algorithmic bytes of one GPU's 8 192-sample share of the step / step time; the "
                                 "per-kernel roofline and DRAM traffic are reported by the N=1 run"},
        }
        print(json.dumps(line), flush=True)
    # leave without tearing the communicator down: destroy_process_group() after CUDA-graph captured
    # collectives was observed to hang on this stack (torch 2.11 / NCCL 2.28); every rank has finished
    # its work and rank 0 has printed, so a plain exit is safe.
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)
