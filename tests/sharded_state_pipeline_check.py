"""Pipelined, peer-memory and fused sharded steps == the eager update_embedding, bit for bit, in update modes 3 and 4
(losses, every owned row, the bias, and the optimizer state: this rank's shard and the bias state), over NCCL.

Not collected by pytest (no test_ prefix): run as a program, one process per GPU,
    python tests/sharded_state_pipeline_check.py --mode 3 [--graph]       # world 1 (tests/test_gpu_sharded_state.py runs this)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 \
        tests/sharded_state_pipeline_check.py --mode 4
--mode 3: Adagrad, 4: SparseAdam (eager only: its steps cannot be captured).  --graph: every model steps through its
captured graphs; afterwards enable_adagrad() again drops them and the next eager step equals a fresh model's.
Prints "STATE_PIPELINE_CHECK_OK ..." on rank 0 and exits 0, or raises."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fm_for_online_recommendation_b200 import sharded as sh  # noqa: E402

SIZES = [7, 3, 40, 2, 1000, 13]


def _model(mode):
    m = sh.ShardedFM(SIZES, 4, n=0.01, seed=3)
    if mode == 3:
        m.enable_adagrad(eps=1e-6, initial_accumulator_value=0.05)
    else:
        m.enable_sparse_adam()
    return m


def _same(a, b, what):
    assert torch.equal(a.table, b.table), (what, "owned rows differ")
    assert torch.equal(a.bias, b.bias), (what, "bias differs")
    sa, sb = a.local_state(), b.local_state()
    for x, y in zip(sa, sb):
        assert np.array_equal(np.asarray(x), np.asarray(y)), (what, "state differs")


def main():
    graph = "--graph" in sys.argv
    mode = int(sys.argv[sys.argv.index("--mode") + 1])
    assert mode in (3, 4) and not (graph and mode == 4)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29543")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    B, steps = 128, 7
    rng = np.random.RandomState(200 + rank)
    batches = []
    for i in range(steps):
        if i % 2:
            Xi = np.stack([np.minimum(rng.zipf(1.3, size=B) - 1, fs - 1) for fs in SIZES], 1)
        else:
            Xi = np.stack([rng.randint(0, fs, size=B) for fs in SIZES], 1)
        Y = (rng.uniform(size=B) < 0.4).astype(np.float32)
        batches.append((Xi, Y))
    a = _model(mode)
    enc = [a.encode(Xi, Y) for Xi, Y in batches]
    paths = [("pipelined", "prepare", "capture_pipelined", "update_embedding_pipelined"),
             ("peers", "prepare_peers", "capture_peers", "update_embedding_peers"),
             ("fused", "prepare_fused", "capture_fused", "update_embedding_fused")]
    if graph:
        a.capture(*enc[0])
        step_a = a.step_graphed
    else:
        step_a = a.update_embedding
    la = [float(step_a(ids, y).item()) for ids, y in enc]
    for name, prepare, capture, eager in paths:
        b = _model(mode)
        if graph:
            # capture trains two warm-up steps on enc[0], as a.capture did
            getattr(b, capture)(*enc[0])
            step_b = b.step_graphed_pipelined
        else:
            step_b = getattr(b, eager)
        getattr(b, prepare)(enc[0][0])
        lb = []
        for i in range(steps):
            nxt = enc[i + 1][0] if i + 1 < steps else (enc[0][0] if graph else None)
            lb.append(float(step_b(enc[i][1], nxt).item()))
        torch.cuda.synchronize()
        b.check_overflow()
        b.check_exchange()
        assert la == lb, (name, la, lb)
        _same(a, b, name)
        if mode == 4:
            assert a._sa.step == b._sa.step == steps, (name, a._sa.step, b._sa.step)
    if graph:
        # enable_adagrad() after a capture: the graphs are gone, the sums start over, the next step is a fresh one's
        c = _model(mode)
        c.capture(*enc[0])
        c.enable_adagrad(eps=1e-6, initial_accumulator_value=0.05)
        assert not hasattr(c, "_graph")
        d = _model(mode)
        d.table.copy_(c.table)
        d.bias.copy_(c.bias)
        lc = float(c.update_embedding(*enc[1]).item())
        ld = float(d.update_embedding(*enc[1]).item())
        assert lc == ld, (lc, ld)
        _same(c, d, "re-enabled after capture")
    a.check_overflow()
    ok = torch.ones(1, device="cuda")
    dist.all_reduce(ok)
    if rank == 0:
        print(f"STATE_PIPELINE_CHECK_OK world={world} mode={mode} graph={int(graph)} losses={la[:3]}", flush=True)
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0)   # see sharded.bench_main: no communicator teardown after graph-captured collectives


if __name__ == "__main__":
    main()
