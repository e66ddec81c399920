"""Step time of the row-sharded FM step at cfg5's per-rank shape (BASELINE.json configs[4]: 39 fields, 33 M rows, k = 10,
B = 8 192 samples per rank) in update modes 0 (the reference's fresh-Adam sign step), 3 (Adagrad) and 4 (SparseAdam on the
tables, Adam on the bias), for the three-kernel peer-memory path (update_embedding_peers) and the one-kernel path
(update_embedding_fused), measured alternately in one process.  Run under torchrun, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29533 \
        tools/bench_sharded_state.py [--steps 200] [--rounds 5] [--out profiles/sharded_state_cfg5.json]

Every step runs eagerly (mode 4 cannot be captured; the other modes are run the same way so that the comparison is fair),
on 8 rotating batches with the next batch's ids exchanged and sorted beside the step.  Each round times `steps` steps of
every (path, mode) in turn with CUDA events, so that clock and neighbour noise falls on all of them alike; rank 0 writes
every round's time (the slowest rank's), the median, the algorithmic bytes per step of one rank and the card's name and
power limit.  Needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import feature_sizes, synth_batches  # noqa: E402


def algorithmic_bytes(B, F, k, mode):
    """bytes one rank's share of the step must move (bench_main's step_bytes: ids, rows read and written, delta/loss),
    plus the state of every coordinate updated: mode 3 reads and writes one sum, mode 4 two moments"""
    per = 8 * F * (k + 1) + 8 * F + 8
    if mode == 3:
        per += 8 * F * (k + 1)
    if mode == 4:
        per += 16 * F * (k + 1)
    return B * per


def card():
    name = torch.cuda.get_device_name(torch.cuda.current_device())
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the record says so instead of guessing
        q = "unavailable (%s)" % e
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_state_cfg5.json"))
    args = ap.parse_args()
    from fm_for_online_recommendation_b200 import sharded as sh
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world, rank = dist.get_world_size(), dist.get_rank()
    sizes = feature_sizes("cfg5")
    F, k, B, NB = len(sizes), 10, args.batch, 8
    host = synth_batches(sizes, B, NB, 1234 + rank)
    runs = {}
    for path in ("three_kernel", "fused"):
        for mode in (0, 3, 4):
            m = sh.ShardedFM(sizes, k, n=1e-4, seed=0)
            if mode == 3:
                m.enable_adagrad()
            if mode == 4:
                m.enable_sparse_adam()
            enc = [m.encode(Xi, Y) for Xi, Y in host]
            if path == "fused":
                if not m.fused_supported(B):
                    raise SystemExit(f"fused sharded step: B={B} not supported at {world} GPUs")
                m.prepare_fused(enc[0][0])
                step = m.update_embedding_fused
            else:
                m.prepare_peers(enc[0][0])
                step = m.update_embedding_peers
            runs[(path, mode)] = {"m": m, "enc": enc, "step": step, "pos": 0}

    def run(key, n):
        r = runs[key]
        for _ in range(n):
            i = r["pos"]
            r["step"](r["enc"][i % NB][1], r["enc"][(i + 1) % NB][0])
            r["pos"] = i + 1

    for key in runs:                         # two rounds over the rotating batches: rows warm, every shape launched
        run(key, 2 * NB + 2)
    torch.cuda.synchronize()
    dist.barrier()
    times = {key: [] for key in runs}
    for _ in range(args.rounds):
        for key in runs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(key, args.steps)
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            times[key].append(float(ms.item()) * 1000.0 / args.steps)
    for r in runs.values():
        r["m"].check_overflow()
        r["m"].check_exchange()
    if rank == 0:
        name, power = card()
        rec = {"workload": "row-sharded FM step, cfg5 per-rank shape: B=%d per rank, F=%d, k=%d, 33 M rows, %d GPU(s), "
                           "eager steps, rotating %d batches" % (B, F, k, world, NB),
               "device": name, "power_limit_and_max_sm_clock": power, "world": world, "steps_per_round": args.steps,
               "rounds": args.rounds, "paths": {}}
        for (path, mode), ts in times.items():
            med = float(np.median(ts))
            nbytes = algorithmic_bytes(B, F, k, mode)
            rec["paths"].setdefault(path, {})[{0: "0_adam_sign", 3: "3_adagrad", 4: "4_sparse_adam"}[mode]] = {
                "us_per_step_median": round(med, 2), "us_per_step_rounds": [round(t, 2) for t in ts],
                "algorithmic_bytes_per_step_per_rank": nbytes, "algorithmic_bytes_per_sample": nbytes // B,
                "algorithmic_GB_per_s_per_rank": round(nbytes / (med * 1e-6) / 1e9, 1)}
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
        print(json.dumps(rec), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)   # see sharded.bench_main: no communicator teardown


if __name__ == "__main__":
    main()
