"""Step time of the cfg5 update_embedding step (BASELINE.json configs[4]: 39 fields, 33 M rows, k = 10, B = 8192, the
FM step of DeepFMAdam) in update modes 0 (the reference's fresh-Adam sign step), 1 (SGD) and 3 (Adagrad), measured
alternately in one process on the rotating batches bench.py uses (16 batches, the sort of the next batch riding along).

    python tools/bench_adagrad.py [--steps 200] [--rounds 5] [--out profiles/adagrad_cfg5.json]

Each round times `steps` steps of every mode with CUDA events, the modes in turn, so that clock and neighbour noise falls
on all of them alike; the record holds every round's time per mode, the median, the algorithmic bytes per step
(ids + position words + rows read and written + delta/loss, plus the sums read and written in mode 3) and the card's name
and power limit.  Needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import feature_sizes, synth_batches  # noqa: E402


def algorithmic_bytes(B, F, k, mode):
    """bytes the step must move per batch (fm_step.cu header): ids 4F + position/flag words 4F + rows read and written
    2 * 4F(k+1) + delta/loss 8, per sample; mode 3 also reads and writes the sums of every coordinate it updates"""
    per = 4 * F + 4 * F + 8 * F * (k + 1) + 8
    if mode == 3:
        per += 8 * F * (k + 1)
    return B * per


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the record says so instead of guessing
        q = "unavailable (%s)" % e
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "adagrad_cfg5.json"))
    args = ap.parse_args()
    import fm_for_online_recommendation_b200 as pkg
    pkg.require_cuda()
    torch.cuda.set_device(0)
    sizes = feature_sizes("cfg5")
    F, k, B, NB = len(sizes), 10, args.batch, 16
    models = {}
    for mode in (0, 1, 3):
        torch.manual_seed(0)
        m = pkg.DeepFMAdam(sizes, embedding_size=k, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-4,
                           update_mode=min(mode, 1))
        if mode == 3:
            m.enable_adagrad()
        models[mode] = m
    host = synth_batches(sizes, B, NB, 1234)
    enc = {mode: [m.encode(Xi, None, Y) for Xi, Y in host] for mode, m in models.items()}
    pos = {mode: 0 for mode in models}

    def run(mode, n):
        m, e = models[mode], enc[mode]
        for _ in range(n):
            i = pos[mode]
            m._fm_step(e[i % NB], 0, e[(i + 1) % NB])
            pos[mode] = i + 1

    for mode in models:                      # two epochs of the rotating batches: graphs captured, rows warm
        run(mode, 2 * NB + 2)
    torch.cuda.synchronize()
    times = {mode: [] for mode in models}
    for _ in range(args.rounds):
        for mode in models:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(mode, args.steps)
            e1.record()
            torch.cuda.synchronize()
            times[mode].append(e0.elapsed_time(e1) * 1000.0 / args.steps)
    name, power = card()
    rec = {"workload": "cfg5 update_embedding (DeepFMAdam FM step), B=%d, F=%d, k=%d, rotating %d batches" % (B, F, k, NB),
           "device": name, "power_limit_and_max_sm_clock": power, "steps_per_round": args.steps, "rounds": args.rounds,
           "modes": {}}
    for mode, ts in times.items():
        med = float(np.median(ts))
        nbytes = algorithmic_bytes(B, F, k, mode)
        rec["modes"][{0: "0_adam_sign", 1: "1_sgd", 3: "3_adagrad"}[mode]] = {
            "us_per_step_median": round(med, 2), "us_per_step_rounds": [round(t, 2) for t in ts],
            "algorithmic_bytes_per_step": nbytes, "algorithmic_bytes_per_sample": nbytes // B,
            "algorithmic_GB_per_s": round(nbytes / (med * 1e-6) / 1e9, 1)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
