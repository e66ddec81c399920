#!/usr/bin/env python
"""bench.py -- train samples/s (fwd + bwd + update) of the FM hot path on B200, with roofline and
CPU-baseline evidence.  Contract: see DESIGN.md "Measurement".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg5|cfg4]
                    [--dump-outputs DIR]

A "step" is one `update_embedding` (forward_fm + BCEWithLogits + sparse backward + fresh-Adam row
update, the reference's pre-training hot loop main_experiment.py:92-105) over one batch of 8192
synthetic Criteo-shaped samples per GPU.  Workload cfg5 = BASELINE.json configs[4]: 39 fields,
33 M embedding rows (1.6 GB packed, far larger than the 126 MB L2), k = 10.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CRITEO_SMALL13 = [63, 113, 126, 51, 224, 148, 100, 79, 104, 9, 32, 57, 82]
CRITEO_TINY = CRITEO_SMALL13 + [1457, 555, 176373, 129683, 305, 19, 11887, 632, 3, 41738, 5170, 175446, 3170, 27,
                                11356, 165602, 10, 4641, 2030, 4, 172761, 18, 15, 57903, 86, 44549]


def feature_sizes(workload):
    if workload == "cfg4":
        return list(CRITEO_TINY)  # main_experiment.py:56-58, sum = 1 006 628
    if workload == "cfg5":
        return CRITEO_SMALL13 + [1_269_185] * 26  # 13 dense-bucket fields + 26 categorical, sum = 33 000 000 - 4
    raise SystemExit(f"unknown workload {workload}")


def synth_batches(sizes, B, nb, seed):
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(nb):
        Xi = np.stack([rng.randint(0, fs, size=B) for fs in sizes], 1).astype(np.int64)
        Y = (rng.uniform(size=B) < 0.3).astype(np.float32)
        out.append((Xi, Y))
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region, every 200 ms like the profiling recipe's clocks
    line (a 50 ms loop slowed the host entry point's submissions by a third: every poll takes the driver's lock)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.p = None
        self.gpu = gpu_index
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:   # the sampler never got a line out (very short run): one synchronous query, flagged as such
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout
                f = [x.strip() for x in out.strip().splitlines()[0].split(",")]
                sm.append(float(f[0])); mx.append(float(f[1]))
                reasons.add("sampled after the timed region")
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def cpu_port_rate(sizes, k, B, budget_s, seed=0, threads=None):
    """The oracle port (C; ORC_THREADS host threads: samples in parallel in the forward pass, fields in parallel in
    the backward pass, same results as one thread) timed on this box's host cores on the same workload."""
    from oracle.deep import OracleDeep
    os.environ["ORC_THREADS"] = str(threads or os.cpu_count() or 1)
    orc = OracleDeep("DeepFMAdam", sizes, k, 3, 400, lr=1e-4, seed=seed)
    batches = synth_batches(sizes, B, 4, 99)
    ones = np.ones((B, len(sizes)), np.float32)
    orc.update_embedding(batches[0][0], ones, batches[0][1])  # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        Xi, Y = batches[n % len(batches)]
        orc.update_embedding(Xi, ones, Y)
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= 20000:
            break
    dt = time.perf_counter() - t0
    return n * B / dt, n, dt


def reference_classes_rate(B=8192, steps=5, threads=None):
    """The reference's OWN classes (oracle/_ref, copied there unmodified by __graft_entry__.build()) on this box's host
    cores: DeepFMAdam(use_cuda=False).update_embedding at BASELINE.json configs[3]'s shape (the Criteo-tiny tables of
    main_experiment.py:56-58; the 33 M-row tables of configs[4] would need minutes per step: the reference's Adam step is
    dense over every row).  ndarray inputs (the reference converts them per call)."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref, "models")):
        return {"unavailable": "oracle/_ref not populated (run __graft_entry__.build() where the reference checkout exists)"}
    import types
    import torch
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib"); mpl.use = lambda *a, **k: None
        plt = types.ModuleType("matplotlib.pyplot"); mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl; sys.modules["matplotlib.pyplot"] = plt
    sys.path.insert(0, ref)
    try:
        from models.models_online_deep.deepfm_adam import DeepFMAdam as RefDeepFMAdam
        threads = threads or os.cpu_count() or 1
        torch.set_num_threads(threads)
        torch.manual_seed(0)
        sizes = list(CRITEO_TINY)
        m = RefDeepFMAdam(sizes, embedding_size=10, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-4, use_cuda=False)
        batches = synth_batches(sizes, B, 2, 99)
        ones = np.ones((B, len(sizes)), np.float32)
        m.update_embedding(batches[0][0], ones, batches[0][1])   # warm-up
        t0 = time.perf_counter()
        for i in range(steps):
            m.update_embedding(batches[i % 2][0], ones, batches[i % 2][1])
        dt = time.perf_counter() - t0
        rec = {"value": steps * B / dt, "unit": "samples/s", "cores": threads, "kind": "reference",
               "sample": f"{steps} DeepFMAdam(use_cuda=False).update_embedding steps of B={B} at configs[3]'s shape "
                         f"(F=39, R=1006628, k=10) in {dt:.1f}s, torch {torch.__version__} CPU, {threads} threads"}
        # SURVEY.md 8(d): the same step with the scripts' real inputs (Python lists of lists, converted by the reference on
        # every call: deepfm_adam.py:47-48,57-58) and on ONE host thread
        lists = [(b[0].tolist(), ones.tolist(), b[1].tolist()) for b in batches]
        t0 = time.perf_counter()
        for i in range(2):
            m.update_embedding(*lists[i % 2])
        rec["list_inputs"] = {"value": 2 * B / (time.perf_counter() - t0), "unit": "samples/s", "cores": threads,
                              "sample": "2 steps, Xi / Xv / Y as Python lists (the scripts' interface)"}
        torch.set_num_threads(1)
        t0 = time.perf_counter()
        for i in range(2):
            m.update_embedding(batches[i % 2][0], ones, batches[i % 2][1])
        rec["one_thread"] = {"value": 2 * B / (time.perf_counter() - t0), "unit": "samples/s", "cores": 1,
                             "sample": "2 steps, ndarray inputs, torch.set_num_threads(1)"}
        torch.set_num_threads(threads)
        return rec
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": f"{type(exc).__name__}: {exc}"}
    finally:
        sys.path.remove(ref)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]


def cfg4_fit_record(lib, steps=30):
    """BASELINE.json configs[3]: DeepFMAdam.fit (forward + tower backward + table / tower / bias updates) at B = 8192 with
    the tcgen05 3xTF32 tower: a second, tensor-bound record carried inside the bench line."""
    import torch
    import fm_for_online_recommendation_b200 as pkg
    B, k, L, H = 8192, 10, 3, 400
    torch.manual_seed(0)
    m = pkg.DeepFMAdam(CRITEO_TINY, embedding_size=k, num_hidden_layers=L, neuron_per_hidden_layer=H, n=1e-4)
    enc = [m.encode(Xi, None, Y) for Xi, Y in synth_batches(CRITEO_TINY, B, 4, 7)]
    for i in range(4):
        m._deep_fit_graphed(enc[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        m._deep_fit_graphed(enc[i % 4])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    flop = 2 * B * (k * H + (L - 1) * H * H) * 3          # forward + dX + dW products of the tower
    peaks, _ = measured_peaks()
    tf32x3_peak = 1100.0 / 3                                # nominal dense TF32 (1.1 PFLOP/s) / 3 products per fp32-grade product
    hedge = None
    try:   # DeepFMOnn.fit at the same shape (hedge backpropagation, single backward pass with per-head injection)
        torch.manual_seed(0)
        mo = pkg.DeepFMOnn(CRITEO_TINY, embedding_size=k, num_hidden_layers=L, neuron_per_hidden_layer=H, n=1e-4, batch_size=B)
        for i in range(4):
            mo._hedge_fit_graphed(enc[i % 4])
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for i in range(steps):
            mo._hedge_fit_graphed(enc[i % 4])
        h1.record()
        torch.cuda.synchronize()
        hms = h0.elapsed_time(h1) / steps
        hedge = {"workload": "cfg4: DeepFMOnn.fit (hedge backpropagation), same shape", "ms_per_step": hms,
                 "value": B / (hms * 1e-3), "unit": "samples/s"}
        del mo
    except Exception as exc:  # noqa: BLE001
        hedge = {"unavailable": f"{type(exc).__name__}: {exc}"}
    return {"hedge_fit": hedge, "workload": "cfg4: DeepFMAdam.fit, B=8192, k=10, tower 10-400-400-400, F=39, R=1006628", "steps": steps,
            "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": "samples/s",
            "roofline": {"bound": "tensor", "achieved": flop / (ms * 1e-3) / 1e12, "peak": tf32x3_peak, "unit": "TFLOP/s",
                         "frac": flop / (ms * 1e-3) / 1e12 / tf32x3_peak,
                         "note": "tower flops (1.944 MFLOP/sample) over the WHOLE fit step (gather, sort and row updates "
                                 "included); peak = nominal dense TF32 / 3 (3xTF32 split); measured bf16 peak for scale: "
                                 f"{peaks.get('bf16_tflops')} TFLOP/s"},
            "tensor_core_error_flag": int(lib.fmb_gemm_tc_error())}


def run_reference(args):
    """--impl reference: the reference is pure Python/PyTorch and cannot travel to the GPU box, so this
    arm times the CPU oracle port of the same step (oracle/fm_oracle.c) on all the host cores (ORC_THREADS)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sizes = feature_sizes(args.workload)
    B = args.batch
    threads = os.cpu_count() or 1
    os.environ["ORC_THREADS"] = str(threads)
    from oracle.deep import OracleDeep
    orc = OracleDeep("DeepFMAdam", sizes, 10, 3, 400, lr=1e-4, seed=0)
    batches = synth_batches(sizes, B, 4, 99)
    ones = np.ones((B, len(sizes)), np.float32)
    for w in range(max(1, min(args.warmup, 2))):
        orc.update_embedding(batches[0][0], ones, batches[0][1])
    K = args.steps
    t0 = time.perf_counter()
    for i in range(K):
        Xi, Y = batches[i % len(batches)]
        orc.update_embedding(Xi, ones, Y)
    dt = time.perf_counter() - t0
    v = K * B / dt
    line = {"impl": "reference", "metric": "train samples/sec (fwd+bwd+update)", "value": v, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": K, "warmup": args.warmup, "ms_per_step": dt / K * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, sizes),
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": threads, "kind": "port",
                             "sample": f"{K} update_embedding steps of B={B} (oracle/fm_oracle.c, {threads} host threads: "
                                       "samples in parallel forward, fields in parallel backward)"},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "cpu_baseline_reference": reference_classes_rate()}
    print(json.dumps(line))


def workload_config(args, sizes):
    return {"workload": f"{args.workload}: DeepFMAdam.update_embedding, Criteo-shaped F={len(sizes)} fields, "
                        f"R={sum(sizes)} rows, k=10, batch {args.batch} per GPU",
            "batch_per_gpu": args.batch, "fields": len(sizes), "rows": int(sum(sizes)), "k": 10,
            "update": "fresh-Adam sign step (reference)", "l2": "tables larger than L2; a different batch every step"}


DUMP_BUDGET_BYTES = 64 << 20
DUMP_UPDATED_ROWS, DUMP_SAMPLE_ROWS, DUMP_SEED = 1 << 19, 1 << 18, 20240601


def dump_outputs(out_dir, model, batch, loss):
    """--dump-outputs: what the last timed step computed, as DIR/<name>.npy, so that two builds can be compared output
    for output.  The step returns its loss and updates the bias and the table rows its batch hits; the whole table is
    too large to store (2 GB at cfg5), so the trained columns (V, then w1) are written for the rows that step updated
    (ascending row id, a seeded subset above DUMP_UPDATED_ROWS) and for a fixed, seeded sample of all rows.  The row ids
    are written beside them (float64, exact)."""
    import torch
    k = model.embedding_size
    rng = np.random.RandomState(DUMP_SEED)
    updated = np.unique(batch.ids.cpu().numpy())
    if len(updated) > DUMP_UPDATED_ROWS:
        updated = np.sort(rng.choice(updated, DUMP_UPDATED_ROWS, replace=False))
    sample = np.unique(rng.randint(0, model._R, size=DUMP_SAMPLE_ROWS))

    def rows(ids):
        idx = torch.from_numpy(ids.astype(np.int64)).to(model.device)
        return model._table.index_select(0, idx)[:, :k + 1].cpu().numpy()

    out = {"loss": loss.reshape(1).cpu().numpy(), "bias": model.bias.detach().reshape(-1).cpu().numpy(),
           "updated_row_ids": updated.astype(np.float64), "updated_rows": rows(updated),
           "sample_row_ids": sample.astype(np.float64), "sample_rows": rows(sample)}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= DUMP_BUDGET_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import fm_for_online_recommendation_b200 as pkg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1 and args.dump_outputs:
        raise SystemExit("--dump-outputs is supported with --gpus 1 only")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sizes = feature_sizes(args.workload)
    F, k, B = len(sizes), 10, args.batch
    K, W = args.steps, max(args.warmup, 3)
    lib = pkg.require_cuda()

    if world > 1:
        # two multi-GPU designs (DESIGN.md section 5): FMB_SHARD=1 = owner-side pooled partials + owner sort of the global
        # batch (sharded.py; the faster one today), FMB_SHARD=2 = per-rank partial gradients, O(B*F) work per rank,
        # reference-order forward (sharded2.py)
        if os.environ.get("FMB_SHARD", "1") == "2":
            from fm_for_online_recommendation_b200 import sharded2
            return sharded2.bench_main(args, sizes, workload_config(args, sizes))
        from fm_for_online_recommendation_b200 import sharded
        return sharded.bench_main(args, sizes, workload_config(args, sizes))

    torch.manual_seed(0)
    model = pkg.DeepFMAdam(sizes, embedding_size=k, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-4)
    NB = 16
    host = synth_batches(sizes, B, NB, 1234 + rank)
    enc = [model.encode(Xi, None, Y) for Xi, Y in host]
    host_ids = [np.ascontiguousarray((Xi + model._offsets_np[:-1][None, :]).astype(np.int32)) for Xi, _ in host]
    host_y = [Y for _, Y in host]
    stream = torch.cuda.current_stream()
    sess = model._get_session(B)

    def step(i):
        # step on batch i; the sort of batch i+1 (it depends on the ids only) is started right behind it on a side
        # stream, so it overlaps this step's backward kernels.  Every step still sorts exactly one batch.
        return model._fm_step(enc[i % NB], 0, None if args.no_presort else enc[(i + 1) % NB])

    sampler = ClockSampler(local)       # started before the warm-up: forking nvidia-smi must not sit in front of the timed region
    base = max(W, 2 * NB + 2)           # two epochs of the rotating batches; the timed loop CONTINUES the sequence
    for i in range(base):
        step(i)
    torch.cuda.synchronize()
    launches0 = lib.fmb_session_launches(sess)
    graphs0 = lib.fmb_session_graph_count(sess)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    th0 = time.perf_counter()
    for i in range(K):
        last_loss = step(base + i)
    host_ms = (time.perf_counter() - th0) * 1e3 / K     # time the host needs to SUBMIT one step (no sync inside)
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    assert lib.fmb_session_graph_count(sess) == graphs0, "a step graph was captured inside the timed region"
    launches = lib.fmb_session_launches(sess) - launches0
    if args.dump_outputs:   # before the host-path measurements below train the same table further
        dump_outputs(args.dump_outputs, model, enc[(base + K - 1) % NB], last_loss)

    # ---- e2e: HOST buffers through the C-ABI host entry point, every step: H2D of that step's ids/labels
    # from pinned host memory + the step + D2H of its loss.  Two input slots: the copies of step t+1
    # overlap the kernels of step t (fmb_session_fm_step_host_async / fmb_session_wait_loss).
    loss = C.c_float()
    tptr, bptr = C.c_void_p(model._table.data_ptr()), C.c_void_p(model.bias.data_ptr())
    pin_ids = [torch.from_numpy(a).pin_memory() for a in host_ids]
    pin_y = [torch.from_numpy(np.ascontiguousarray(y)).pin_memory() for y in host_y]
    st = C.c_void_p(stream.cuda_stream)
    losses = []

    NSLOT = lib.fmb_session_host_slots()      # 4 input slots: the host submits up to three steps ahead of the GPU

    def submit(i):
        j = i % NB
        rc = lib.fmb_session_fm_step_host_async(sess, i % NSLOT, C.c_void_p(pin_ids[j].data_ptr()), None,
                                                C.c_void_p(pin_y[j].data_ptr()), B, tptr, bptr, model._key_bits, 0,
                                                model._lr, 0, st)
        assert rc == 0, lib.fmb_last_error()

    def collect(i):
        rc = lib.fmb_session_wait_loss(sess, i % NSLOT, C.byref(loss))
        assert rc == 0, lib.fmb_last_error()
        losses.append(loss.value)

    def run_host(n, base):
        # every step: H2D of ITS ids and labels, the step, its loss read back on the host -- collected NSLOT - 1 steps
        # later, so that the copies and the sort of the following steps overlap the kernels of this one
        for i in range(n):
            submit(base + i)
            if i >= NSLOT - 1:
                collect(base + i - (NSLOT - 1))
        for i in range(max(0, n - (NSLOT - 1)), n):
            collect(base + i)

    # warm-up of the host path: every slot's graphs (pre-sort, step) captured and replayed, and at least 50 ms of steps --
    # the first milliseconds of host-to-device traffic after a device-resident phase run at a fraction of the link's rate
    # (tools/e2e_trace.py: 103 M samples/s for the first 20 steps of a fresh process, 160-180 M after that)
    n_warm_host = max(W, 3 * NSLOT)
    run_host(n_warm_host, 0)
    t_w = time.perf_counter()
    while time.perf_counter() - t_w < 0.05 and n_warm_host < 4000:
        run_host(4 * NSLOT, n_warm_host)
        n_warm_host += 4 * NSLOT
    torch.cuda.synchronize()
    # five windows of exactly K steps each (wall clock around submit ... last loss read back, synchronised on both sides);
    # the median is reported: one host hiccup (the loop is a Python thread on a shared box) costs a window, not the number
    e2e_windows = []
    for wdw in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_host(K, 8000 + wdw * K)
        torch.cuda.synchronize()
        e2e_windows.append(time.perf_counter() - t0)
    e2e_s = float(np.median(e2e_windows))
    assert len(losses) == n_warm_host + 5 * K and all(np.isfinite(losses))
    # the same through the blocking entry point (copy, step, wait), for reference
    def host_step(i):
        j = i % NB
        rc = lib.fmb_session_fm_step_host(sess, host_ids[j].ctypes.data_as(C.c_void_p), None,
                                          host_y[j].ctypes.data_as(C.c_void_p), B, tptr, bptr, model._key_bits, 0,
                                          model._lr, 0, C.byref(loss), st)
        assert rc == 0, lib.fmb_last_error()

    for i in range(W):
        host_step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        host_step(W + i)
    torch.cuda.synchronize()
    e2e_blocking_s = time.perf_counter() - t0
    clocks = sampler.stop()

    # ---- per-kernel device time (CUDA events on the launching stream, warm L2 like the real step) for the roofline
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    N = B * F
    delta = torch.empty(B, device="cuda"); lossv = torch.empty(B, device="cuda")
    wsb = lib.fmb_sort_workspace_bytes(N); ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    sk = torch.empty(N, dtype=torch.int32, device="cuda"); pm = torch.empty(N, dtype=torch.int32, device="cuda")
    pf = torch.empty(N, dtype=torch.int32, device="cuda")
    bwsb = lib.fmb_bwd_workspace_bytes(N, k); bws = torch.empty(bwsb, dtype=torch.uint8, device="cuda")
    lossd = torch.empty(1, device="cuda")
    st = C.c_void_p(stream.cuda_stream)
    # Per-kernel device time: `reps` back-to-back launches of ONE kernel between two CUDA events on the launching stream,
    # over the rotating batches (16 x 20 MB of rows > L2), divided by reps -- the kernel's average duration without the
    # launch latency an event pair around a single launch adds (~5 us: 26.5 against 20 us for the fused kernel).
    # The kernels are the session's: the per-field sort (radix kernel of the dense fields + hash kernel of the sparse
    # fields, here one after the other), the fused kernel, the run kernel over the run list, the bias step.
    phases = {"sort": 0.0, "fm_step_fused": 0.0, "fm_bwd_runs": 0.0, "finish": 0.0}
    from fm_for_online_recommendation_b200._lib import RunList
    by_field = B <= lib.fmb_sort_fields_max_batch()
    nseg_, cap_ = C.c_int(1), C.c_int(N // 2 + 1)
    if by_field:
        lib.fmb_runlist_shape(B, F, C.byref(nseg_), C.byref(cap_))
    sparse_ok = 0 if os.environ.get("FMB_SPARSE") == "0" else 1
    NP = min(NB, 8) if B <= 16384 else 2          # batches with their own sort outputs
    sks = [torch.empty(N, dtype=torch.int32, device="cuda") for _ in range(NP)]
    pfs = [torch.zeros(N, dtype=torch.int32, device="cuda") for _ in range(NP)]
    rls = [torch.empty((nseg_.value * cap_.value, 4), dtype=torch.int32, device="cuda") for _ in range(NP)]
    rcs = [torch.zeros(2 * nseg_.value, dtype=torch.int32, device="cuda") for _ in range(NP)]
    rlds = [RunList(rls[j].data_ptr(), rcs[j].data_ptr(), nseg_.value, cap_.value) for j in range(NP)]

    def k_sort(j):
        e = enc[j % NP]
        if by_field:
            if sparse_ok:
                pfs[j % NP].zero_()      # contract of FMB_SORT_SPARSE_OK: position words of rows hit once are not written
            rc = lib.fmb_sort_fields_ex(p(e.ids), B, F, p(model._field_off_dev), p(sks[j % NP]), p(pm), p(pfs[j % NP]),
                                        C.byref(rlds[j % NP]), sparse_ok, st)
        else:
            rcs[j % NP].zero_()
            rc = lib.fmb_sort_segment(p(e.ids), N, model._key_bits, p(ws), wsb, p(sks[j % NP]), p(pm), None, None, st)
            assert rc == 0, lib.fmb_last_error()
            rc = lib.fmb_pos_flags_ex(p(sks[j % NP]), p(pm), N, p(pfs[j % NP]), C.byref(rlds[j % NP]), st)
        assert rc == 0, lib.fmb_last_error()

    def k_fused(j):
        e = enc[j % NP]
        rc = lib.fmb_fm_step_fused(p(e.ids), None, p(e.y), tptr, bptr, p(pfs[j % NP]), B, F, k, 0, model._lr, 0, p(delta),
                                   p(lossv), p(bws), bwsb, st)
        assert rc == 0, lib.fmb_last_error()

    def k_runs(j):      # over the contributions staged by the last fused launch (batch NP - 1)
        assert lib.fmb_fm_backward_runs_list(p(sks[(NP - 1) % NP]), N, tptr, F, k, model._lr, 0, None,
                                             C.byref(rlds[(NP - 1) % NP]), p(bws), bwsb, st) == 0

    def k_finish(j):
        assert lib.fmb_finish_step(p(delta), p(lossv), B, bptr, model._lr, 0, p(lossd), st) == 0

    reps = max(8, min(K, 40))
    ev0_, ev1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, fn in (("sort", k_sort), ("fm_step_fused", k_fused), ("fm_bwd_runs", k_runs), ("finish", k_finish)):
        for j in range(NP):          # warm-up (and, for the sort, the outputs the next kernels consume)
            fn(j)
        torch.cuda.synchronize()
        ev0_.record(stream)
        for j in range(reps):
            fn(j)
        ev1_.record(stream)
        torch.cuda.synchronize()
        phases[name] = ev0_.elapsed_time(ev1_) / reps
    peaks, peak_src = measured_peaks()
    kp1 = k + 1
    # algorithmic bytes per launch of the dominant kernel (DESIGN.md section 3): ids + position words + rows read + rows
    # written + delta/loss = the whole step's 8F(k+1) + 8F + 8 per sample (SURVEY.md 8d)
    step_bytes = B * (8 * F * kp1 + 8 * F + 8)
    alg_bytes = {"fm_step_fused": step_bytes}
    dom = "fm_step_fused"
    traffic, traffic_src = None, None
    try:   # DRAM bytes of that kernel from the last `ncu --set full` capture of this command (profiles/), per launch
        with open(os.path.join(ROOT, "profiles", "r2_final2_dram_traffic.json")) as f:
            tr = json.load(f)
        if B == 8192 and args.workload == "cfg5":
            kk = [x for x in tr if x.startswith("fm_step_fused_kernel")][0]
            traffic = int(tr[kk]["dram_read_bytes"] + tr[kk]["dram_write_bytes"])
            traffic_src = "profiles/r2_final2_dram_traffic.json (ncu --set full, cold cache, B=8192)"
    except Exception:
        traffic = None
    dom_kernels = "fm_step_fused_kernel (gather + logit + loss + single-hit row updates + staging)"
    achieved = alg_bytes[dom] / (phases[dom] * 1e-3) / 1e9

    value = B * K / (ms * 1e-3)
    line = {
        "metric": "train samples/sec (fwd+bwd+update)", "value": value, "unit": "samples/s", "n_gpus": 1,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, sizes),
        "clocks": clocks,
        "e2e": {"value": B * K / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": 4 * B * F + 4 * B,
                "d2h_bytes_per_step": 4,
                "api": "fmb_session_fm_step_host_async + fmb_session_wait_loss (pinned host ids/y in, loss out, "
                       "four slots: the copies and the sort of the next steps overlap the kernels of step t)",
                "windows": [round(B * K / w) for w in e2e_windows], "window_stat": "median of 5 windows of K steps",
                "blocking_value": B * K / e2e_blocking_s},
        "host_submit_ms_per_step": host_ms,
        "gpu_launches": int(launches), "step_graphs_cached": int(lib.fmb_session_graph_count(sess)),
        "roofline": {"bound": "hbm", "kernel": dom_kernels, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                     "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": alg_bytes[dom],
                     "phase_ms": phases,
                     "whole_step_GBps": step_bytes / (ms / K * 1e-3) / 1e9},
    }
    if not args.no_extra:
        try:
            line["cfg4_fit"] = cfg4_fit_record(lib)
        except Exception as exc:  # noqa: BLE001 -- the headline line must not die with the extra record
            line["cfg4_fit"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
    if not args.no_cpu_baseline:
        v, n, dt = cpu_port_rate(sizes, k, B, args.cpu_budget)
        line["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": os.cpu_count() or 1, "kind": "port",
                                "sample": f"{n} update_embedding steps of B={B} in {dt:.1f}s "
                                          f"(oracle/fm_oracle.c, all {os.cpu_count()} host threads)"}
        line["cpu_baseline_reference"] = reference_classes_rate()
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=["cfg5", "cfg4"])
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg4 DeepFMAdam.fit record")
    ap.add_argument("--no-presort", action="store_true", help="sort each batch inside its own step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is supported with --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
