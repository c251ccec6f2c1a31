#!/usr/bin/env python
"""Benchmark of the Tacotron synthesis forward path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path -- embeddings -> encoder CBHG ->
attention decoder loop -> post-net CBHG -> linear dense -- over one synthetic
batch: BASELINE.json config 3, multispeaker free-running synthesis, batch 32
per GPU, ~100 pinyin symbols, max_iters=200 at r=5 (1000 mel frames per
utterance), mel + post-net linear output.  Metric: mel frames/s (whole job).

 * value : inputs already resident in HBM, K back-to-back steps between CUDA
           events, barrier + synchronize on both sides, max over ranks.
 * e2e   : the same step through the C-ABI host calls (taco_forward_host_begin /
           _wait / _end) with HOST buffers: H2D of ids/lengths/speakers and D2H of
           mel, linear and alignments inside the timed region; several batches in
           flight (one handle, stream and pinned buffer set each).
 * roofline : the decoder loop kernel (the dominant kernel): algorithmic bytes
           per launch (SURVEY.md §8d: 12.90 MB/step fp32 at N=32,T_in=100) over
           its CUDA-event duration, against the measured HBM copy peak.
 * cpu_baseline : the CPU oracle (restatement of the reference's TF graph; TF
           itself cannot run here) on the host cores, one full batch.

Extra keys of the line (informational, none of them changes `value`):
 single_stream   one batch in flight (step latency);
 throughput_mode the same two legs with taco_set_decoder_clusters(4);
 bf16_mode       taco_set_gemm_mode(2) (plain bf16 operands; NOT the headline precision);
 latency_batch1  p50 of one utterance, T_in 20..200, and down to the waveform;
 vocoder         taco_griffin_lim on the batch's linear output (100 iterations);
 config1 / config2 / config4 / config5 / e2e_synthesize   the other BASELINE.json configurations (bench_configs.py):
                 single speaker, teacher forced in both BN modes, global batch 256 sharded (strong scaling) with a timed
                 NCCL gather, the full batch-1 latency sweep (p50 + p99, r = 5 and r = 1), and the reference
                 Synthesizer.synthesize shape (ids -> wav + alignment);
 e2e.ms_per_step_runs   the three timed end-to-end regions (the median is `e2e.value`), e2e.d2h_floor_ms_per_step the
                 device-to-host copy time of one batch's outputs alone (measured link rate);
 gpu_launches    kernels of this library launched inside the timed region (CUDA-graph replays count their kernel nodes).
The forward and the vocoder replay CUDA graphs after their second identical call (taco_set_cuda_graphs).

`--impl reference` times that CPU restatement alone (rank 0 only).
`--dump-outputs DIR` writes, after the timed steps, what the last step returned for rank 0's first batch as DIR/<name>.npy
(float32 / float64, 46 MB): mel_outputs and alignments whole, linear_outputs_sampled at the seeded frame indices
linear_outputs_frames, and steps.  Inputs and weights are seeded, so two builds (or the two --impl arms, which run the
same batch) can be compared output for output.
N > 1: launched under torchrun, one rank per GPU, each rank runs its own batch
of 32 utterances (weak scaling, no collective on the data path).
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "mel_frames_per_s"
UNIT = "frames/s"
BATCH, T_IN, MAX_ITERS, R, ID_NUM = 32, 100, 200, 5, 60
DUMP_LINEAR_FRAMES, DUMP_MAX_BYTES = 250, 64 * 10**6   # --dump-outputs: 46 MB at config 3


def bind_to_gpu_numa_node(torch, local: int):
    """Pin this rank's host threads (and so, by first touch, its pinned output buffers) to the NUMA node its GPU hangs off:
    with eight ranks copying 144 MB per batch each to buffers that all sit on one node, the device-to-host rate fell to
    13 GB/s per GPU (VERDICT round 1).  Returns {"node": n, "cpus": k} or None when the topology cannot be read."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        if bus is None:
            out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                                 capture_output=True, text=True, timeout=20).stdout.strip()
            bus_id = out.lower()
            if bus_id.startswith("00000000:"):
                bus_id = "0000:" + bus_id[len("00000000:"):]
        else:
            dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
            dev_id = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
            bus_id = "%04x:%02x:%02x.0" % (dom, bus, dev_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus_id) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus": len(allowed)}
    except Exception:
        return None


def make_batch(seed: int):
    """BASELINE.md config 3 inputs: lengths ~U{60..100}, ids in the pinyin-phone block, pad id 0."""
    rng = np.random.default_rng(seed)
    lengths = rng.integers(60, T_IN + 1, (BATCH,)).astype(np.int32)
    ids = rng.integers(7108, 7325, (BATCH, T_IN)).astype(np.int32)
    for i in range(BATCH):
        ids[i, lengths[i]:] = 0
    spk = rng.integers(0, ID_NUM, (BATCH,)).astype(np.int32)
    return ids, lengths, spk


def workload_config(n_gpus: int):
    return {
        "workload": "BASELINE config 3: multispeaker free-running synthesis, batch %d per GPU, T_in<=%d "
                    "(lengths U{60..100}), max_iters=%d, r=%d (%d mel frames/utterance), mel + post-net linear"
                    % (BATCH, T_IN, MAX_ITERS, R, MAX_ITERS * R),
        "global_batch": BATCH * n_gpus,
        "frames_per_step": BATCH * n_gpus * MAX_ITERS * R,
        "parallelism": "utterance-sharded replicas x%d (no data-path collective)" % n_gpus,
        "weights": "random init with the reference's initializers (seed 1234); 8.80 M params",
        "l2": "per-step working set ~0.5 GB (post-net activations) exceeds the 126 MB L2; weights (35 MB) stay resident",
    }


_JSON_OUT = None


def emit(line) -> None:
    """The one JSON line of the run, on the process's original stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        self.lines = []
        exe = shutil.which("nvidia-smi")
        if exe is None:
            return
        try:
            self.proc = subprocess.Popen([exe, "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_restatement_seconds(n_threads: int, batch: int = BATCH):
    """One full batch through the oracle (the reference graph restated op by op on torch CPU)."""
    import torch
    from oracle import taco_oracle as O
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    torch.set_num_threads(n_threads)
    hp = HParams(outputs_per_step=R, max_iters=MAX_ITERS)
    w = O.W(random_init(hp, ID_NUM, seed=1234))
    ids, lengths, spk = make_batch(1)
    ids, lengths, spk = ids[:batch], lengths[:batch], spk[:batch]
    t0 = time.perf_counter()
    out = O.tacotron_forward(w, hp, ids, lengths, identities=spk, id_num=ID_NUM)
    dt = time.perf_counter() - t0
    frames = out["mel_outputs"].shape[0] * out["mel_outputs"].shape[1]
    return dt, frames, out


def dump_arrays(mel, linear, alignments, steps):
    """What a caller of the timed path receives from one step, as host float arrays (torch tensors on any device in):
    mel [N, T, 80] and alignments [N, T_in, steps] whole, linear [N, T, 1025] (131 MB at config 3) at DUMP_LINEAR_FRAMES
    frame indices drawn with a fixed seed (stored as linear_outputs_frames), and the decoder step count."""
    frames = np.sort(np.random.default_rng(0).choice(linear.shape[1], min(DUMP_LINEAR_FRAMES, linear.shape[1]), replace=False))
    arrays = {"mel_outputs": mel.cpu().numpy(), "alignments": alignments.cpu().numpy(),
              "linear_outputs_sampled": linear.cpu().numpy()[:, frames], "linear_outputs_frames": frames.astype(np.float64),
              "steps": np.float64(steps)}
    arrays = {k: np.ascontiguousarray(v, np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    return arrays


def write_dump(path: str, arrays) -> None:
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_reference(args):
    """`--impl reference`: the CPU restatement of the reference graph, host cores only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    times, frames = [], 0
    for i in range(args.warmup + args.steps):
        dt, frames, out = cpu_restatement_seconds(cores)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        write_dump(args.dump_outputs, dump_arrays(out["mel_outputs"], out["linear_outputs"], out["alignments"], out["steps"]))
    ms = 1e3 * float(np.mean(times))
    value = frames / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "one full batch (32 utterances x 1000 frames) per step; CPU restatement of the "
                                   "reference TF graph in torch-CPU fp32 (TensorFlow 1.x is not installable here)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def run_ours(args):
    import torch
    from tacotron_multispeaker_b200 import _abi
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(torch, local) if os.environ.get("TACO_BENCH_NUMA", "1") != "0" else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    hp = HParams(outputs_per_step=R, max_iters=MAX_ITERS)
    weights = random_init(hp, ID_NUM, seed=1234)
    dev = torch.device("cuda", local)
    T_out = MAX_ITERS * R
    n_dev = max(1, args.inflight)            # lanes of the device-resident measurement
    n_lanes = max(n_dev, args.e2e_lanes)     # lanes of the end-to-end measurement (their D2H traffic needs more of them)
    # One handle (own weights copy, workspace and CUDA stream) per batch in flight: the decoder loop
    # occupies 112 of the 148 SMs for 2.2 ms, another batch's encoder / post-net (GEMMs, 64-CTA BiGRU) fills the rest and the gaps.
    # more waiting host threads than cores (8 ranks x 6 lanes on 16 cores): let the C ABI's waits sleep instead of spin
    if "TACO_BLOCKING_SYNC" not in os.environ and world * (n_lanes + 1) > (os.cpu_count() or 1):
        os.environ["TACO_BLOCKING_SYNC"] = "1"
    lanes = []
    for li in range(n_lanes):
        e = Engine(hp, ID_NUM, local)
        e.load_weights(weights)
        ids_h, len_h, spk_h = make_batch(1 + rank + 100 * li)
        lanes.append(dict(
            eng=e, stream=torch.cuda.Stream(device=dev),
            ids=torch.from_numpy(ids_h).to(dev), lengths=torch.from_numpy(len_h).to(dev),
            spk=torch.from_numpy(spk_h).to(dev), host=(ids_h, len_h, spk_h),
            outs=(torch.zeros(BATCH, T_out, hp.num_mels, device=dev),
                  torch.zeros(BATCH, T_out, hp.num_freq, device=dev),
                  torch.zeros(BATCH, T_IN, MAX_ITERS, device=dev))))
    eng = lanes[0]["eng"]
    ids_h, len_h, spk_h = lanes[0]["host"]

    def step(l):
        return l["eng"].forward(l["ids"], l["lengths"], l["spk"], out=l["outs"])

    def timed(active, n_steps):
        """n_steps forward passes spread over the lanes in `active` (one host thread + stream each);
        device time from a common start event to the last lane's end event."""
        barrier()
        start = torch.cuda.Event(enable_timing=True)
        start.record()
        ends, taken = [], []

        def work(l, k):
            with torch.cuda.stream(l["stream"]):
                l["stream"].wait_event(start)
                st = 0
                for _ in range(k):
                    l["last"] = step(l)
                    st = l["last"][3]
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                ends.append(ev)
                taken.append(st)
        share = [n_steps // len(active) + (1 if i < n_steps % len(active) else 0) for i in range(len(active))]
        if len(active) == 1:
            work(active[0], share[0])
        else:
            ths = [threading.Thread(target=work, args=(l, k)) for l, k in zip(active, share) if k > 0]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        barrier()
        ms = max(start.elapsed_time(ev) for ev in ends)
        if dist is not None:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms, taken[0]

    # ---- device-resident throughput ----
    for l in lanes:
        with torch.cuda.stream(l["stream"]):
            for _ in range(max(args.warmup, 3)):
                step(l)
        l["eng"].check_ids()
    dev_lanes = lanes[:n_dev]
    sampler = ClockSampler(local) if rank == 0 else None
    timed(dev_lanes, 2 * n_dev)                      # warm the concurrent schedule too
    if sampler is not None and sampler.proc is not None:   # nvidia-smi needs a moment to start: wait for its first sample
        t_dead = time.time() + 3.0
        while not sampler.lines and time.time() < t_dead:
            time.sleep(0.02)
    launches0 = sum(l["eng"].launch_count() for l in lanes)
    t_wall0 = time.time()
    ms_total, steps_taken = timed(dev_lanes, args.steps)
    launches = sum(l["eng"].launch_count() for l in lanes) - launches0
    # lane 0 always takes part and recomputes its one batch every step; the legs below overwrite its output buffers
    dump = dump_arrays(*lanes[0]["last"]) if args.dump_outputs and rank == 0 else None
    ms_per_step = ms_total / args.steps
    frames_per_step = BATCH * steps_taken * R * world
    value = frames_per_step / (ms_per_step / 1e3)
    # the same K steps strictly one after the other on one stream (step latency)
    ms_single, _ = timed(lanes[:1], args.steps)
    single = {"ms_per_step": ms_single / args.steps, "value": frames_per_step / (ms_single / args.steps / 1e3),
              "unit": UNIT, "note": "one batch in flight (step latency)"}
    t_wall1 = time.time()                            # clocks sampled over both timed regions (GPU busy throughout)
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None

    # ---- decoder-kernel roofline (measured live, CUDA events on the launch stream) ----
    eng.set_profiling(True)
    dk = []
    for _ in range(3):
        step(lanes[0])
        dk.append(eng.last_stage_ms())
    eng.set_profiling(False)
    stage = {k: float(np.mean([d[k] for d in dk])) for k in dk[0]}
    geo = eng.decoder_geometry(BATCH)
    w_dec = 1399936 + 20560 * R                                       # SURVEY §8d
    bytes_step = w_dec * 4 + 2 * BATCH * T_IN * 256 * 4 + BATCH * (2 * 4 * 256 + 80 + 80 * R + T_IN) * 4
    alg_bytes = bytes_step * steps_taken
    achieved = alg_bytes / (stage["decoder_kernel"] / 1e3) / 1e9
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # DRAM traffic of that kernel per launch from the committed ncu capture (dram__bytes_read.sum + dram__bytes_write.sum)
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r2_decoder_traffic.json")
    if os.path.exists(tpath) and os.environ.get("TACO_DEC_IMPL", "cw") == "cw":
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"], tj["source"]
    kname = ("decoder_cw_kernel (cluster 16, <=%d utterances per cluster, %d clusters)" % (geo["samples_per_cluster"], geo["num_clusters"])
             if os.environ.get("TACO_DEC_IMPL", "cw") == "cw" else
             "decoder_kernel<S=%d,CS=%d>" % (geo["samples_per_cluster"], geo["cluster_size"]))
    roofline = {"bound": "hbm", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": stage["decoder_kernel"],
                "us_per_decoder_step": 1e3 * stage["decoder_kernel"] / steps_taken,
                "stage_ms": stage}

    # ---- end to end through the C-ABI host entry point (pinned host buffers) ----
    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype).pin_memory().numpy()
    for l in lanes:
        hi, hl, hs = l["host"]
        l["pin"] = dict(ids=pinned((BATCH, T_IN), torch.int32), lens=pinned((BATCH,), torch.int32),
                        spk=pinned((BATCH,), torch.int32), mel=pinned((BATCH, T_out, hp.num_mels), torch.float32),
                        lin=pinned((BATCH, T_out, hp.num_freq), torch.float32),
                        al=pinned((BATCH, T_IN, MAX_ITERS), torch.float32))
        l["pin"]["ids"][:], l["pin"]["lens"][:], l["pin"]["spk"][:] = hi, hl, hs

    # Lanes must not fall into lockstep (all computing, then all copying).  taco_forward_host_begin only enqueues; a lane
    # holds one of the compute slots until its decoder loop is done (its post-net then fills the SMs the next lane's
    # decoder leaves free) and gives it up before its 144 MB of D2H.  Measured on B200 (lanes, slots -> M frames/s):
    # round 1: (2,1) 6.2-7.2, (3,2) 6.4, (4,2) 8.3-8.4, (5,2) 8.3, (6,2) 8.8, (6,3) 8.7, (8,2) 8.5;
    # round 2 (faster GEMMs, CUDA-graph forward, >= 4 batches per lane timed): (5,2) 11.0, (6,2) 10.5, (6,3) 8.9, (8,3) 11.1, (8,2) 11.5;
    # at the end of round 2 (median of three regions): (6,2) 10.3, (8,2) 11.3, (10,2) 11.8, (12,2) 11.9, (10,3) 11.1 -> ten lanes.
    n_slots = int(os.environ.get("TACO_E2E_SLOTS", 2 if n_lanes >= 3 else 1))
    release_stage = int(os.environ.get("TACO_E2E_RELEASE", 0))   # 0: when the decoder loop is done, 1: all kernels
    compute_slots = threading.Semaphore(n_slots)

    def e2e_step(l):
        b = l["pin"]
        with compute_slots:
            l["eng"].forward_host_begin(b["ids"], b["lens"], b["spk"], None, False, _abi.BN_MOVING, b["mel"], b["lin"], b["al"])
            l["eng"].forward_host_wait(release_stage)
        return l["eng"].forward_host_end()

    def e2e_timed(active, n_steps):
        barrier()
        share = [n_steps // len(active) + (1 if i < n_steps % len(active) else 0) for i in range(len(active))]

        def work(l, k):
            with torch.cuda.stream(l["stream"]):
                for _ in range(k):
                    e2e_step(l)
        t0 = time.perf_counter()
        if len(active) == 1:
            work(active[0], share[0])
        else:
            ths = [threading.Thread(target=work, args=(l, k)) for l, k in zip(active, share) if k > 0]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dist is not None:
            tt = torch.tensor([dt], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        return dt / n_steps
    for l in lanes:
        with torch.cuda.stream(l["stream"]):
            e2e_step(l)
    # enough steps that filling and draining the pipeline (first forward before any copy, last copy after all kernels:
    # ~6 ms together) do not dominate the wall-clock average: every lane runs at least four batches
    k_e2e = max(4 * n_lanes, args.steps)
    e2e_timed(lanes, 2 * n_lanes)
    e2e_runs = [e2e_timed(lanes, k_e2e) for _ in range(3)]      # the host-side lane schedule makes single regions vary by ~10 %:
    e2e_s = sorted(e2e_runs)[1]                                 # three timed regions of k_e2e batches each, the median is reported
    e2e_single_s = e2e_timed(lanes[:1], max(2, k_e2e // 4))
    pb = lanes[0]["pin"]
    e2e = {"value": frames_per_step / e2e_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_s, "steps": k_e2e,
           "ms_per_step_runs": [1e3 * x for x in e2e_runs],
           "single_stream_ms_per_step": 1e3 * e2e_single_s,
           "h2d_bytes_per_step": int(pb["ids"].nbytes + pb["lens"].nbytes + pb["spk"].nbytes),
           "d2h_bytes_per_step": int(pb["mel"].nbytes + pb["lin"].nbytes + pb["al"].nbytes),
           "api": "taco_forward_host_begin/_wait/_end (C ABI, pinned host buffers; H2D + forward + D2H per step; %d lanes, "
                  "at most %d of them between _begin and the end of their decoder loop)" % (n_lanes, n_slots),
           "host_waits": "blocking" if os.environ.get("TACO_BLOCKING_SYNC", "0") not in ("", "0") else "spinning",
           "host_cores": os.cpu_count(), "numa_binding": numa}

    # what the link alone allows: one batch's outputs copied device -> pinned host with nothing else running
    lin_pin = torch.from_numpy(pb["lin"])
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lin_pin.copy_(lanes[0]["outs"][1], non_blocking=True)
    torch.cuda.synchronize()
    c0.record()
    for _ in range(4):
        lin_pin.copy_(lanes[0]["outs"][1], non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    d2h_gbs = 4 * pb["lin"].nbytes / (c0.elapsed_time(c1) * 1e6)
    e2e["d2h_link_gbs"] = d2h_gbs
    e2e["d2h_floor_ms_per_step"] = e2e["d2h_bytes_per_step"] / (d2h_gbs * 1e6)

    # ---- the same two legs in the decoder's throughput geometry (informational) ----
    # taco_set_decoder_clusters(4): 4 clusters of 8 utterances (64 SMs for 2.9 ms) instead of 7 clusters of 5/4 (112 SMs
    # for 2.2 ms).  The headline legs above and the roofline use the default (latency) geometry.
    thr = None
    thr_clusters = int(os.environ.get("TACO_BENCH_CLUSTERS", "4"))
    if not args.no_throughput_mode:
        for l in lanes:
            l["eng"].set_decoder_clusters(thr_clusters)
        timed(dev_lanes, 2 * n_dev)
        ms_t, st_t = timed(dev_lanes, max(n_dev, args.steps // 2))
        ms_t /= max(n_dev, args.steps // 2)
        e2e_timed(lanes, 2 * n_lanes)
        e2e_t = e2e_timed(lanes, k_e2e)
        thr = {"decoder_geometry": "%d clusters x 16 CTAs, <= %d utterances each" % (thr_clusters, -(-BATCH // thr_clusters)),
               "value": frames_per_step / (ms_t / 1e3), "ms_per_step": ms_t, "unit": UNIT,
               "e2e": {"value": frames_per_step / e2e_t, "ms_per_step": 1e3 * e2e_t, "unit": UNIT}}
        for l in lanes:
            l["eng"].set_decoder_clusters(0)

    # ---- the plain-bf16 mode (informational; NOT the headline: the reference computes in fp32) ----
    # taco_set_gemm_mode(2): one bf16 product per k-step in the dense layers and the decoder's mat-vecs instead of the fp32-class
    # three; stated tolerance 1e-2 on the decoder outputs / 5e-2 on the whole path (tests/test_gpu_parity.py), measured 4.4e-3 on
    # mel and 1.4e-3 on linear against the default mode at this size.
    bf16 = None
    if not args.no_throughput_mode:
        for l in lanes:
            l["eng"].set_gemm_mode(2)
        timed(dev_lanes, 2 * n_dev)
        ms_b, _ = timed(dev_lanes, max(n_dev, args.steps // 2))
        ms_b /= max(n_dev, args.steps // 2)
        ms_b1, _ = timed(lanes[:1], 4)
        bf16 = {"what": "taco_set_gemm_mode(2): plain bf16 operands, fp32 accumulation (dense layers and decoder mat-vecs); BiGRU in fp32",
                "value": frames_per_step / (ms_b / 1e3), "ms_per_step": ms_b, "single_stream_ms_per_step": ms_b1 / 4, "unit": UNIT,
                "tolerance": "1e-2 decoder outputs, 5e-2 whole path (max-abs, stated in tests/test_gpu_parity.py)"}
        for l in lanes:
            l["eng"].set_gemm_mode(1)

    # ---- the second half of BASELINE.json's metric: p50 batch-1 utterance latency (config 5 shapes, r=5, 200 steps) ----
    lat = None
    if not args.no_latency and world == 1:
        import statistics
        lat = {"what": "one utterance, device resident, one stream; CUDA events around taco_forward (gather -> linear "
                       "output, step count read back), p50 over 30 runs per input length", "unit": "ms", "p50": {}}
        lat_stream = lanes[0]["stream"]          # a non-default stream: taco_forward replays its CUDA graph there
        lat_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(lat_stream):
            out1 = (torch.zeros(1, T_out, hp.num_mels, device=dev), torch.zeros(1, T_out, hp.num_freq, device=dev), None)
            for t_in in (20, 60, 100, 200):
                rng1 = np.random.default_rng(500 + t_in)
                ids1 = torch.from_numpy(rng1.integers(7108, 7325, (1, t_in)).astype(np.int32)).to(dev)
                len1 = torch.tensor([t_in], dtype=torch.int32, device=dev)
                spk1 = torch.tensor([3], dtype=torch.int32, device=dev)
                al1 = torch.zeros(1, t_in, MAX_ITERS, device=dev)
                ts = []
                for i in range(33):
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record()
                    eng.forward(ids1, len1, spk1, out=(out1[0], out1[1], al1))
                    a1.record()
                    a1.synchronize()
                    if i >= 3:
                        ts.append(a0.elapsed_time(a1))
                lat["p50"]["T_in=%d" % t_in] = statistics.median(ts)
            # the same utterance down to the waveform (reference Synthesizer.synthesize: + Griffin-Lim, 100 iterations)
            ts = []
            wav1 = None
            for i in range(13):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                _, lin1, _, _ = eng.forward(ids1, len1, spk1, out=(out1[0], out1[1], al1))
                if wav1 is None:
                    wav1 = eng.griffin_lim(lin1)
                else:
                    eng.griffin_lim(lin1, out=wav1)
                a1.record()
                a1.synchronize()
                if i >= 3:
                    ts.append(a0.elapsed_time(a1))
        lat["p50_with_griffin_lim_T_in=200"] = statistics.median(ts)
        torch.cuda.current_stream().wait_stream(lat_stream)

    # ---- the step after the path (informational): Griffin-Lim vocoder on the last linear output of lane 0 ----
    voc = None
    if not args.no_vocoder and world == 1:
        lin = lanes[0]["outs"][1]
        voc_stream = lanes[0]["stream"]
        voc_stream.wait_stream(torch.cuda.current_stream())
        torch.cuda.set_stream(voc_stream)                      # non-default stream + a fixed output buffer: graph replay
        wav = eng.griffin_lim(lin)                             # warm-up (workspace growth)
        torch.cuda.synchronize()
        voc_l0 = eng.launch_count()
        voc_sampler = ClockSampler(local)
        t_dead = time.time() + 3.0
        while voc_sampler.proc is not None and not voc_sampler.lines and time.time() < t_dead:
            time.sleep(0.02)
        eng.griffin_lim(lin, out=wav)                          # second warm-up (captures the graph)
        eng.griffin_lim(lin, out=wav)
        vt0 = time.time()
        v_calls = []
        for _ in range(5):
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            v0.record()
            eng.griffin_lim(lin, out=wav)
            v1.record()
            v1.synchronize()
            v_calls.append(v0.elapsed_time(v1))
        vt1 = time.time()
        torch.cuda.synchronize()
        torch.cuda.set_stream(torch.cuda.default_stream(dev))
        voc_clocks = voc_sampler.stop(vt0, vt1)
        v_ms = float(np.median(v_calls))                       # per-call device times; the median is reported
        voc = {"what": "taco_griffin_lim: %d iterations + inverse pre-emphasis on the batch's linear spectrograms "
                       "(reference synthesizer.py:27,50); not part of `value`" % hp.griffin_lim_iters,
               "ms_per_batch": v_ms, "us_per_iteration": 1e3 * v_ms / hp.griffin_lim_iters,
               "frames_per_s": frames_per_step / (v_ms / 1e3), "launches_per_batch": (eng.launch_count() - voc_l0) // 7, "ms_per_call": v_calls,
               "audio_seconds_per_batch": BATCH * wav.shape[-1] / hp.sample_rate, "clocks": voc_clocks}

    # ---- the other configurations BASELINE.json names (extra keys; bench_configs.py) ----
    extra = {}
    if not args.no_configs:
        import bench_configs
        from tacotron_multispeaker_b200 import sharding
        extra = bench_configs.run(torch, Engine, HParams, random_init, _abi, sharding, dev, local, rank, world, dist, barrier,
                                  eng, hp, ID_NUM, args.steps, quick=args.quick_configs)

    # ---- CPU restatement on the host cores (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        dt, frames, _ = cpu_restatement_seconds(cores)
        cpu = {"value": frames / dt, "unit": UNIT, "cores": cores, "kind": "port", "seconds": dt,
               "sample": "one full batch (32 utterances x 1000 frames), torch-CPU fp32 restatement of the reference "
                         "TF graph (TensorFlow 1.x cannot be installed here)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(world), inflight="%d batches in flight per GPU (one handle + CUDA stream "
                                                            "each); single_stream = one at a time" % n_dev),
            "single_stream": single, "e2e": e2e, "throughput_mode": thr, "bf16_mode": bf16, "latency_batch1": lat, "vocoder": voc, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "decoder_geometry": geo,
        }
        line.update(extra)
        emit(line)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    for l in lanes:
        l["eng"].close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU restatement leg")
    ap.add_argument("--inflight", type=int, default=4, help="batches in flight per GPU (handles/streams), device-resident leg")
    ap.add_argument("--e2e-lanes", type=int, default=10, help="batches in flight per GPU in the end-to-end leg")
    ap.add_argument("--no-latency", action="store_true", help="skip the batch-1 latency leg")
    ap.add_argument("--no-vocoder", action="store_true", help="skip the informational Griffin-Lim leg")
    ap.add_argument("--no-throughput-mode", action="store_true", help="skip the informational 4-cluster decoder legs")
    ap.add_argument("--no-configs", action="store_true", help="skip the legs for BASELINE configs 1, 2, 4, 5 and the synthesize-shaped e2e")
    ap.add_argument("--quick-configs", action="store_true", help="fewer runs in those legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last step returned (rank 0, first batch) as DIR/<name>.npy")
    args = ap.parse_args()
    # stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner on stdout when
    # NCCL_DEBUG is set): file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved one.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
