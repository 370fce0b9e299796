#!/usr/bin/env python
"""bench.py -- encrypted images/s on CryptoNets-MNIST (N=8192), the headline metric of BASELINE.json.

A step = one pass of the reference's timed region ("Batch-Time": after EncryptLayer, before Decrypt,
`CryptoNets/CryptoNets.cs:31,74`) over one 8192-image batch of synthetic MNIST-shaped inputs:
conv 5x5/2 (845 outputs) -> square -> dense 845->100 -> square -> dense 100->10, P plaintext moduli (default 2, the
reference's configuration, `CryptoNets.cs:17`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--plain-moduli 1|2] [--dump-outputs DIR]
                                                                                B200 arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                                          CPU arm: the in-repo C++ oracle (the
        reference's C#/SEAL path cannot be built here) on all host cores, each step a bounded sample of the same workload.

Prints ONE JSON line (rank 0).  `value` is the whole-job aggregate with inputs resident in HBM; `e2e` goes through the
public API with host (pinned) ciphertext buffers; `roofline` is the NTT kernel family measured live with CUDA events on
the library's stream."""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 8192
WORKLOAD = "CryptoNets-MNIST N=8192 k=5: conv5x5s2(845) > square > dense845x100 > square > dense100x10, 8192 images/batch"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    """Threads the CPU arm may use: the scheduler affinity of this process (what `Defaults.ThreadCount = ProcessorCount` amounts to inside a
    container), not the machine's logical CPU count."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def host_info():
    info = {"affinity_cpus": host_threads(), "logical_cpus": os.cpu_count()}
    try:
        with open("/proc/cpuinfo") as f:
            models = [l.split(":", 1)[1].strip() for l in f if l.startswith("model name")]
        info["cpu_model"] = models[0] if models else None
    except Exception:
        pass
    try:
        info["numa_nodes"] = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
    except Exception:
        pass
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    return info


class CpuWorkload:
    """The CryptoNets-MNIST batch on the CPU oracle (`oracle/`, the C++ restatement of the SEAL 3.2 path; the C#/SEAL reference cannot be
    built here).  Inputs are uniform residues drawn from the same seed family as the GPU arm's images (ciphertext words are computationally
    uniform; the arithmetic does not depend on their values); weights are the shipped ones.  Thread model: the oracle's parallel_for pulls
    output indices dynamically, as `HE Wrapper/Utils.cs:46-88` does."""

    LAYERS = ("conv1", "square2", "dense3", "square4", "dense5")

    def __init__(self, primes, seed=20240917):
        from oracle.oracle_py import Oracle
        from cryptonets_b200.layers import ConvolutionEngine
        from cryptonets_b200.networks import cryptonets_weights, transpose
        w = cryptonets_weights()
        ce = ConvolutionEngine()
        ce.InputShape, ce.KernelShape, ce.Stride, ce.Upperpadding, ce.MapCount = [28, 28], [5, 5], [2, 2], [1, 1], [5, 1]
        ce.Prepare()
        self.ch = []
        for ci, t in enumerate(primes):
            o = Oracle(t, 8192, -1, 10, 20)
            o.keygen(1)
            rng = np.random.default_rng(seed + ci)
            q = np.array(o.q, dtype=np.uint64)

            def rand_cts(n, rng=rng, q=q, o=o):
                a = rng.integers(0, 1 << 43, (n, 2, o.k, 8192), dtype=np.uint64)
                return (a % q[None, None, :, None]).reshape(n, o.ct_words)

            def lift(x, t=t):
                x = np.rint(x)
                return np.where(x < 0, x + t, x).astype(np.uint64)

            d = dict(o=o, x=rand_cts(784), a1=rand_cts(845), a2=rand_cts(100))
            d["gather"] = np.array([[ce.Location(c, off, ce.InputShape) for off in ce.Offsets] for c in ce.Corners] * 5, dtype=np.int32)
            w0 = np.array([[w["Weights_0"][m * 26 + ce.Location(None, off, ce.KernelShape)] for off in ce.Offsets] for m in range(5)]) * 32
            d["wconv"] = lift(np.repeat(w0, 169, axis=0))
            d["bconv"] = lift(np.repeat(np.array([w["Weights_0"][(m + 1) * 26 - 1] for m in range(5)]) * 512, 169))
            d["w1"] = lift(transpose(w["Weights_1"], 845, 100).reshape(100, 845) * 1024)
            d["b1"] = lift(np.rint(w["Biases_2"] * 1000.0) % t)
            d["w3"] = lift(w["Weights_3"].reshape(10, 100) * 32)
            d["b3"] = lift(np.rint(w["Biases_3"] * 1000.0) % t)
            # output buffers allocated (and their pages touched) once: the timed passes measure arithmetic, not the kernel's page faults
            for name, n in (("o_conv", 845), ("o_sq1", 845), ("o_d3", 100), ("o_sq2", 100), ("o_d5", 10)):
                d[name] = np.ones(n * o.ct_words, np.uint64)
            self.ch.append(d)

    def step(self, threads, strides=(1, 1, 1, 1, 1)):
        """One pass over the batch; strides[i] > 1 computes every strides[i]-th output of layer i and scales its time.  Returns the
        per-layer seconds (already scaled), summed over the plaintext moduli."""
        sec = dict.fromkeys(self.LAYERS, 0.0)
        for d in self.ch:
            o = d["o"]
            calls = (("conv1", lambda st: o.mac_layer(d["x"], d["gather"], d["wconv"], d["bconv"], 845, 25, threads=threads, m_begin=0, m_step=st, out=d["o_conv"])),
                     ("square2", lambda st: o.square_layer(d["a1"], threads=threads, begin=0, step=st, out=d["o_sq1"])),
                     ("dense3", lambda st: o.mac_layer(d["a1"], None, d["w1"], d["b1"], 100, 845, threads=threads, m_begin=0, m_step=st, out=d["o_d3"])),
                     ("square4", lambda st: o.square_layer(d["a2"], threads=threads, begin=0, step=st, out=d["o_sq2"])),
                     ("dense5", lambda st: o.mac_layer(d["a2"], None, d["w3"], d["b3"], 10, 100, threads=threads, m_begin=0, m_step=st, out=d["o_d5"])))
            for (name, fn), st in zip(calls, strides):
                t0 = time.perf_counter()
                fn(st)
                sec[name] += (time.perf_counter() - t0) * st
        return sec

    @staticmethod
    def sample_strides(threads):
        """Strides whose sampled item counts stay whole multiples of the thread count (no partial last wave that the scaling would
        multiply): conv 845 and square 845 outputs, dense 100, square 100, dense 10."""
        def stride(n):
            waves_full = -(-n // threads)
            if waves_full <= 2:
                return 1
            keep = 2 * threads  # two full waves
            return max(1, n // keep)
        return (stride(845), stride(845), stride(100), stride(100), 1)


def cpu_measure(primes, threads, steps, warmup, budget_s=150.0, single_thread=True):
    """Times `steps` passes after `warmup` untimed ones.  Every pass is the FULL batch (all 845/845/100/100/10 outputs of every layer)
    when the run fits the time budget; otherwise the two big layers are sampled in whole thread-waves and the first timed pass is still a
    full one, so the line reports how far the sampled estimate is from the full measurement."""
    wl = CpuWorkload(primes)
    t0 = time.perf_counter()
    first = wl.step(threads)  # warm-up pass 1: full batch, also the size probe
    first_s = time.perf_counter() - t0
    full_total = sum(first.values())
    use_full = full_total * (steps + warmup) <= budget_s
    strides = (1, 1, 1, 1, 1) if use_full else CpuWorkload.sample_strides(threads)
    for _ in range(max(0, warmup - 1)):
        wl.step(threads, strides)
    per_layer = dict.fromkeys(CpuWorkload.LAYERS, 0.0)
    totals = []
    for _ in range(steps):
        sec = wl.step(threads, strides)
        totals.append(sum(sec.values()))
        for k_, v in sec.items():
            per_layer[k_] += v / steps
    mean_s = float(np.mean(totals))
    info = {"mode": "full batch every step" if use_full else "sampled: strides %s per layer (conv1, square2, dense3, square4, dense5), whole thread-waves, times scaled by the stride" % (strides,),
            "seconds_per_batch": mean_s, "per_layer_seconds": per_layer, "full_batch_probe_seconds": full_total, "probe_wall_seconds": first_s,
            "sampled_vs_full": None if use_full else mean_s / full_total, "step_seconds_min_max": [float(np.min(totals)), float(np.max(totals))]}
    if single_thread:  # one thread on a slice: 2 square outputs, 2 dense3 outputs, 8 conv outputs per modulus, scaled to the batch
        st = (845 // 8, 845 // 2, 100 // 2, 100 // 2, 10 // 2)
        sec1 = wl.step(1, st)
        info["single_thread_seconds_per_batch"] = sum(sec1.values())
        info["single_thread_images_per_s"] = BATCH / sum(sec1.values())
        info["single_thread_sample"] = "1 thread, every %d/%d/%d/%d/%d-th output of the five layers, scaled" % st
    return mean_s, info


def cpu_line_config(plain_moduli, world):
    return {"workload": WORKLOAD, "plain_moduli": plain_moduli, "parallelism": "replica-per-gpu x%d" % world,
            "l2": "inputs larger than L2 (784 ct x 640 KiB per modulus)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if args.workload != "cryptonets":
        return run_reference_lola(args)
    from cryptonets_b200.networks import CRYPTONETS_PRIMES
    primes = CRYPTONETS_PRIMES[: args.plain_moduli]
    threads = host_threads()
    sec, info = cpu_measure(primes, threads, args.steps, args.warmup, budget_s=float(os.environ.get("CNHE_CPU_BUDGET_S", "200")))
    value = BATCH / sec
    print(json.dumps({
        "impl": "reference", "metric": "encrypted images/sec (CryptoNets-MNIST, N=8192)", "value": value, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic (uniform residues from the GPU arm's seed family; shipped CryptoNets weights)",
        "config": cpu_line_config(len(primes), world),
        "notes": "in-repo C++ oracle of the SEAL 3.2 path on the host cores; the C#/SEAL reference cannot be built here",
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": info["mode"], "detail": info, "host": host_info()},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))



def quiesce_python_gc():
    """The cyclic collector's generation-2 pass walks the whole heap that torch, numpy and the network leave behind: 30-35 ms on the GPU
    box, about once every nine CryptoNets batches -- longer than a batch of device time, so the GPU ran dry behind it
    (profiles/r02_e2e_gc.txt).  Everything allocated during set-up is parked in the permanent generation; what the steps allocate is
    still collected (young generations), a full pass now has almost nothing to walk."""
    gc.collect()
    gc.freeze()
    return "gc.freeze() after set-up"


# --------------------------------------------------------------------------------------------------------- B200 arm
def build_network(factory):
    """The CryptoNets-MNIST layer chain without its reader/encrypt layers (those sit before the timer)."""
    from cryptonets_b200.layers import PoolLayer, SquareActivation
    from cryptonets_b200.networks import cryptonets_weights, transpose

    class Src:
        Factory = factory

        def GetOutputScale(self):
            return 16.0

        def PrepareNetwork(self):
            pass

    w = cryptonets_weights()
    conv1 = PoolLayer(Source=Src(), InputShape=[28, 28], KernelShape=[5, 5], Upperpadding=[1, 1], Stride=[2, 2], MapCount=[5, 1], WeightsScale=32,
                      Weights=w["Weights_0"])
    act2 = SquareActivation(Source=conv1)
    dense3 = PoolLayer(Source=act2, InputShape=[845], KernelShape=[845], Stride=[1000], MapCount=[100], Weights=transpose(w["Weights_1"], 845, 100),
                       Bias=w["Biases_2"], WeightsScale=1024)
    act4 = SquareActivation(Source=dense3)
    dense5 = PoolLayer(Source=act4, InputShape=[100], KernelShape=[100], Stride=[1000], MapCount=[10], Weights=w["Weights_3"], Bias=w["Biases_3"],
                       WeightsScale=32)
    layers = [conv1, act2, dense3, act4, dense5]
    dense5.PrepareNetwork()
    return layers


def forward(layers, m):
    for layer in layers:
        nxt = layer.Apply(m)
        if layer is not layers[0]:
            m.Dispose()
        m = nxt
    return m


def dump_outputs(path, eng, scores):
    """Writes what one step returned, so that two builds can be compared output for output on the same seeded inputs:
    score_ciphertexts.npy, every residue word of the 10 score ciphertexts, shape (10, plaintext moduli, 2, coefficient moduli, N), and
    scores.npy, their decryption, shape (images, 10).  Both float64, which holds residues below 2^53 exactly."""
    words = np.stack([[v.vec.export_raw(ch, 0) for ch in range(eng.P)] for v in scores.vectors]).reshape(len(scores.vectors), eng.P, 2, eng.k, eng.N)
    if int(words.max()) >= 1 << 53:
        raise ValueError("ciphertext words need more than 53 bits: float64 would round them")
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "score_ciphertexts.npy"), words.astype(np.float64))
    np.save(os.path.join(path, "scores.npy"), np.asarray(scores.Decrypt(), dtype=np.float64))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from cryptonets_b200.he import B200BfvFactory, B200BfvMatrix, B200BfvVector
    from cryptonets_b200.interfaces import EMatrixFormat
    from cryptonets_b200.networks import CRYPTONETS_PRIMES, synthetic_mnist

    from cryptonets_b200 import parallel
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # host threads and (first-touch) pinned staging buffers next to the GPU they feed: the 8-GPU e2e number moves 1 GB per step per rank
    numa = parallel.bind_to_gpu_numa(local) if os.environ.get("CNHE_NUMA_BIND", "1") != "0" else {"bound": False}
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    primes = CRYPTONETS_PRIMES[: args.plain_moduli]
    f = B200BfvFactory(primes, BATCH, seed=1 + rank, device=local)
    eng = f.engine
    layers = build_network(f)
    # every rank owns one batch (replicas over batches: the only split the slot packing allows, SURVEY 8e)
    imgs = synthetic_mnist(BATCH, seed=20240917 + rank)
    x_raw = np.rint(imgs / 256.0 * 16.0)
    xm = f.GetEncryptedMatrix(x_raw, EMatrixFormat.ColumnMajor, 1)
    xm.RegisterScale(16.0)
    eng.sync()

    def barrier():
        eng.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the device-resident number is taken on ONE stream so that the per-kernel CUDA-event times are not inflated by kernels of the
    # other plaintext-modulus channel running concurrently; warm up in the same mode (the block recycler is per stream)
    eng.set_option("multi_stream", 0)
    # the one exchange of the path: every batch's score ciphertexts (10 ct x P) are all-gathered over NVLink, on the device, inside the
    # timed region (cryptonets_b200/parallel.py); with one rank it degenerates to the packing copy
    gatherer = parallel.ScoreGatherer(eng, 10, torch.device("cuda", local))

    def step_resident():
        out_ = forward(layers, xm)
        gatherer.gather([v.vec for v in out_.vectors])
        return out_

    host_gc = quiesce_python_gc()
    for _ in range(args.warmup):
        step_resident().Dispose()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:  # one nvidia-smi loop per job, on the rank that reports
        sampler.start()
    launches0 = eng.launch_count()
    eng.prof_enable(True)
    eng.timer_start()
    last = None
    for _ in range(args.steps):
        if last is not None:
            last.Dispose()
        last = step_resident()
    ms = eng.timer_stop_ms()
    gatherer.finish()
    barrier()
    prof = eng.prof_collect()
    eng.prof_enable(False)
    launches = eng.launch_count() - launches0
    clocks = sampler.stop()
    if world > 1:
        tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    value = BATCH * args.steps * world / (ms * 1e-3)

    # informational: the same K steps with one CUDA stream per plaintext-modulus channel (the two channels' kernels overlap each other's
    # tails; per-launch event times are then inflated by the concurrency, which is why the roofline above is taken on one stream)
    eng.set_option("multi_stream", 1)
    for _ in range(2):
        step_resident().Dispose()
    barrier()
    eng.timer_start()
    for _ in range(args.steps):
        step_resident().Dispose()
    ms2 = eng.timer_stop_ms()
    barrier()
    if world > 1:
        t2 = torch.tensor([ms2], dtype=torch.float64, device="cuda")
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms2 = float(t2.item())
    value_two_streams = BATCH * args.steps * world / (ms2 * 1e-3)

    # ---- e2e: host (pinned) ciphertexts in, score ciphertexts out, through the public API
    host_in = torch.empty(eng.P * 784 * eng.ct_words, dtype=torch.int64).pin_memory()
    host_out = torch.empty(eng.P * 10 * eng.ct_words, dtype=torch.int64).pin_memory()
    raw = eng.export_raw_many([v.vec for v in xm.vectors], host_in.data_ptr())
    del raw

    def e2e_import():
        vecs = eng.import_raw_many(host_in.data_ptr(), 784, 1, BATCH, 16.0)  # asynchronous: runs on the library's upload stream
        return B200BfvMatrix(f, [B200BfvVector(f, v) for v in vecs], EMatrixFormat.ColumnMajor, CopyVectors=False)

    depth = max(1, int(os.environ.get("CNHE_E2E_DEPTH", "1")))  # batches queued ahead of the one whose scores the host waits for (2 measured slower: the
    # upload of batch i+1 then has to wait for a slot of batch i-2 and no longer hides under batch i-1: tools/e2e_timeline.py, DEPTH=1|2)
    host_outs = [host_out] + [torch.empty_like(host_out).pin_memory() for _ in range(depth)]

    def e2e_run(steps):
        """`steps` batches: host ciphertexts in, score ciphertexts back on the host, pipelined the way a serving loop is: batch i+1 is
        uploaded and queued while batch i computes, and the host waits for the scores of batch i-depth.  Every batch's scores are on the
        host before the timed region ends."""
        nxt = e2e_import()
        pending = []
        for s_ in range(steps):
            cur = nxt
            out = forward(layers, cur)
            cur.Dispose()
            gatherer.gather([v.vec for v in out.vectors])  # NVLink all-gather of this batch's scores, queued behind its kernels
            ticket = eng.export_raw_many_async([v.vec for v in out.vectors], host_outs[s_ % (depth + 1)].data_ptr())
            out.Dispose()  # stream-ordered: released after the copies above
            if s_ + 1 < steps:
                nxt = e2e_import()
            pending.append(ticket)
            if len(pending) > depth:
                eng.export_wait(pending.pop(0))
        for ticket in pending:
            eng.export_wait(ticket)
        gatherer.finish()

    eng.set_option("multi_stream", int(os.environ.get("CNHE_E2E_MULTI_STREAM", "1")))
    e2e_run(max(8, args.warmup))  # reaches the steady state of the upload slots and of the block recycler at pipeline depth 2
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())
    e2e_value = BATCH * args.steps * world / e2e_s

    out = None
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        fam = prof["ntt_forward"]
        # dominant family: forward NTT (incl. the digit-decomposing variant of relinearisation)
        achieved = fam["bytes"] / (fam["ms"] * 1e-3) / 1e9 if fam["ms"] > 0 else 0.0
        # the forward transform is limited by FP64 issue (8 DP instructions per butterfly: 100 % of the pipe = 0.85 of this HBM figure), not by
        # HBM itself; it is reported against the measured HBM copy bandwidth because that is the roofline SURVEY.md 8d prescribes
        roof = {"bound": "hbm", "limited_by": "fp64-issue (ncu: 63 % of the FP64 pipe busy, math_pipe_throttle the top stall; 100 % of the pipe would be 0.85 of this HBM figure)", "kernel": "k_ntt_forward_fp / k_ntt_forward_digits_fp (N=8192), 16*N algorithmic bytes per transform", "achieved": achieved,
                "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "peak_source": peak_kind + " copy bandwidth (MEASURED_PEAKS.json)",
                # ncu (profiles/r02_top_kernels_ncu.txt, same figures as round 1's capture): one k_ntt_forward_digits_fp launch of 16000 transforms moved 42.4 MB + 994.7 MB of
                # DRAM traffic against 2097.2 MB algorithmic (16N per transform; the digit source is shared by 125 transforms through
                # L2) -- ratio 0.495, applied to this run's mean launch (waves are larger than the captured one)
                "traffic": 0.495 * fam["bytes"] / max(1, fam["launches"]),
                "traffic_source": "ncu dram bytes / algorithmic bytes = 0.495 for k_ntt_forward_digits_fp<13,1> (profiles/r02_top_kernels_ncu.txt), scaled to this run's mean launch",
                "launches_timed": fam["launches"], "algorithmic_bytes_per_launch": fam["bytes"] / max(1, fam["launches"]),
                "avg_launch_ms": fam["ms"] / max(1, fam["launches"]), "share_of_step": fam["ms"] / ms if ms else None,
                "families_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items()}}
        if numa.get("previous_cpus"):  # the CPU leg uses every core the job may use, not just the GPU's NUMA node
            os.sched_setaffinity(0, numa["previous_cpus"])
        cpu_threads = host_threads()
        # bounded CPU leg beside the GPU number: one warm-up pass (full batch) + two timed passes, sampled if the host is slow
        cpu_sec, cpu_info = cpu_measure(primes, cpu_threads, steps=2, warmup=1, budget_s=25.0, single_thread=False)
        out = {
            "metric": "encrypted images/sec (CryptoNets-MNIST, N=8192)", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic MNIST-shaped uint8 images (80% zeros), shipped CryptoNets weights, device-generated keys",
            "config": cpu_line_config(len(primes), world),
            "clocks": clocks, "gpu_launches": int(launches), "numa": {k_: v for k_, v in numa.items() if k_ != "previous_cpus"}, "host_gc": host_gc,
            "collective": {"op": "all_gather_into_tensor (NCCL) of the score ciphertexts, every step, inside both timed regions",
                           "bytes_per_rank_per_step": int(eng.P * 10 * eng.ct_words * 8)},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": int(host_in.numel() * 8), "d2h_bytes_per_step": int(host_out.numel() * 8)},
            "value_two_streams": {"value": value_two_streams, "unit": "images/s", "ms_per_step": ms2 / args.steps,
                                  "note": "same steps, one CUDA stream per plaintext modulus; not used for the roofline"},
            "roofline": roof,
            "cpu_baseline": {"value": BATCH / cpu_sec, "unit": "images/s", "cores": cpu_threads, "kind": "port", "sample": cpu_info["mode"],
                             "detail": cpu_info, "host": host_info()},
            "readme_anchor_images_per_s": 320.0,
        }
        if args.dump_outputs:  # the last step of the timed loop above, its scores still held in `last`
            dump_outputs(args.dump_outputs, eng, last)
    last.Dispose()
    xm.Dispose()
    f.Dispose()
    if world > 1:
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out))


# --------------------------------------------------------------------------------------------------------- LoLa workloads (configs 3, 4)
def lola_workloads():
    from cryptonets_b200 import networks as nets
    return {
        # name: (builder, plaintext primes, N, decomposition bit count, the reference's SmallModulusCount, image maker, description)
        "lola_small": (nets.lola_small, nets.LOLA_SMALL_PRIMES, 8192, 40, 3, nets.synthetic_mnist,
                       "LoLa-small MNIST N=8192 k=3 w=40 (LoLaCryptonets.cs:280-329): LLPoolLayer conv > vectorize > square > LLDenseLayer 845x10, 1 image/inference"),
        "lola_cifar": (nets.lola_cifar, nets.CIFAR_PRIMES, 16384, 60, 8, nets.synthetic_cifar,
                       "LoLa-CIFAR N=16384 k=8 w=60 (LolaCifarCryptoNet.cs:27-131): conv 83 maps > vectorize > square > dense 5488x16268 (rotate-and-sum) > square > dense 5488x10, 1 image/inference, shipped weights"),
    }


def _layer_chain(net):
    out, p = [], net
    while p is not None and hasattr(p, "Source"):
        out.append(p)
        p = p.Source
    return out[::-1]


def run_lola(args):
    import torch
    import torch.distributed as dist
    from cryptonets_b200.he import B200BfvFactory, B200BfvMatrix, B200BfvVector
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    builder, primes, N, dbc, k, imgs_of, desc = lola_workloads()[args.workload]
    # --shard-rows (lola_cifar): ALL ranks work on the same image -- same keys, same input ciphertexts (the seeded sampler makes them
    # identical without any exchange) -- and split the 5488 rows of the big dense layer (strong scaling of one inference's latency);
    # default: every rank owns its own image (replicas over images, weak scaling, SURVEY 8e)
    shard = args.shard_rows and world > 1 and args.workload == "lola_cifar"
    f = B200BfvFactory(primes, N, DecompositionBitCount=dbc, GaloisDecompositionBitCount=dbc, SmallModulusCount=k, seed=1 if shard else 1 + rank,
                       device=local)
    eng = f.engine
    if shard:
        net, reader = builder(f, imgs_of(1, seed=20240917), shard=(rank, world, None))
    else:
        net, reader = builder(f, imgs_of(1, seed=20240917 + rank))
    net.PrepareNetwork()
    chain = _layer_chain(net)
    enc_layer, rest = chain[1], chain[2:]
    plain_in = chain[0].GetNext()
    xm = enc_layer.Apply(plain_in)  # the client's ciphertexts: before the reference's timer (TimingLayer after EncryptLayer)
    eng.sync()

    def forward(m):
        first = m
        for layer in rest:
            nxt = layer.Apply(m)
            if m is not first:
                m.Dispose()
            m = nxt
        return m

    def barrier():
        eng.sync()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng.set_option("multi_stream", 0)
    quiesce_python_gc()
    for _ in range(args.warmup):
        forward(xm).Dispose()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.op_counts(reset=True)
    launches0 = eng.launch_count()
    eng.prof_enable(True)
    eng.timer_start()
    for _ in range(args.steps):
        forward(xm).Dispose()
    ms = eng.timer_stop_ms()
    barrier()
    prof = eng.prof_collect()
    eng.prof_enable(False)
    counts = {k_: v // args.steps for k_, v in eng.op_counts(reset=True).items()}
    launches = eng.launch_count() - launches0
    clocks = sampler.stop()
    if world > 1:
        tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    images_per_step = 1 if shard else world
    value = args.steps * images_per_step / (ms * 1e-3)

    # ---- e2e: the image's ciphertexts come from pinned host memory every step, the score ciphertexts go back to the host
    vecs = xm.vectors
    n_in, blocks = len(vecs), vecs[0].vec.blocks
    host_in = torch.empty(eng.P * n_in * blocks * eng.ct_words, dtype=torch.int64).pin_memory()
    eng.export_raw_many([v.vec for v in vecs], host_in.data_ptr())
    dim0, scale0, fmt0 = vecs[0].vec.dim, vecs[0].vec.scale, vecs[0].vec.format
    probe = forward(xm)
    out_words = eng.P * sum(v.vec.blocks for v in probe.vectors) * eng.ct_words
    probe.Dispose()
    host_out = torch.empty(out_words, dtype=torch.int64).pin_memory()

    def e2e_step():
        imported = eng.import_raw_many(host_in.data_ptr(), n_in, blocks, dim0, scale0, fmt0)
        m = B200BfvMatrix(f, [B200BfvVector(f, v) for v in imported], xm.Format, CopyVectors=False)
        out = forward(m)
        m.Dispose()
        ticket = eng.export_raw_many_async([v.vec for v in out.vectors], host_out.data_ptr())
        out.Dispose()
        eng.export_wait(ticket)

    eng.set_option("multi_stream", 1)
    for _ in range(max(2, args.warmup)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())
    out = None
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        fam = prof["ntt_forward"]
        achieved = fam["bytes"] / (fam["ms"] * 1e-3) / 1e9 if fam["ms"] > 0 else 0.0
        cpu = lola_cpu_estimate(args.workload, counts)
        out = {
            "metric": "encrypted images/sec (%s, one image per inference)" % args.workload, "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "latency_ms": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic image (uniform uint8 pixels), shipped weights, device-generated keys",
            "config": {"workload": desc, "plain_moduli": len(primes),
                       "parallelism": ("rows of the 5488-row dense layer sharded x%d (one image)" % world) if shard else "replica-per-gpu x%d" % world,
                       "l2": "key-switching keys (%d Galois elements) and digit waves larger than L2" % eng.n_galois},
            "clocks": clocks, "gpu_launches": int(launches), "operations_per_inference": counts,
            "e2e": {"value": args.steps * images_per_step / e2e_s, "unit": "images/s", "h2d_bytes_per_step": int(host_in.numel() * 8),
                    "d2h_bytes_per_step": int(host_out.numel() * 8)},
            "roofline": {"bound": "hbm", "limited_by": "fp64-issue (ncu: 63 % of the FP64 pipe busy, math_pipe_throttle the top stall; 100 % of the pipe would be 0.85 of this HBM figure)", "kernel": "forward NTT family (digit transforms of the Galois / relinearisation key switch), 16*N algorithmic bytes per transform",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         "peak_source": peak_kind + " copy bandwidth (MEASURED_PEAKS.json)", "traffic": None, "launches_timed": fam["launches"],
                         "share_of_step": fam["ms"] / ms if ms else None, "families_ms_per_step": {k_: v["ms"] / args.steps for k_, v in prof.items()}},
            "cpu_baseline": cpu,
        }
    xm.Dispose()
    f.Dispose()
    if world > 1:
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out))


def lola_cpu_estimate(workload, counts, threads=None):
    """CPU leg for a LoLa inference: the CPU oracle (test infrastructure; timed here, never used for results) runs each evaluator operation
    the network issues -- rotation hop, dense multiply_plain, multiply + relinearise -- on one thread, and the per-inference operation
    counts of the GPU run (the reference's OperationsCount) scale them.  Dividing by the host's thread count assumes the reference's
    ParallelProcessInEnv scales perfectly over the rows of every layer: an upper bound on what the CPU can do."""
    from oracle.oracle_py import Oracle
    _, primes, N, dbc, k, _, _ = lola_workloads()[workload]
    threads = threads or host_threads()
    t = primes[0]
    o = Oracle(t, N, k, dbc, dbc)
    o.keygen(1)
    rng = np.random.default_rng(0)
    q = np.array(o.q, dtype=np.uint64)
    ct = (rng.integers(0, 1 << 62, (2, o.k, N), dtype=np.uint64) % q[None, :, None]).reshape(-1)
    plain = rng.integers(0, t, N, dtype=np.uint64)

    def best(fn, reps=3):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts)

    per_op = {
        "Rotation": best(lambda: o.rotate_rows(ct, 1)),
        "ColumnRotation": best(lambda: o.rotate_columns(ct)),
        "PlainMultiplication": best(lambda: o.multiply_plain(ct, plain)),
        "Multiplication": best(lambda: o.relinearize(o.multiply(ct, ct))),  # Multiply + Relinearize (counted once: Relinarization follows every Multiplication)
        "Addition": best(lambda: o.add(ct, ct)),
        "ScalarMultiplication": best(lambda: o.mac_layer(ct, None, np.array([3], dtype=np.uint64), None, 1, 1, threads=1)),
    }
    per_op["Subtraction"] = per_op["AddManyItemCount"] = per_op["PlainAddition"] = per_op["Addition"]
    one_thread = len(primes) * sum(per_op.get(name, 0.0) * n for name, n in counts.items())
    sec = one_thread / threads
    return {"value": 1.0 / sec, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": "one-thread oracle time of each evaluator operation x the per-inference operation counts, divided by %d threads (ideal scaling: upper bound for the CPU)" % threads,
            "single_thread_seconds_per_image": one_thread, "per_op_seconds": per_op, "host": host_info()}


def run_reference_lola(args):
    """CPU arm of a LoLa workload: needs the per-inference operation counts, which come from a recorded GPU run (profiles/; the B200 arm
    reports them as "operations_per_inference")."""
    path = os.path.join(ROOT, "profiles", "r02_opcounts_%s.json" % args.workload)
    counts = json.load(open(path))
    threads = host_threads()
    cpu = lola_cpu_estimate(args.workload, counts, threads)
    desc = lola_workloads()[args.workload][6]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    print(json.dumps({
        "impl": "reference", "metric": "encrypted images/sec (%s, one image per inference)" % args.workload, "value": cpu["value"], "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / cpu["value"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": {"workload": desc, "plain_moduli": len(lola_workloads()[args.workload][1]),
                                                                            "parallelism": "replica-per-gpu x%d" % world},
        "cpu_baseline": cpu, "e2e": {"value": cpu["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_microbench(args):
    """BASELINE config 5: NTT and multiply+relinearise micro-benchmark, GPU (libcnhe) next to the CPU oracle (this leg is a
    cpu_baseline: the oracle is timed, never used for results) on the box's host cores.  N in {4096, 8192, 16384}, k = 2..6
    coefficient moduli (prefixes of SEAL's default tables).  One JSON line per case."""
    from cryptonets_b200.engine import Engine
    from oracle.oracle_py import Oracle
    PEAK = 6580.3
    try:
        PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    threads = host_threads()
    cases = [(4096, 2), (4096, 3), (8192, 2), (8192, 4), (8192, 5), (16384, 4), (16384, 6)]
    t = {4096: 40961, 8192: 65537, 16384: 65537}
    rng = np.random.default_rng(0)
    for N, k in cases:
        eng = Engine([t[N]], N, 10, 20, k)
        eng.keygen(1)
        eng.set_option("multi_stream", 0)
        q = np.array(eng.q, dtype=np.uint64)
        n_polys = (1 << 27) // N // k * k  # 1 GiB of residue polynomials
        d = eng.dev_from(rng.integers(0, 1 << 35, n_polys * N, dtype=np.uint64))
        res = {"N": N, "k": k}
        for inverse in (False, True):
            for _ in range(2):
                eng.raw_ntt(d, d, n_polys, 0, k, inverse)
            eng.timer_start()
            for _ in range(5):
                eng.raw_ntt(d, d, n_polys, 0, k, inverse)
            ms = eng.timer_stop_ms() / 5
            res["gpu_%s_Mpolys_s" % ("intt" if inverse else "ntt")] = round(n_polys / ms / 1e3, 2)
            res["gpu_%s_frac_hbm" % ("intt" if inverse else "ntt")] = round(16.0 * N * n_polys / (ms * 1e-3) / 1e9 / PEAK, 3)
        eng.dev_free(d)
        # multiply + relinearise of n ciphertexts
        n = 256 if N <= 8192 else 128
        cts = (rng.integers(0, 1 << 62, (n, 2, k, N), dtype=np.uint64) % q[None, None, :, None]).astype(np.uint64)
        a = eng.dev_from(cts)
        out = eng.dev_alloc(n * 2 * k * N)
        for _ in range(2):
            eng.raw_multiply_relin(0, a, a, n, out)
        eng.timer_start()
        for _ in range(3):
            eng.raw_multiply_relin(0, a, a, n, out)
        res["gpu_square_relin_us_per_ct"] = round(eng.timer_stop_ms() / 3 * 1e3 / n, 2)
        eng.close()
        # CPU oracle, all host threads
        orc = Oracle(t[N], N, k, 10, 20)
        orc.keygen(1)
        cpu_polys = threads * 64 // k * k
        host = rng.integers(0, 1 << 35, cpu_polys * N, dtype=np.uint64)
        hp = host.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
        orc.L.orc_ntt_batch(orc.h, 0, hp, cpu_polys, 0, threads)  # in place; first call warms the pages and the thread pool
        t0 = time.perf_counter()
        for _ in range(3):
            orc.L.orc_ntt_batch(orc.h, 0, hp, cpu_polys, 0, threads)
        res["cpu_ntt_Mpolys_s"] = round(3 * cpu_polys / (time.perf_counter() - t0) / 1e6, 3)
        m = min(n, 2 * threads)
        t0 = time.perf_counter()
        orc.square_layer(cts[:m].reshape(m, -1), threads=threads)
        res["cpu_square_relin_us_per_ct"] = round((time.perf_counter() - t0) * 1e6 / m, 1)
        res["cpu_threads"] = threads
        res["speedup_ntt"] = round(res["gpu_ntt_Mpolys_s"] / res["cpu_ntt_Mpolys_s"], 1)
        res["speedup_square_relin"] = round(res["cpu_square_relin_us_per_ct"] / res["gpu_square_relin_us_per_ct"], 1)
        print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--plain-moduli", type=int, default=2, choices=[1, 2])
    ap.add_argument("--workload", default="cryptonets", choices=["cryptonets", "lola_small", "lola_cifar", "microbench"],
                    help="cryptonets = BASELINE config 2 (the headline metric); lola_small / lola_cifar = configs 3 / 4 (one image per inference); "
                         "microbench = config 5 (one JSON line per case)")
    ap.add_argument("--microbench", action="store_true", help="same as --workload microbench")
    ap.add_argument("--shard-rows", action="store_true", help="lola_cifar on several GPUs: one image, the big dense layer's rows split over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="cryptonets on the B200: after the timed steps, write the score ciphertexts of the "
                                                          "last timed step and their decryption to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "cryptonets" or args.microbench):
        ap.error("--dump-outputs covers the cryptonets workload on the B200")
    if args.microbench or args.workload == "microbench":
        run_microbench(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.workload != "cryptonets":
        run_lola(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
