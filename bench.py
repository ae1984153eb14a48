#!/usr/bin/env python
"""bench.py -- frames/sec of x-vector extraction (80-d fbank, 200-frame chunks, batches of 256) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1).  A STEP is one pass of the hot path over one rank's shard of
BASELINE.json configs[3]: 125 000 utterances (1 M over 8 GPUs) x 200 frames x 80-d, resident in HBM, through
`xvb_extractor_extract_shard` in configs[1] batches (256 x 200) -- split -> tdnn1..5 (statistics pooling fused
into tdnn5's epilogue) -> Chan merge -> tdnn6.affine, batches alternating between two lanes -- and, for N > 1, the
one exchange of the path: every GPU ends the step holding the whole (N x 125 000, 512) embedding table.  By default
the table's copies are mapped into one another over NVLink (CUDA IPC) and every batch's embeddings are stored into
all of them while the next batches run (csrc/peer.cu), a one-word all-reduce being the step's rendezvous; with
XVB_BENCH_GATHER=nccl (or if the mapping is refused) it is one NCCL all-gather after the shard.  After the warm-up the
shard sizes follow each rank's measured speed (whole batches, total unchanged; XVB_BENCH_BALANCE=0: equal shards).
A step lasts ~0.36 s, K steps several seconds: the timed region runs at SUSTAINED clocks; the `burst` block repeats
round 1's measurement (one batch timed alone).

  value        whole-job frames/s, inputs resident in HBM (CUDA events on the launching stream, barrier +
               synchronize both sides, max over ranks); weak scaling: per-GPU work is fixed
  e2e          the same shard through the C-ABI host-buffer call `xvb_extractor_extract_shard_host`: pinned host
               features -> H2D (copy stream, four device slots: the copies run ahead of both lanes) -> stack -> D2H of
               the embeddings, host clock
  roofline     the tcgen05 TDNN GEMM: algorithmic FLOPs (SURVEY 8d: 5 630 976 FLOP/frame) / summed per-launch
               CUDA-event durations taken inside a sustained pass, against MEASURED_PEAKS' sustained bf16 peak;
               `burst` carries the isolated-batch figures against the burst peak.  The kernel executes 3 bf16
               MMAs per algorithmic MAC (bf16x3 split), reported as executed_*.
  config4      BASELINE configs[3] back end on the gathered table: submean + length-norm, all-pairs cosine through
               the fused GEMM->histogram kernel (rows sharded over ranks, counters all-reduced), EER; per-phase ms
  config3_ecapa / config5   ECAPA-TDNN c1024 (128 x 300 batches) over a 125 000-utterance shard per GPU, and
               PLDA scoring of those enrolment embeddings against 10 000 test embeddings (fused histogram, EER)
  cpu_baseline the oracle port of the reference's CPU PyTorch path on this box's host cores (N = 1 only)

`--impl reference` times that CPU port alone (the reference is Python/torch and cannot travel to the GPU box; the
oracle restates it op for op, pinned by tests/golden) on a bounded sample of the same workload per step.
XVB_BENCH_UTTS / XVB_BENCH_ECAPA_UTTS shrink the shards for smoke runs (the JSON line states the sizes used).

--dump-outputs DIR writes what the timed path returned in its last step, after the timed region, as float32 .npy files:
DIR/embeddings.npy holds the embedding table (native: the gathered (N x shard, 512) table; reference: the step's batch),
cut to a fixed seeded sample of DUMP_ROWS rows when longer.  The inputs are seeded, so two builds run with the same
arguments can be compared output for output; for that, N > 1 keeps equal shards (no balancing by measured speed).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, T, F, D = 256, 200, 80, 512
SHARD_UTTS = int(os.environ.get("XVB_BENCH_UTTS", "125000"))       # BASELINE configs[3]: 1 M utterances / 8 GPUs
FLOP_PER_FRAME = 5630976          # SURVEY.md 8(d): 2*(2 807 808 MAC/frame) + 2*1 536 000/200
GEMM_FLOP_PER_BATCH = FLOP_PER_FRAME * B * T
GEMM_LAUNCHES_PER_BATCH = 6
POOL_BYTES_PER_BATCH = 1212000 * B  # SURVEY.md 8(d): 4*(C*T + 2C) B/utt, C=1500, T=200
EB, ET, ED = 128, 300, 192          # BASELINE configs[2]: ECAPA-TDNN c1024, batch 128 x 300 frames
ECAPA_SHARD_UTTS = int(os.environ.get("XVB_BENCH_ECAPA_UTTS", "125000"))   # configs[4]: 1 M enrolment utterances / 8
ECAPA_TEST_UTTS = 10000
ECAPA_FLOP_PER_FRAME = 25701908   # SURVEY.md 8(d) at T = 300
SPK_OFFSET = 0.1                  # synthetic speakers: x = N(0,1) + 0.1 * m[spk]  (EER of a few % on random weights)
UTTS_PER_SPK = 100
METRIC = "frames/sec x-vector extraction (80-d fbank)"
UNIT = "frames/s"
CPU_THREADS = 32                  # fixed thread count of the host arm (more threads than this slows ATen's small convs)
DUMP_ROWS = 16384                 # --dump-outputs: at most this many embedding rows (32 MB of float32)


def workload_config(world):
    return {"workload": "x-vector TDNN (pytorch/model/xvector.py), 80-d fbank, 200-frame chunks, batches of 256 "
                        "(BASELINE configs[1]) over a %d-utterance shard per GPU (configs[3]: 1 M utterances on 8 GPUs), "
                        "extracted_embedding=far" % SHARD_UTTS,
            "batch": B, "frames_per_utt": T, "feat_dim": F, "utts_per_gpu_per_step": SHARD_UTTS,
            "l2_policy": "inputs larger than L2: %.1f GB of features per step per GPU, ~1.1 GB of activations per batch"
                         % (SHARD_UTTS * T * F * 4 / 1e9),
            "weights": "seeded synthetic checkpoint of the reference architecture"}


def dump_outputs(dirname, **arrays):
    """Each (rows, ...) tensor as DIR/<name>.npy in float32; longer than DUMP_ROWS rows: a fixed seeded sample of rows."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if a.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))
            a = a[torch.from_numpy(rows).to(a.device)]
        np.save(os.path.join(dirname, name + ".npy"), a.detach().float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"],
                "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clock/throttle sampling during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window(self, t0, t1):
        sm, smax, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                mhz, smax_i = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            smax = smax_i
            if t0 <= ts <= t1:
                sm.append(mhz)
                try:
                    power.append(float(parts[6]))
                except ValueError:
                    pass
                for n, v in zip(names, parts[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_mhz_min": min(sm) if sm else None,
                "sm_max_mhz": smax, "power_w_max": max(power) if power else None, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()


def pin_to_gpu_numa_node(local_rank):
    """Run this process on the CPUs of its GPU's NUMA node, so that pinned host buffers (first touch) and the
    threads that drive the copies sit next to the GPU's PCIe root (VERDICT r1 #5: e2e swung 62.8 <-> 72.9 M
    frames/s with the placement).  Best effort; reports what it did."""
    info = {"node": None, "cpus": None, "pinned": False}
    try:
        sel = str(local_rank)
        try:
            u = str(torch.cuda.get_device_properties(local_rank).uuid)
            sel = u if u.startswith("GPU-") else "GPU-" + u
        except Exception:
            pass
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", sel],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0].strip()
        dom, rest = out.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:].lower(), rest.lower())
        node = int(open(path).read().strip())
        info["node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info["cpus"], info["pinned"] = len(cpus), True
    except Exception as err:  # noqa: BLE001  (sysfs / nvidia-smi layout differences: run unpinned, say so)
        info["error"] = repr(err)[:120]
    return info


def make_checkpoint():
    from oracle import nnet as onn  # synthetic seeded weights of the BASELINE architecture (no datasets here)
    return onn.make_state_dict(onn.xvector_spec(F), 102)


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_port_step(sd, x):
    from oracle import nnet as onn
    return onn.xvector_forward(sd, x, "far")


def cpu_port_setup():
    from oracle import nnet as onn
    sd = make_checkpoint()
    x = torch.from_numpy(onn.synthetic_feats(B, T, F, 1024)).transpose(1, 2).contiguous()   # one full configs[1] batch
    threads = max(1, min(CPU_THREADS, os.cpu_count() or 1, len(os.sched_getaffinity(0))))
    torch.set_num_threads(threads)
    return sd, x, threads


def cpu_baseline(budget_s):
    """The oracle port on a bounded sample: whole 256 x 200 batches (batched forward: the form most favourable to
    the reference) for about `budget_s` seconds, plus the reference's literal one-utterance-per-call loop."""
    from oracle import nnet as onn
    sd, x, threads = cpu_port_setup()
    with torch.no_grad():
        cpu_port_step(sd, x[:32])
        n, t0 = 0, time.perf_counter()
        while n < 2 or time.perf_counter() - t0 < budget_s * 0.7:
            cpu_port_step(sd, x)
            n += 1
        batched = n * B * T / (time.perf_counter() - t0)
        feats = x.transpose(1, 2).contiguous().numpy()
        m, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < budget_s * 0.3:
            onn.extract_embedding(lambda z: onn.xvector_forward(sd, z, "far"), feats[m % B])
            m += 1
        per_utt = m * T / (time.perf_counter() - t0)
    return {"value": batched, "unit": UNIT, "cores": threads, "host_cpus": os.cpu_count() or 1, "kind": "port",
            "sample": "%d whole 256 x 200 batches, batched forward of the oracle port (torch CPU ops incl. the masked "
                      "taps), %d threads; the reference's literal batch-1 extract_embedding loop on the same "
                      "utterances: %.0f frames/s" % (n, threads, per_utt),
            "per_utterance_value": per_utt}


def run_reference(args, rank, world):
    if rank != 0:
        return
    sd, x, threads = cpu_port_setup()
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 3))):
            cpu_port_step(sd, x)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = cpu_port_step(sd, x)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, embeddings=out.squeeze(2))
    value = args.steps * B * T / dt
    sample = ("each step = one whole 256 x 200 batch of the step's %d (a bounded sample of the same workload), batched "
              "forward of the oracle port, %d host threads" % ((SHARD_UTTS + B - 1) // B, threads))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "host_cpus": os.cpu_count() or 1, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ synthetic shards
def synthetic_shard(n, t, f, first_global, n_spk, dev, seed):
    """(n, t, f) fp32 on the device: N(0,1) frames + SPK_OFFSET * m[spk] (one 80-d offset per synthetic speaker, the
    same table on every rank), speaker of global utterance g = g % n_spk.  Returns (feats, spk int32)."""
    gm = torch.Generator(device=dev)
    gm.manual_seed(1024)                       # the reference's own seed (runXvector.py:176): speaker table
    m = torch.randn(n_spk, f, device=dev, generator=gm)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    spk = ((torch.arange(n, device=dev, dtype=torch.int64) + first_global) % n_spk)
    x = torch.empty(n, t, f, device=dev, dtype=torch.float32)
    step = 8192
    for i in range(0, n, step):
        j = min(n, i + step)
        x[i:j].normal_(generator=g)
        x[i:j] += SPK_OFFSET * m[spk[i:j]][:, None, :]
    return x, spk.to(torch.int32)


def pinned_copy(x):
    h = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
    h.copy_(x)
    torch.cuda.synchronize()
    return h


def balance_shards(speed, n_total, batch, cap):
    """Shard sizes proportional to `speed` (one entry per rank) in whole batches by largest remainder, the odd tail of
    n_total to the fastest rank; None if that would exceed `cap` utterances on a rank or leave one without a batch."""
    speed = np.asarray(speed, dtype=np.float64)
    q, rem = divmod(int(n_total), int(batch))
    share = q * speed / speed.sum()
    batches = [int(x) for x in np.floor(share)]
    for r in np.argsort(-(share - np.floor(share)), kind="stable")[: q - sum(batches)]:
        batches[int(r)] += 1
    n_rank = [b * batch for b in batches]
    n_rank[int(np.argmax(speed))] += rem
    if sum(n_rank) != n_total or max(n_rank) > cap or min(n_rank) < batch:
        return None
    return n_rank


class Timer:
    def __init__(self, world, dev):
        self.world, self.dev = world, dev

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([v], device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)

    def wall(self, fn):
        """fn() bracketed by barrier + synchronize; host-clock milliseconds, max over ranks."""
        self.barrier()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        self.barrier()
        return r, self.max_over_ranks(ms)


# ------------------------------------------------------------------------------------------ C1 latency
def c1_latency(dev):
    """BASELINE configs[0] on the GPU path: one (200, 23) MFCC utterance through the plugin call
    `model.extract_embedding(ndarray) -> CPU tensor`, and the same utterance through the oracle port on the host."""
    from asv_subtools_b200.model.xvector import Xvector
    from oracle import nnet as onn
    sd = onn.make_state_dict(onn.xvector_spec(23), 101)
    m = Xvector(23, 10, training=False, extracted_embedding="far")
    m.load_state_dict(sd, strict=True)
    m.to(dev).eval()
    feats = onn.synthetic_feats(1, 200, 23, 5)[0]
    for _ in range(10):
        m.extract_embedding(feats)
    ts = []
    for _ in range(200):
        t0 = time.perf_counter()
        m.extract_embedding(feats)
        ts.append(time.perf_counter() - t0)
    gpu_ms = statistics.median(ts) * 1e3
    torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
    cs = []
    for _ in range(20):
        t0 = time.perf_counter()
        onn.extract_embedding(lambda z: onn.xvector_forward(sd, z, "far"), feats)
        cs.append(time.perf_counter() - t0)
    return {"workload": "Xvector(23) one 200-frame utterance, extract_embedding(ndarray)->CPU tensor (BASELINE configs[0])",
            "gpu_ms_per_utt": gpu_ms, "cpu_port_ms_per_utt": statistics.median(cs) * 1e3, "cpu_threads": 8}


# ------------------------------------------------------------------------------------------ x-vector blocks
XV_KERNELS = ["split_frames", "tdnn1", "tdnn2", "tdnn3", "tdnn4", "tdnn5+pool_partials", "pool_finalize", "tdnn6.affine(split-K+reduce)"]


def profile_sustained(ex, feats, emb, n_batches):
    """Per-kernel CUDA-event times inside a back-to-back pass (events on the launching stream, recorded by the
    library around every kernel of every batch): means over the full batches of the pass."""
    n = min(feats.shape[0], n_batches * B)
    n -= n % B
    ex.set_profiling(True)
    ex.extract_shard(feats[:n], B, out=emb[:n])
    per_batch = len(XV_KERNELS) + 1                       # + the gap to the next batch's first event
    t = np.array(ex.kernel_times_ms(max_n=(n // B) * per_batch + 8))
    ex.set_profiling(False)
    nb = (t.shape[0] + 1) // per_batch
    t = np.concatenate([t, [0.0]])[: nb * per_batch].reshape(nb, per_batch)
    t = t[2:] if nb > 4 else t                            # the first batches still ramp
    return t[:, :len(XV_KERNELS)].mean(axis=0), float(t[:-1, -1].mean()) if t.shape[0] > 1 else 0.0


def burst_block(ex, feats, steps, pk):
    """Round 1's measurement: `steps` single 256 x 200 batches timed alone after idle (burst clocks), and the
    per-kernel times of such isolated batches."""
    xs = [feats[i * B:(i + 1) * B] for i in range(8)]
    for i in range(3):
        ex.extract(xs[i])
    torch.cuda.synchronize()
    time.sleep(0.5)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        ex.extract(xs[i % 8])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ex.set_profiling(True)
    per = []
    for i in range(10):
        ex.extract(xs[i % 8])
        per.append(ex.kernel_times_ms())
        time.sleep(0.02)
    ex.set_profiling(False)
    per = np.median(np.array(per), axis=0)
    gemm_ms = float(per[1:6].sum() + per[7])
    ach = GEMM_FLOP_PER_BATCH / (gemm_ms * 1e-3) / 1e12
    return {"what": "%d single 256 x 200 batches timed alone (%.1f ms region, burst clocks): round 1's measurement" % (steps, ms * steps),
            "value": B * T / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms, "gemm_ms_per_batch": gemm_ms,
            "kernel_ms": {n: float(v) for n, v in zip(XV_KERNELS, per)},
            "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["bf16_burst"], "unit": "TFLOP/s", "frac": ach / pk["bf16_burst"],
                         "executed_tflops": 3 * ach, "executed_frac": 3 * ach / pk["bf16_burst"],
                         "peak_source": pk["src"] + " bf16 burst (kernel timed in isolation)"}}


def stats_pool_block(dev, pk):
    """The standalone statistics-pooling kernel on the BASELINE tensor (the product path pools inside tdnn5's
    epilogue; the north star also asks for this kernel's HBM fraction)."""
    from asv_subtools_b200 import ops
    pool_in = [torch.randn(B, T, 1500, device=dev) for _ in range(3)]   # 3 x 307 MB >> L2
    for i in range(3):
        ops.stats_pool(pool_in[i % 3])
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(12):
        ops.stats_pool(pool_in[i % 3])
    p1.record()
    torch.cuda.synchronize()
    ms = p0.elapsed_time(p1) / 12
    gbs = POOL_BYTES_PER_BATCH / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "stats_pool_tma_kernel (standalone, (256,200,1500) fp32, 12 back-to-back launches over "
                                      "3 rotating inputs)", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": gbs / pk["hbm_gbs"], "traffic": None,
            "traffic_static": {"bytes_per_launch": 313000000, "source": "profiles/r01x_pool_ncu_summary.txt (builder-run ncu --set full)",
                               "algorithmic_bytes": POOL_BYTES_PER_BATCH},
            "ms": ms, "peak_source": pk["src"]}


# ------------------------------------------------------------------------------------------ back end (configs 3/4)
def config4_block(tm, full, spk_full, rank, world, verify_single):
    """BASELINE configs[3] back end on the gathered (n, 512) table: global-mean subtraction + length normalisation
    (score/process.sh submean + norm), all-pairs cosine (score/score.sh cosine) through the fused GEMM -> trial
    histogram kernel with the rows sharded over ranks by 256-row unit and one all-reduce of the counters per
    pass, EER (binary_metrics.py) by zooming.  Per-phase milliseconds, max over ranks."""
    from asv_subtools_b200 import ops
    from asv_subtools_b200.score import trial_histogram as th
    n = full.shape[0]
    x, prep_ms = tm.wall(lambda: ops.center_length_norm(full, ops.column_mean(full)))
    try:                                                      # warm the histogram kernel on a corner of the table
        th.zoom_eer(x[:4096].contiguous(), spk_full[:4096].contiguous(), passes=1, group=False)
    except ValueError:
        pass
    pilot = 32 if n >= 1 << 16 else 0

    def eer_job(**kw):
        try:
            return th.zoom_eer(x, spk_full, passes=3, pilot=pilot, **kw)
        except ValueError:       # the pilot's bracket missed the crossing of the full set: locate it with a full pass
            return th.zoom_eer(x, spk_full, passes=4, pilot=0, **kw)
    res, eer_ms = tm.wall(lambda: eer_job(rank=rank, world=world))
    lo, hi = res["lo"], res["hi"]

    def one_pass():
        h = ops.trial_histogram(x, spk_full, x, spk_full, lo, hi, 2048, symmetric=True, unit_first=rank, unit_stride=world)
        return th._reduce(h, None)
    _, pass_ms = tm.wall(one_pass)
    trials = n * (n - 1) // 2
    out = {"what": "all pairs of the gathered %d x 512 table, each once (j > i): %.3e trials" % (n, trials),
           "prep_ms": prep_ms, "eer_ms": eer_ms, "eer_passes": res["passes"], "pilot_stride": pilot,
           "narrow_pass_ms": pass_ms, "trials": trials, "trials_per_s": trials / (pass_ms * 1e-3),
           "algorithmic_tflops": 2 * D * trials / (pass_ms * 1e-3) / 1e12, "executed_tflops": 3 * 2 * D * trials / (pass_ms * 1e-3) / 1e12,
           "eer": res["eer"], "threshold": res["threshold"], "counted": int(res["hist"].sum()),
           "count_ok": int(res["hist"].sum()) == trials}
    if verify_single and world > 1:
        # the same job on ONE GPU (rank 0 sweeps every row unit, no all-reduce): the sharded EER must equal it
        one = None
        if rank == 0:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            one = eer_job(group=False)
            torch.cuda.synchronize()
            out["single_gpu_eer_ms"] = (time.perf_counter() - t0) * 1e3
            out["single_gpu_eer"] = one["eer"]
            out["eer_equals_single_gpu"] = bool(one["eer"] == res["eer"])
        tm.barrier()
    return out


def ecapa_blocks(tm, dev, rank, world, pk, steps_hint):
    """BASELINE configs[2] and [4]: ECAPA-TDNN c1024 over this rank's shard of enrolment utterances (128 x 300
    batches), then two-covariance PLDA (score/pyplda/gaussian-plda-scoring.py) of every enrolment embedding against
    10 000 test embeddings through the fused histogram kernel.  Enrolment rows stay where they were extracted; only
    the 10 000 x 192 test table is all-gathered and the counters all-reduced (SURVEY 8e)."""
    import torch.distributed as dist
    from asv_subtools_b200.model.ecapa_tdnn_xvector import ECAPA_TDNN
    from asv_subtools_b200.score import trial_histogram as th
    from asv_subtools_b200.score.plda_train import PldaEstimation, PldaStats
    from oracle import nnet as onn
    canon = dict(training=False, extracted_embedding="near",
                 ecapa_params={"channels": 1024, "embd_dim": 192, "mfa_conv": 1536,
                               "bn_params": {"momentum": 0.5, "affine": True, "track_running_stats": True}},
                 fc2_params={"nonlinearity": "", "bn": True, "bn_params": {"momentum": 0.5, "affine": False,
                                                                            "track_running_stats": True}})
    m = ECAPA_TDNN(F, 10, **canon)
    m.load_state_dict(onn.make_state_dict(onn.ecapa_spec(F), 201), strict=True)
    m.to(dev).eval()
    ex = m.extractor()
    n = ECAPA_SHARD_UTTS
    n_total = n * world
    n_spk = max(2, n_total // UTTS_PER_SPK)
    feats, spk = synthetic_shard(n, ET, F, rank * n, n_spk, dev, 4096 + rank)
    emb = torch.empty(n, ED, device=dev)
    ex.extract_shard(feats[:4 * EB], EB, out=emb[:4 * EB])        # warm-up: plans, workspace
    tm.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ex.extract_shard(feats, EB, out=emb)
    e1.record()
    tm.barrier()
    ms = tm.max_over_ranks(e0.elapsed_time(e1))
    launches = ex.last_launches
    frames = n_total * ET
    # end to end through the host-buffer shard call on a bounded part of the shard (pinned host memory)
    n_e2e = min(n, 64 * EB)
    host = pinned_copy(feats[:n_e2e])
    host_out = torch.empty(n_e2e, ED, dtype=torch.float32, pin_memory=True)
    ex.extract_shard_host(host.data_ptr(), 4 * EB, ET, host_out.data_ptr(), EB)
    _, e2e_ms = tm.wall(lambda: ex.extract_shard_host(host.data_ptr(), n_e2e, ET, host_out.data_ptr(), EB))
    ok = bool(torch.isfinite(host_out).all()) and bool(torch.allclose(host_out, emb[:n_e2e].cpu(), atol=0, rtol=0))
    ach = ECAPA_FLOP_PER_FRAME * n * ET / (ms * 1e-3) / 1e12
    c3 = {"workload": "ECAPA-TDNN c1024 (SE-Res2Block + attentive stats pooling), 80-d fbank, 300-frame chunks, batches of 128 "
                      "(BASELINE configs[2]) over a %d-utterance shard per GPU, extracted_embedding=near" % n,
          "value": frames / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms / ((n + EB - 1) // EB), "shard_ms": ms,
          "gpu_launches": launches,
          "e2e": {"value": world * n_e2e * ET / (e2e_ms * 1e-3), "unit": UNIT, "utts": n_e2e, "h2d_bytes": n_e2e * ET * F * 4,
                  "d2h_bytes": n_e2e * ED * 4, "api": "xvb_ecapa_extract_shard_host", "equals_device_path": ok},
          "roofline": {"bound": "tensor", "kernel": "whole ECAPA step (tdnn_gemm_bf16x3_kernel launches + res2net_chain_kernel + "
                                                    "bandwidth kernels), algorithmic FLOPs of SURVEY 8d / shard time",
                       "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"],
                       "executed_tflops": 3 * ach, "executed_frac": 3 * ach / pk["bf16_sustained"],
                       "peak_source": pk["src"] + " bf16 sustained (%.1f s region)" % (ms * 1e-3), "traffic": None}}
    del feats, host
    # ---- configs[4]: test set = 10 000 utterances sharded over ranks, extracted, all-gathered (7.7 MB)
    nt_local = (ECAPA_TEST_UTTS + world - 1) // world
    tfeats, tspk_local = synthetic_shard(nt_local, ET, F, rank * nt_local, n_spk, dev, 8192 + rank)
    temb_local = ex.extract_shard(tfeats, EB)
    del tfeats
    if world > 1:
        temb = torch.empty(world * nt_local, ED, device=dev)
        tspk = torch.empty(world * nt_local, dtype=torch.int32, device=dev)
        _, gather_ms = tm.wall(lambda: (dist.all_gather_into_tensor(temb, temb_local), dist.all_gather_into_tensor(tspk, tspk_local)))
    else:
        temb, tspk, gather_ms = temb_local, tspk_local, 0.0
    temb, tspk = temb[:ECAPA_TEST_UTTS].contiguous(), tspk[:ECAPA_TEST_UTTS].contiguous()
    # PLDA model: rank 0 trains on its first enrolment embeddings (PldaEstimation, 10 EM iterations), everyone gets it
    ntrain = min(n, 20000)
    params = torch.zeros(ED + 2 * ED * ED, dtype=torch.float64, device=dev)
    train_ms = 0.0
    if rank == 0:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        est = PldaEstimation(PldaStats.from_matrix(emb[:ntrain], spk[:ntrain].cpu().numpy())).estimate(10)
        torch.cuda.synchronize()
        train_ms = (time.perf_counter() - t0) * 1e3
        params = torch.from_numpy(np.concatenate([est.mean.reshape(-1), est.within_var.reshape(-1), est.between_var.reshape(-1)])).to(dev)
    if world > 1:
        dist.broadcast(params, 0)
    from asv_subtools_b200.score.backend import PldaModel
    p = params.cpu().numpy()
    model = PldaModel(p[:ED], p[ED:ED + ED * ED].reshape(ED, ED), p[ED + ED * ED:].reshape(ED, ED))
    from asv_subtools_b200 import ops
    proj = ops.project(emb, model.l2_d)
    rt, ct = model.terms(emb), model.terms(temb)
    sample = ops.plda_matrix(emb[:2048].contiguous(), temb, model.l2_d, rt[:2048].contiguous(), ct)
    smin, smax = float(sample.min()), float(sample.max())
    if world > 1:
        mm = torch.tensor([-smin, smax], device=dev, dtype=torch.float64)
        dist.all_reduce(mm, op=dist.ReduceOp.MAX)
        smin, smax = -float(mm[0]), float(mm[1])
    span = smax - smin
    lo, hi = smin - 0.25 * span, smax + 0.25 * span
    del sample
    # every rank sweeps ITS OWN enrolment rows (rank=0, world=1 inside the call); the counters are all-reduced
    res, eer_ms = tm.wall(lambda: th.zoom_eer(proj, spk, temb, tspk, lo=lo, hi=hi, passes=3, row_term=rt, col_term=ct))
    wlo, whi = res["lo"], res["hi"]

    def one_pass():
        h = ops.trial_histogram(proj, spk, temb, tspk, wlo, whi, 2048, row_term=rt, col_term=ct)
        return th._reduce(h, None)
    _, pass_ms = tm.wall(one_pass)
    trials = n_total * ECAPA_TEST_UTTS
    c5 = {"what": "PLDA (two-covariance, gaussian-plda-scoring.py) of %d enrolment x %d test ECAPA embeddings (192-d): %.3e "
                  "trials, enrolment rows stay on the GPU that extracted them" % (n_total, ECAPA_TEST_UTTS, trials),
          "enroll_extract_ms": ms, "test_allgather_ms": gather_ms, "plda_train_ms_rank0": train_ms, "plda_train_utts": ntrain,
          "eer_ms": eer_ms, "eer_passes": res["passes"], "narrow_pass_ms": pass_ms, "trials": trials,
          "trials_per_s": trials / (pass_ms * 1e-3), "algorithmic_tflops": 2 * ED * trials / (pass_ms * 1e-3) / 1e12,
          "eer": res["eer"], "counted": int(res["hist"].sum()), "count_ok": int(res["hist"].sum()) == trials,
          "score_window_first_pass": [lo, hi]}
    return c3, c5


# ------------------------------------------------------------------------------------------ GPU arm
def run_native(args, rank, world, local_rank):
    import torch.distributed as dist
    numa = pin_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tm = Timer(world, dev)
    pk = peaks()

    from asv_subtools_b200.model.xvector import Xvector
    sd = make_checkpoint()
    model = Xvector(F, 10, training=False, extracted_embedding="far")
    model.load_state_dict(sd, strict=True)
    model.cuda().eval()
    ex = model.extractor()

    n = SHARD_UTTS
    n_total = n * world
    n_spk = max(2, n_total // UTTS_PER_SPK)
    # N > 1: room for a shard up to 8 % larger than nominal -- after the warm-up the shard sizes follow the measured speeds
    cap = n if world == 1 else n + ((n * 8 // 100 + B - 1) // B) * B
    feats_cap, spk_cap = synthetic_shard(cap, T, F, rank * cap, n_spk, dev, 2048 + rank)
    emb_cap = torch.empty(cap, D, device=dev)
    feats, spk, emb = feats_cap[:n], spk_cap[:n], emb_cap[:n]
    # The path's one exchange: every GPU needs the whole (N x n, 512) table.  Default: the table's copies are mapped
    # into one another over NVLink (CUDA IPC) and every batch's embeddings are stored into all of them while the next
    # batches run (csrc/peer.cu); a step then ends with a one-word all-reduce as the rendezvous.  XVB_BENCH_GATHER=nccl
    # (or a refused mapping): one NCCL all-gather after the shard.
    table, gather_kind = None, "none"
    if world > 1:
        gather_kind = "nccl"
        if os.environ.get("XVB_BENCH_GATHER", "p2p") != "nccl":
            try:
                from asv_subtools_b200.parallel import PeerTable
                table = PeerTable(n, D, total_rows=n_total)
                gather_kind = "p2p"
            except RuntimeError as err:
                if rank == 0:
                    print("bench.py: peer table unavailable (%s): NCCL all-gather" % err, file=sys.stderr)
    full = table.tensor if table is not None else (torch.empty(n_total, D, device=dev) if world > 1 else emb)
    spk_full = torch.empty(n_total, dtype=torch.int32, device=dev) if world > 1 else spk
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_gather_into_tensor(spk_full, spk)
    if table is not None:
        table.attach(ex)

    def exchange():
        if table is not None:
            dist.all_reduce(flag)                      # rendezvous: every rank's peer stores are complete
        elif world > 1:
            dist.all_gather_into_tensor(full, emb)     # (N x n, 512) fp32 over NVLink

    def step():
        ex.extract_shard(feats, B, out=emb)
        exchange()

    # ---- device-resident throughput (sustained) --------------------------------------------------
    warm_ms = []
    for _ in range(args.warmup):
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        ex.extract_shard(feats, B, out=emb)
        w1.record()
        exchange()
        warm_ms.append((w0, w1))
    # Shard sizes by measured speed (N > 1, peer table only: its rows need not be equal per rank).  Under the power cap the
    # GPUs of a box settle at different clocks (1447-1522 MHz in profiles/r04k) and a step ends when the slowest is done;
    # the reference balances its jobs the same way, by length (splitDataByLength.sh).  The total stays N x SHARD_UTTS.
    n_rank, row0, balance = [n] * world, rank * n, None
    if table is not None and os.environ.get("XVB_BENCH_BALANCE", "1") != "0" and not args.dump_outputs:
        torch.cuda.synchronize()
        mine = statistics.mean(a.elapsed_time(b) for a, b in warm_ms[-2:])
        times = torch.zeros(world, dtype=torch.float64, device=dev)
        times[rank] = mine
        dist.all_reduce(times)
        speed = 1.0 / times.cpu().numpy()
        if os.environ.get("XVB_BENCH_FAKE_SPEED"):                  # test knob: pretend the ranks differ (comma-separated factors)
            speed = speed * np.array([float(v) for v in os.environ["XVB_BENCH_FAKE_SPEED"].split(",")][:world])
        cut = balance_shards(speed, n_total, B, cap)
        if cut is not None:
            n_rank = cut
            row0 = sum(n_rank[:rank])
            n_mine = n_rank[rank]
            feats, spk, emb = feats_cap[:n_mine], spk_cap[:n_mine], emb_cap[:n_mine]
            table.attach(ex, row0)
            balance = {"kind": "static: shard sizes proportional to each rank's measured shard rate over the last two warm-up steps, "
                               "in whole batches, total unchanged", "utts_per_rank": n_rank,
                       "warmup_shard_ms_per_rank": [float(x) for x in times.cpu().numpy()]}
            step()                                                  # one more warm-up step at the new sizes
        else:
            n_rank = [n] * world
    n_mine = n_rank[rank]
    if world > 1:                                                   # speaker ids in table order (shards may be unequal now)
        pad = torch.full((world * cap,), -1, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(pad, spk_cap)
        spk_full = torch.cat([pad[r * cap:r * cap + n_rank[r]] for r in range(world)]).contiguous()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    tm.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    wall0 = time.time()
    ev[0].record()
    for i in range(args.steps):
        ex.extract_shard(feats, B, out=emb)
        ev[2 * i + 1].record()
        exchange()
        ev[2 * i + 2].record()
    tm.barrier()
    wall1 = time.time()
    ms = tm.max_over_ranks(ev[0].elapsed_time(ev[-1]))
    extract_ms = tm.max_over_ranks(statistics.median(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)))
    gather_ms = tm.max_over_ranks(statistics.median(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)))
    launches_per_step = ex.last_launches
    assert torch.isfinite(emb).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, embeddings=full)
    # the collective alone: inside a step its CUDA-event span also holds the wait for the slowest rank's shard
    gather_alone_ms, p2p_equals_nccl = 0.0, None
    if world > 1:
        check = torch.empty(world * cap, D, device=dev)
        tm.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            dist.all_gather_into_tensor(check[:n_total], emb_cap[:n])      # the nominal (N x n, 512) collective
        g1.record()
        tm.barrier()
        gather_alone_ms = tm.max_over_ranks(g0.elapsed_time(g1) / 5)
        if table is not None:              # the peer-stored table must be what NCCL gathers (padded shards), bit for bit
            dist.all_gather_into_tensor(check, emb_cap)
            ok = all(torch.equal(check[r * cap:r * cap + n_rank[r]], full[sum(n_rank[:r]):sum(n_rank[:r + 1])]) for r in range(world))
            same = torch.tensor([1 if ok else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            p2p_equals_nccl = bool(same.item())
        del check
    clocks_value = sampler.window(wall0, wall1) if sampler else None

    # ---- end to end through the host-buffer C-ABI shard call ----------------------------------------
    if table is not None:
        table.detach(ex)                                   # the end-to-end leg below measures the plain host-buffer call
    host = pinned_copy(feats)
    host_out = torch.empty(n_mine, D, dtype=torch.float32, pin_memory=True)
    ex.extract_shard_host(host.data_ptr(), min(n_mine, 8 * B), T, host_out.data_ptr(), B)      # warm: slots, copy stream
    e2e_steps = max(3, min(args.steps, 10))
    tm.barrier()
    wall2 = time.time()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ex.extract_shard_host(host.data_ptr(), n_mine, T, host_out.data_ptr(), B)   # returns with the embeddings on the host
    e2e_host_ms = (time.perf_counter() - t0) * 1e3
    tm.barrier()
    wall3 = time.time()
    e2e_ms = tm.max_over_ranks(e2e_host_ms)
    e2e_equal = bool(torch.equal(host_out, emb.cpu()))
    clocks_e2e = sampler.window(wall2, wall3) if sampler else None
    # what bounds e2e: the host->device link.  Same pinned buffer, copy alone, CUDA events.
    nb_link = min(n_mine, 64 * B)
    dst = torch.empty(nb_link, T, F, device=dev)
    dst.copy_(host[:nb_link], non_blocking=True)
    torch.cuda.synchronize()
    l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0.record()
    for _ in range(4):
        dst.copy_(host[:nb_link], non_blocking=True)
    l1.record()
    torch.cuda.synchronize()
    h2d_gbs = 4 * dst.numel() * 4 / (l0.elapsed_time(l1) * 1e-3) / 1e9
    del dst, host

    # ---- per-kernel CUDA-event times inside a sustained pass (roofline) -------------------------------
    for _ in range(2):
        ex.extract_shard(feats, B, out=emb)               # back under load before the profiled pass
    kern_ms, gap_ms = profile_sustained(ex, feats, emb, 200)
    gemm_ms = float(kern_ms[1:6].sum() + kern_ms[7])
    burst = burst_block(ex, feats, 20, pk) if rank == 0 or world == 1 else None
    pool = stats_pool_block(dev, pk) if rank == 0 else None
    if sampler:
        sampler.stop()

    # ---- BASELINE configs[3] back end on the gathered table ---------------------------------------------
    if world > 1 and table is None:
        dist.all_gather_into_tensor(full, emb)
    if table is not None:                                  # refill through the peer path (the e2e leg ran detached)
        table.attach(ex, row0)
        ex.extract_shard(feats, B, out=emb)
        table.detach(ex)
        table.barrier()
    c4 = config4_block(tm, full, spk_full, rank, world, verify_single=True)
    del feats, feats_cap
    torch.cuda.empty_cache()
    c3, c5 = ecapa_blocks(tm, dev, rank, world, pk, args.steps)
    if table is not None:
        tm.barrier()                                       # nobody unmaps while a peer may still read
        del full
        table.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    frames_per_step = n_total * T
    value = frames_per_step * args.steps / (ms * 1e-3)
    achieved = GEMM_FLOP_PER_BATCH / (gemm_ms * 1e-3) / 1e12
    gather_bytes = n_total * D * 4
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (bf16x3 split operands on tcgen05, fp32 accumulate in TMEM)", "data": "synthetic",
        "config": workload_config(world),
        "timed_region_s": ms * 1e-3,
        "balance": balance,
        "exchange": {"kind": gather_kind, "p2p_equals_nccl": p2p_equals_nccl,
                     "what": "p2p: every batch's embeddings are stored into all N table copies over NVLink peer mappings (CUDA IPC) "
                             "while the next batches run, a one-word all-reduce ends the step; nccl: one all-gather after the shard"},
        "phases_ms": {"extract_shard": extract_ms, "all_gather_in_step": gather_ms, "all_gather_alone": gather_alone_ms,
                      "all_gather_bytes_out": gather_bytes,
                      "all_gather_busbw_gbs": (gather_bytes * (world - 1) / world) / (gather_alone_ms * 1e-3) / 1e9 if world > 1 and gather_alone_ms > 0 else None,
                      "note": "medians over the timed steps, max over ranks; all_gather_in_step spans from the end of this rank's shard "
                              "to the end of the step's exchange (p2p: the rendezvous all-reduce; nccl: the all-gather), i.e. it includes "
                              "waiting for the slowest rank; all_gather_alone = the NCCL all-gather of the (N x %d, 512) fp32 table timed "
                              "by itself after a barrier (5 back to back), which is what the bus bandwidth is quoted on" % n},
        "shard_pipeline": "two lanes: batches alternate between twin workspaces on two streams (XVB_LANES=%s)" % os.environ.get("XVB_LANES", "1"),
        "e2e": {"value": frames_per_step * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / e2e_steps,
                "steps": e2e_steps, "h2d_bytes_per_step": n_mine * T * F * 4, "d2h_bytes_per_step": n_mine * D * 4,
                "api": "xvb_extractor_extract_shard_host (pinned host features in, host embeddings out; the H2D of batch k+1 "
                       "on a copy stream overlaps the kernels of batch k; host clock, max over ranks)",
                "equals_device_path": e2e_equal, "h2d_link_gbs_measured": h2d_gbs,
                "h2d_link_bound": world * h2d_gbs * 1e9 / (F * 4),
                "h2d_link_bound_note": "frames/s the host->device link alone allows at 320 B/frame per GPU", "numa": numa,
                "clocks": clocks_e2e},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks_value,
        "roofline": {"bound": "tensor",
                     "kernel": "tdnn_gemm_bf16x3_kernel (6 launches per 256 x 200 batch; tdnn5 pools over time in its epilogue, "
                               "tdnn6 is split-K + a reduce)",
                     "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                     "regime": "sustained: per-launch CUDA events inside a back-to-back pass of 200 batches",
                     "peak_source": pk["src"] + " bf16 sustained (kernel timed inside a seconds-long step)",
                     "algorithmic_flop_per_launch_avg": GEMM_FLOP_PER_BATCH / GEMM_LAUNCHES_PER_BATCH,
                     "launch_ms_avg": gemm_ms / GEMM_LAUNCHES_PER_BATCH, "gemm_ms_per_batch": gemm_ms,
                     "executed_tflops": 3 * achieved, "executed_frac": 3 * achieved / pk["bf16_sustained"],
                     "note": "3 bf16 MMAs per algorithmic MAC (hi*hi + lo*hi + hi*lo) to hold 1e-4 parity: the algorithmic "
                             "fraction is capped at 1/3 by construction",
                     "traffic": None,
                     "traffic_static": {"bytes_per_launch_avg": 122224000, "algorithmic_bytes_note": "42 MB per batch must move "
                                        "(features in, embeddings out, weights); the rest is the hi/lo activation planes between layers",
                                        "source": "profiles/r05_gemm_ncu_summary.txt: dram__bytes_read + dram__bytes_write summed "
                                        "over the six GEMM launches of one batch / 6 (builder-run ncu --set full; not measured by "
                                        "this run)"}},
        "kernel_ms": dict({k: float(v) for k, v in zip(XV_KERNELS, kern_ms)}, inter_batch_gap=gap_ms,
                          regime="sustained pass, mean per batch"),
        "burst": burst,
        "roofline_stats_pool": pool,
        "config4": dict(c4, extract_ms=extract_ms, all_gather_ms=gather_alone_ms, utts=n_total),
        "config3_ecapa": c3,
        "config5": c5,
    }
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(14.0)
        line["c1_single_utterance"] = c1_latency(dev)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no GPU visible -- the native arm has no CPU fallback")
        run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
