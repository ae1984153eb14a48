"""Ragged against bucketed extraction on one B200, all measurements in one run.

    python tools/bench_ragged.py --out DIR        -> DIR/ragged.json (+ a summary on stdout)

Model: an 80-d x-vector ("far") from a seeded state dict.  Input: 50 000 utterances of synthetic features whose lengths
follow a VoxCeleb1-O-like mix (4 s + lognormal(ln 3 s, 0.8), 100 frames/s, capped at 10 000 frames): about 40 M frames,
13 GB of fp32 features, far more than the 126 MB of L2, held in one pinned host matrix.
Arms, each warmed up once (every batch shape built), then run alternately --reps times:
  (a) today's path: the pipeline's exact-length Batcher (batch 256, 4 M pending frames) + extract_embedding_batch per
      bucket, on views of the same host matrix (no ark I/O);
  (b) Extractor.extract_ragged_shard_host on the pinned matrix (batch 256, 262 144 padded frames per batch);
  (c) the benchmark shape, 125 000 x 200 frames: extract_shard_host against extract_ragged_shard_host on the same pinned
      data -- what the ragged machinery costs where it buys nothing.
Rates are wall-clock over whole calls that end in a device synchronisation: real frames/s counts the utterances' own
frames, padded frames/s the frames the GEMMs processed (B x T per call)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from asv_subtools_b200 import ops  # noqa: E402
from asv_subtools_b200.model.xvector import Xvector  # noqa: E402
from asv_subtools_b200.pipeline.extract_embeddings import Batcher  # noqa: E402
from oracle import nnet as onn  # noqa: E402


def mix_lengths(n, seed):
    rng = np.random.RandomState(seed)
    return np.minimum(400 + rng.lognormal(np.log(300), 0.8, n), 10000).astype(np.int64)


def fill_pinned(rows, dim, seed):
    """(rows, dim) pinned fp32 matrix: a 1 M-row seeded block repeated (generation at memory speed)."""
    host = torch.empty(rows, dim, dtype=torch.float32, pin_memory=True)
    block = torch.from_numpy((np.random.RandomState(seed).standard_normal((1 << 20, dim)) * 0.5).astype(np.float32))
    for r in range(0, rows, block.shape[0]):
        n = min(block.shape[0], rows - r)
        host[r:r + n].copy_(block[:n])
    return host


def rel_rows(a, b):
    d = np.abs(a.astype(np.float64) - b.astype(np.float64)).max(axis=1)
    return float((d / np.maximum(np.abs(b).max(axis=1), 1e-30)).max())


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the name from torch still identifies the card
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown ({})".format(e)}


def spread(rates):
    r = sorted(rates)
    return {"median": r[len(r) // 2], "min": r[0], "max": r[-1], "runs": rates}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--utts", type=int, default=50000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=20261017)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_ragged.py measures on a B200"
    torch.cuda.set_device(0)
    os.makedirs(args.out, exist_ok=True)
    info = {"card": card(), "torch": torch.__version__}

    m = Xvector(80, 10, training=False, extracted_embedding="far")
    m.load_state_dict(onn.make_state_dict(onn.xvector_spec(80), 102), strict=True)
    m.cuda().eval()
    ex = m.extractor()

    # ---- the length mix
    lengths = mix_lengths(args.utts, args.seed)
    off = np.zeros(args.utts + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    t0 = time.time()
    feats = fill_pinned(int(off[-1]), 80, args.seed)
    fv = feats.numpy()
    utts = [fv[off[i]:off[i + 1]] for i in range(args.utts)]
    info["setup_s"] = time.time() - t0
    real = int(off[-1])

    def arm_a():
        batcher, out, padded, calls = Batcher(256), np.empty((args.utts, 512), np.float32), 0, 0

        def run(bucket):
            nonlocal padded, calls
            idx = [i for i, _ in bucket]
            x = np.stack([f for _, f in bucket])
            out[idx] = m.extract_embedding_batch(x).cpu().numpy()
            padded += x.shape[0] * x.shape[1]
            calls += 1
        for i, f in enumerate(utts):
            for bucket in batcher.add(i, f):
                run(bucket)
        for bucket in batcher.flush():
            run(bucket)
        return out, padded, calls

    order, batches = ops.ragged_plan(off, 256, 0)
    tq = [(int(lengths[b].max()) + 31) // 32 * 32 for b in batches]
    padded_b = int(sum(len(b) * t for b, t in zip(batches, tq)))

    def arm_b():
        return ex.extract_ragged_shard_host(feats, off, batch=256, max_frames=0)

    # ---- the benchmark shape
    nc, tc = 125000, 200
    feats_c = fill_pinned(nc * tc, 80, args.seed + 1)
    off_c = np.arange(nc + 1, dtype=np.int64) * tc
    emb_c = torch.empty(nc, 512, dtype=torch.float32, pin_memory=True)

    def arm_c_shard():
        ex.extract_shard_host(feats_c.data_ptr(), nc, tc, emb_c.data_ptr(), batch=256)
        return emb_c

    def arm_c_ragged():
        return ex.extract_ragged_shard_host(feats_c, off_c, batch=256, max_frames=0)

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t, r

    # warm-up: every batch shape of every arm (plans, tensor maps, workspace)
    _, (emb_a, padded_a, calls_a) = timed(arm_a)
    _, emb_b = timed(arm_b)
    emb_cs = timed(arm_c_shard)[1].numpy().copy()
    _, emb_cr = timed(arm_c_ragged)
    times = {"a": [], "b": [], "c_shard": [], "c_ragged": []}
    for _ in range(args.reps):
        times["a"].append(timed(arm_a)[0])
        times["b"].append(timed(arm_b)[0])
        times["c_shard"].append(timed(arm_c_shard)[0])
        times["c_ragged"].append(timed(arm_c_ragged)[0])
    bucket_lengths = len(np.unique(lengths))
    res = dict(info)
    res["mix"] = {"utterances": args.utts, "real_frames": real, "distinct_lengths": bucket_lengths,
                  "length_mean": float(lengths.mean()), "length_median": float(np.median(lengths)),
                  "length_max": int(lengths.max())}
    res["a_bucketed"] = {"calls": calls_a, "padded_frames": padded_a, "padded_fraction": 1 - real / padded_a,
                         "distinct_T": bucket_lengths, "seconds": times["a"],
                         "real_frames_per_s": spread([real / t for t in times["a"]]),
                         "padded_frames_per_s": spread([padded_a / t for t in times["a"]])}
    res["b_ragged"] = {"calls": 1, "batches": len(batches), "padded_frames": padded_b, "padded_fraction": 1 - real / padded_b,
                       "distinct_Tq": len(set(tq)), "seconds": times["b"],
                       "real_frames_per_s": spread([real / t for t in times["b"]]),
                       "padded_frames_per_s": spread([padded_b / t for t in times["b"]])}
    res["speedup_b_over_a_median"] = res["b_ragged"]["real_frames_per_s"]["median"] / res["a_bucketed"]["real_frames_per_s"]["median"]
    res["max_rel_a_vs_b"] = rel_rows(emb_b, emb_a)
    fc = nc * tc
    res["c_bench_shape"] = {"utterances": nc, "frames": tc,
                            "shard_host": {"seconds": times["c_shard"], "frames_per_s": spread([fc / t for t in times["c_shard"]])},
                            "ragged_shard_host": {"seconds": times["c_ragged"], "frames_per_s": spread([fc / t for t in times["c_ragged"]])},
                            "max_rel": rel_rows(emb_cr, emb_cs), "bit_identical": bool(np.array_equal(emb_cr, emb_cs))}
    res["c_ragged_over_shard_time_median"] = float(np.median(times["c_ragged"]) / np.median(times["c_shard"]))
    with open(os.path.join(args.out, "ragged.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "speedup_b_over_a_median", "max_rel_a_vs_b", "c_ragged_over_shard_time_median")}))
    print("a: {} calls, {:.3g} real frames/s;  b: {} batches, {} distinct Tq, padded {:.1%}, {:.3g} real frames/s".format(
        calls_a, res["a_bucketed"]["real_frames_per_s"]["median"], len(batches), len(set(tq)), res["b_ragged"]["padded_fraction"],
        res["b_ragged"]["real_frames_per_s"]["median"]))


if __name__ == "__main__":
    main()
