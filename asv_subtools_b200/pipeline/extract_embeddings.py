# -*- coding:utf-8 -*-
"""Batched embedding extractor -- CLI twin of pytorch/pipeline/onestep/extract_embeddings.py.

Same positionals and flags (extract_embeddings.py:17-45):

    python -m asv_subtools_b200.pipeline.extract_embeddings [--nnet-config F | --model-blueprint P
        --model-creation S] [--use-gpu true] [--gpu-id ID] <model-path> <feats-rspecifier> <vectors-wspecifier>

What differs from the reference loop (:73-83, one utterance per iteration): utterances are read
from the ark stream, bucketed by frame count, and every bucket is extracted in ONE call of
`extract_embedding_batch()` (equal-length utterances need no padding, exactly like
splitDataByLength.sh-balanced jobs); utterances longer than maxChunk fall back to the
per-utterance `extract_embedding()` with the reference's chunk rule.  One `FV` vector is written per
input key (bucket order).  `--shard i/n` keeps every n-th utterance (one process per GPU without
pre-splitting the scp).

`--ragged true` replaces the exact-length buckets: utterances are collected in a window of up to
`max_pending_frames` frames, the window is extracted with ONE `extract_embedding_ragged()` call
(length-sorted batches of mixed lengths, each utterance computed as if alone), and the vectors are
written in input order.  Utterances longer than maxChunk keep the per-utterance chunk rule.
"""
import argparse
import os
import sys
import traceback

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

from asv_subtools_b200 import kaldi_io  # noqa: E402

MAX_CHUNK = 10000


def read_nnet_config(path):
    """`;`-separated two-row CSV written by utils.write_nnet_config (utils.py:189-202)."""
    vals = {}
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if ";" in line:
                k, v = line.split(";", 1)
                vals[k.strip()] = v.strip().strip('"').replace('""', '"')
    return vals["model_blueprint"], vals["model_creation"]


def create_model_from_py(model_blueprint, model_creation):
    """Import a blueprint by path and evaluate the creation string (utils.py:163-186)."""
    if not os.path.exists(model_blueprint):
        raise TypeError("Expected {} to exist.".format(model_blueprint))
    sys.path.insert(0, os.path.dirname(os.path.abspath(model_blueprint)))
    module = __import__(os.path.basename(model_blueprint).split(".")[0])
    return eval("module.{0}".format(model_creation), {"module": module})


class Batcher:
    """Buckets (key, feats) by frame count; yields full buckets, and everything at flush()."""

    def __init__(self, batch_size, max_pending_frames=4_000_000, length=None):
        """`length(item)`: the bucketing key (default: rows of the item); `max_pending_frames` bounds what is held
        back waiting for a bucket to fill (in units of that key), after which everything pending is flushed."""
        self.batch_size, self.max_pending = batch_size, max_pending_frames
        self.buckets, self.pending = {}, 0
        self.length = length or (lambda a: a.shape[0])

    def add(self, key, feats):
        t = self.length(feats)
        b = self.buckets.setdefault(t, [])
        b.append((key, feats))
        self.pending += t
        if len(b) >= self.batch_size:
            self.pending -= t * len(b)
            yield self.buckets.pop(t)
        elif self.pending > self.max_pending:
            yield from self.flush()

    def flush(self):
        for t in sorted(self.buckets):
            yield self.buckets[t]
        self.buckets, self.pending = {}, 0


def run_window(model, window, writer):
    """One ragged call for the window's utterances up to maxChunk frames, the chunk rule for longer ones; vectors are
    written in window (= input) order."""
    short = [f for _, f in window if f.shape[0] <= MAX_CHUNK]
    embs = iter(model.extract_embedding_ragged(short).numpy()) if short else iter(())
    for key, feats in window:
        writer(key, next(embs) if feats.shape[0] <= MAX_CHUNK else model.extract_embedding(feats).numpy())


def extract_stream(model, reader, writer, batch_size=256, shard=(0, 1), log=print, ragged=False,
                   max_pending_frames=4_000_000):
    """reader yields (key, (T,F) float32 ndarray); writer(key, 1-D float32 ndarray).  ragged: windows of up to
    max_pending_frames frames through extract_embedding_ragged(), written in input order."""
    if ragged:
        return _extract_stream_ragged(model, reader, writer, shard, log, max_pending_frames)
    batcher = Batcher(batch_size)
    count = 0

    def run(bucket):
        t = bucket[0][1].shape[0]
        if t > MAX_CHUNK:
            for key, feats in bucket:
                writer(key, model.extract_embedding(feats).numpy())
            return
        x = np.stack([f for _, f in bucket])
        emb = model.extract_embedding_batch(x).cpu().numpy()
        for (key, _), e in zip(bucket, emb):
            writer(key, e)

    for i, (key, feats) in enumerate(reader):
        if i % shard[1] != shard[0]:
            continue
        log("Process utterance for key {0}".format(key))
        feats = np.ascontiguousarray(feats)
        if feats.dtype != np.float32:
            raise TypeError("features of {} are {}, the extractor takes float32 (FM/CM) matrices".format(key, feats.dtype))
        count += 1
        for bucket in batcher.add(key, feats):
            run(bucket)
    for bucket in batcher.flush():
        run(bucket)
    return count


def _extract_stream_ragged(model, reader, writer, shard, log, max_pending_frames):
    window, frames, count = [], 0, 0
    for i, (key, feats) in enumerate(reader):
        if i % shard[1] != shard[0]:
            continue
        log("Process utterance for key {0}".format(key))
        feats = np.ascontiguousarray(feats)
        if feats.dtype != np.float32:
            raise TypeError("features of {} are {}, the extractor takes float32 (FM/CM) matrices".format(key, feats.dtype))
        count += 1
        window.append((key, feats))
        frames += feats.shape[0]
        if frames >= max_pending_frames:
            run_window(model, window, writer)
            window, frames = [], 0
    if window:
        run_window(model, window, writer)
    return count


def main(argv=None):
    ap = argparse.ArgumentParser(description="Extract embeddings from a piece of feats.scp or pipeline (B200)")
    ap.add_argument("--nnet-config", type=str, default="")
    ap.add_argument("--model-blueprint", type=str, default=None)
    ap.add_argument("--model-creation", type=str, default=None)
    ap.add_argument("--use-gpu", type=str, default="true", choices=["true", "false"])
    ap.add_argument("--gpu-id", type=str, default="")
    ap.add_argument("--batch-size", type=int, default=256)
    ap.add_argument("--shard", type=str, default="0/1", help="i/n: keep utterances with index %% n == i")
    ap.add_argument("--ragged", type=str, default="false", choices=["true", "false"],
                    help="true: mixed-length batches (extract_embedding_ragged) over windows of utterances, vectors in input "
                         "order; false: exact-length buckets")
    ap.add_argument("--blueprint-dir", type=str, default="",
                    help="take the blueprint of the same file name from this directory (asv_subtools_b200/model) instead of "
                         "the path stored in nnet.config, so a reference model dir is used as it is")
    ap.add_argument("model_path", metavar="model-path")
    ap.add_argument("feats_rspecifier", metavar="feats-rspecifier")
    ap.add_argument("vectors_wspecifier", metavar="vectors-wspecifier")
    print(" ".join(sys.argv))
    args = ap.parse_args(argv)
    try:
        if args.nnet_config != "":
            blueprint, creation = read_nnet_config(args.nnet_config)
        elif args.model_blueprint is not None and args.model_creation is not None:
            blueprint, creation = args.model_blueprint, args.model_creation
        else:
            raise ValueError("Expected nnet_config or (model_blueprint, model_creation) to exist.")
        if args.blueprint_dir:
            swapped = os.path.join(args.blueprint_dir, os.path.basename(blueprint))
            if not os.path.exists(swapped):
                raise FileNotFoundError("no B200 blueprint named {} in {}".format(os.path.basename(blueprint), args.blueprint_dir))
            blueprint = swapped
        if args.use_gpu != "true":
            raise RuntimeError("asv_subtools_b200 has no CPU path: run with --use-gpu true on a B200")
        model = create_model_from_py(blueprint, creation)
        model.load_state_dict(torch.load(args.model_path, map_location="cpu"), strict=False)
        torch.cuda.set_device(int(args.gpu_id.split(",")[0]) if args.gpu_id != "" else 0)
        model.cuda().eval()
        i, n = (int(v) for v in args.shard.split("/"))
        # native ark reader (csrc/ark_io.cpp): the reference's byte-at-a-time key loop is the wall at GPU rates
        with kaldi_io.open_or_fd(args.vectors_wspecifier, "wb") as w:
            extract_stream(model, kaldi_io.read_mat_ark_native(args.feats_rspecifier),
                           lambda k, v: kaldi_io.write_vec_flt(w, v, key=k), batch_size=args.batch_size, shard=(i, n),
                           ragged=args.ragged == "true")
    except BaseException as err:
        if not isinstance(err, KeyboardInterrupt):
            traceback.print_exc()
        sys.exit(1)


if __name__ == "__main__":
    main()
