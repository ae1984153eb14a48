"""Host side of ragged extraction, no GPU: the batching policy xvb_ragged_plan (the one place it lives), and the
window / input-order logic and `--ragged` flag of pipeline/extract_embeddings.py with a stub model."""
import contextlib

import numpy as np
import pytest
import torch

from asv_subtools_b200 import ops
from asv_subtools_b200._lib import XvbError
from asv_subtools_b200.pipeline import extract_embeddings as ee


def _offsets(lengths):
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    return off


def _mix(n, seed):
    """4 s + lognormal(ln 3 s, 0.8) at 100 frames/s, capped at 10 000 frames (a VoxCeleb1-O-like test set)."""
    rng = np.random.RandomState(seed)
    return np.minimum(400 + rng.lognormal(np.log(300), 0.8, n), 10000).astype(np.int64)


def _round32(x):
    return (x + 31) // 32 * 32


@pytest.mark.parametrize("n,batch,max_frames,seed", [(4874, 256, 0, 1), (2000, 64, 50000, 2), (37, 5, 4096, 3),
                                                     (1000, 256, 262144, 4)])
def test_plan_covers_every_utterance_once_within_limits(n, batch, max_frames, seed):
    lengths = _mix(n, seed)
    if n > 100:
        lengths[17] = 9000   # with max_frames 4096 / 50000 below: a long one forms its own batch
    order, batches = ops.ragged_plan(_offsets(lengths), batch=batch, max_frames=max_frames)
    cap = max_frames if max_frames > 0 else 262144
    assert sorted(order.tolist()) == list(range(n))
    assert np.array_equal(np.concatenate(batches), order)
    prev_max = 0
    for bt in batches:
        lb = lengths[bt]
        assert 1 <= len(bt) <= batch
        tq = _round32(lb.max())
        assert tq % 32 == 0
        assert len(bt) * tq <= cap or len(bt) == 1
        assert np.all(np.diff(lb) >= 0) and lb.min() >= prev_max        # sorted within and across batches
        prev_max = lb.max()
    # stable: equal lengths keep input order
    ls = lengths[order]
    for v in np.unique(ls):
        idx = order[ls == v]
        assert np.all(np.diff(idx) > 0)


def test_plan_is_greedy_and_deterministic():
    lengths = _mix(3000, 9)
    a = ops.ragged_plan(_offsets(lengths), 256, 0)
    b = ops.ragged_plan(_offsets(lengths), 256, 0)
    assert np.array_equal(a[0], b[0]) and len(a[1]) == len(b[1])
    assert all(np.array_equal(x, y) for x, y in zip(a[1], b[1]))
    for cur, nxt in zip(a[1][:-1], a[1][1:]):   # a batch stops only when the next utterance would not fit
        grown = np.concatenate([cur, nxt[:1]])
        assert len(cur) == 256 or len(grown) * _round32(lengths[grown].max()) > 262144


def test_plan_long_utterance_and_equal_lengths():
    order, batches = ops.ragged_plan(_offsets([10, 20000, 10, 10]), batch=256, max_frames=1000)
    assert [b.tolist() for b in batches] == [[0, 2, 3], [1]]
    order, batches = ops.ragged_plan(_offsets([200] * 1000), batch=256, max_frames=0)
    assert np.array_equal(order, np.arange(1000)) and [len(b) for b in batches] == [256, 256, 256, 232]


@pytest.mark.parametrize("lengths,batch", [([5, 0, 3], 4), ([5, -2], 4), ([5, 6], 0)])
def test_plan_rejects_bad_arguments(lengths, batch):
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    off[1:] = np.cumsum(lengths)
    with pytest.raises(XvbError):
        ops.ragged_plan(off, batch=batch)
    with pytest.raises(ValueError):
        ops.ragged_plan(np.zeros(1, dtype=np.int64))


# ---------------------------------------------------------------- pipeline --ragged with a stub model
class _StubModel:
    """Embedding of an utterance = [T, sum of its features]; records the calls it gets."""

    def __init__(self):
        self.ragged_calls, self.single_calls = [], []

    @staticmethod
    def _emb(f):
        return np.array([f.shape[0], f.sum()], dtype=np.float32)

    def extract_embedding_ragged(self, feats_list):
        self.ragged_calls.append([f.shape[0] for f in feats_list])
        return torch.from_numpy(np.stack([self._emb(f) for f in feats_list]))

    def extract_embedding(self, feats):
        self.single_calls.append(feats.shape[0])
        return torch.from_numpy(self._emb(feats))


def _utts(n, seed):
    rng = np.random.RandomState(seed)
    return [("utt{:03d}".format(i), rng.standard_normal((int(rng.randint(1, 12)), 3)).astype(np.float32)) for i in range(n)]


def test_ragged_stream_windows_and_input_order(monkeypatch):
    monkeypatch.setattr(ee, "MAX_CHUNK", 8)        # utterances of 9..11 frames take the per-utterance chunk rule
    utts = _utts(40, 5)
    model, out = _StubModel(), []
    count = ee.extract_stream(model, iter(utts), lambda k, v: out.append((k, v)), ragged=True, max_pending_frames=50,
                              log=lambda *_: None)
    assert count == 40
    assert [k for k, _ in out] == [k for k, _ in utts]
    for (k, v), (_, f) in zip(out, utts):
        assert np.array_equal(v, _StubModel._emb(f)), k
    assert sum(len(c) for c in model.ragged_calls) == sum(1 for _, f in utts if f.shape[0] <= 8)
    assert sorted(model.single_calls) == sorted(f.shape[0] for _, f in utts if f.shape[0] > 8)
    assert len(model.ragged_calls) >= 2                                      # 50-frame windows: several calls
    out2 = []
    ee.extract_stream(_StubModel(), iter(utts), lambda k, v: out2.append(k), ragged=True, shard=(1, 3), log=lambda *_: None)
    assert out2 == [k for i, (k, _) in enumerate(utts) if i % 3 == 1]


def test_ragged_flag(monkeypatch, tmp_path):
    seen = {}

    class _Loadable:
        def load_state_dict(self, *a, **k):
            pass

        def cuda(self):
            return self

        def eval(self):
            return self

    monkeypatch.setattr(ee, "create_model_from_py", lambda *a: _Loadable())
    monkeypatch.setattr(ee.torch, "load", lambda *a, **k: {})
    monkeypatch.setattr(ee.torch.cuda, "set_device", lambda *a: None)
    monkeypatch.setattr(ee.kaldi_io, "read_mat_ark_native", lambda spec: iter(()))
    monkeypatch.setattr(ee.kaldi_io, "open_or_fd", lambda *a: contextlib.nullcontext(None))
    monkeypatch.setattr(ee, "extract_stream", lambda *a, **k: seen.update(k))
    args = ["--model-blueprint", "bp.py", "--model-creation", "X()", "m.params", "ark:f.ark", "ark:v.ark"]
    ee.main(args)
    assert seen["ragged"] is False
    ee.main(["--ragged", "true"] + args)
    assert seen["ragged"] is True
    with pytest.raises(SystemExit):
        ee.main(["--ragged", "yes"] + args)
