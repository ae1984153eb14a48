"""Ragged batches through the TDNN x-vector extractor: utterances of different lengths in one call, each computed as the
reference computes it alone (extract_embeddings.py:73-83; every TdnnAffine zero-pads its own input, components.py:117;
pooling over the utterance's own frames, pooling.py:58-67).  Needs a B200 (`-m gpu`)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from asv_subtools_b200 import kaldi_io, ops
from asv_subtools_b200._lib import XvbError
from oracle import nnet as onn

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "asv_subtools_b200", "bin", "xvb-extract")
GEMM_TOL = 3e-5
EMB_TOL = 1e-4
ORDER_TOL = 2e-6   # same frame outputs, pooling partials merged in another order (as fused vs unfused pooling)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def _xvector(dim, seed, pos):
    from asv_subtools_b200.model.xvector import Xvector
    m = Xvector(dim, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(onn.make_state_dict(onn.xvector_spec(dim), seed), strict=True)
    return m.cuda().eval()


def _ragged(utts):
    """list of (T_i, F) arrays -> ((sum_T, F) CUDA tensor, offsets)"""
    off = np.zeros(len(utts) + 1, dtype=np.int64)
    np.cumsum([u.shape[0] for u in utts], out=off[1:])
    return torch.from_numpy(np.concatenate(utts)).cuda(), off


# ---------------------------------------------------------------- 1. masked layer
@pytest.mark.parametrize("context", [[-2, -1, 0, 1, 2], [-3, 0, 3], [0, 2], [0]])
@pytest.mark.parametrize("f32", [False, True])
def test_masked_layer_matches_each_utterance_alone(context, f32):
    lengths = [1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 96]          # Tb multiples +- 1
    B, Tq, Cin, Cout = len(lengths), 96, 64, 256
    rng = np.random.RandomState(sum(context) + 50)
    left, right, tot = onn.context_span(context)
    w = (rng.standard_normal((Cout, Cin, tot)) * np.sqrt(2.0 / (Cin * len(context)))).astype(np.float32)
    b = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    x = np.zeros((B, Tq, Cin), np.float32)
    for i, L in enumerate(lengths):
        x[i, :L] = rng.standard_normal((L, Cin))
    xp = ops.split_f32(torch.from_numpy(x).cuda())
    wp = ops.pack_tdnn_weight(torch.from_numpy(w).cuda(), context)
    lens = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    y = ops.SplitPlanes.empty((B, Tq, Cout), "cuda")
    y.hi.fill_(1.0)
    y.lo.fill_(1.0)
    yf = torch.full((B, Tq, Cout), 7.0, device="cuda") if f32 else None
    ops.tdnn_affine_ex(xp, wp, Cout, context, bias=torch.from_numpy(b).cuda(), relu=True, y=y, y_f32=yf, lengths=lens)
    torch.cuda.synchronize()
    got = y.float().cpu().numpy()
    for i, L in enumerate(lengths):
        with torch.no_grad():
            want = torch.relu(onn.tdnn_affine(torch.from_numpy(x[i:i + 1, :L]).transpose(1, 2), torch.from_numpy(w),
                                              torch.from_numpy(b), context)).transpose(1, 2)[0].numpy()
        assert rel(got[i, :L], want) < GEMM_TOL, (i, L)
        assert torch.all(y.hi[i, L:] == 0) and torch.all(y.lo[i, L:] == 0), (i, L)
        if f32:
            assert rel(yf[i, :L].cpu().numpy(), want) < GEMM_TOL and torch.all(yf[i, L:] == 0), (i, L)


# ---------------------------------------------------------------- 2. goldens
@pytest.mark.parametrize("dim,seed", [(23, 101), (80, 102)])
@pytest.mark.parametrize("pos", ["far", "near"])
def test_ragged_batch_matches_xvector_golden(golden, dim, seed, pos):
    g = golden("xvector")
    m = _xvector(dim, seed, pos)
    f200 = onn.synthetic_feats(4, 200, dim, seed + 1000)
    short = [onn.synthetic_feats(1, T, dim, seed + 3000 + T)[0] for T in (1, 3, 7)]
    utts = [f200[0], short[0], f200[1], short[1], f200[2], short[2], f200[3]]
    x, off = _ragged(utts)
    got = m.extractor().extract_ragged(x, off).cpu().numpy()
    via_list = m.extract_embedding_ragged(utts).numpy()
    want200 = g["xv{}_{}_emb".format(dim, pos)]
    for j, i in enumerate((0, 2, 4, 6)):
        for emb in (got[i], via_list[i]):
            assert rel(emb, want200[j]) < EMB_TOL
            assert np.dot(emb, want200[j]) / (np.linalg.norm(emb) * np.linalg.norm(want200[j])) > 1 - 1e-6
    for T, i in zip((1, 3, 7), (1, 3, 5)):
        want = g["xv{}_far_T{}".format(dim, T)] if pos == "far" else m.extract_embedding(short[(i - 1) // 2]).numpy()
        assert rel(got[i], want) < EMB_TOL and rel(via_list[i], want) < EMB_TOL, T


@pytest.mark.parametrize("pos", ["far", "near"])
def test_ragged_batch_matches_extended_and_snowdar_goldens(golden, pos):
    from asv_subtools_b200.model.extended_xvector import ExtendedXvector
    from asv_subtools_b200.model.snowdar_xvector import Xvector as SnowdarXvector
    g = golden("xvector")
    m = ExtendedXvector(80, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(onn.make_state_dict(onn.extended_xvector_spec(80), 103), strict=True)
    m.cuda().eval()
    feats = onn.synthetic_feats(3, 150, 80, 1103)
    extra = onn.synthetic_feats(1, 7, 80, 77)[0]
    got = m.extract_embedding_ragged([feats[0], extra, feats[1], feats[2]]).numpy()
    for j, i in enumerate((0, 2, 3)):
        assert rel(got[i], g["ext80_{}_emb".format(pos)][j]) < EMB_TOL
    assert rel(got[1], m.extract_embedding(extra).numpy()) < ORDER_TOL
    gs = golden("snowdar")
    sd = onn.make_state_dict(onn.snowdar_xvector_spec(40, extend=False), 301)
    feats = onn.synthetic_feats(3, 120, 40, 1301)
    extra = onn.synthetic_feats(1, 3, 40, 78)[0]
    for p in (("far", "near_affine") if pos == "far" else ("near",)):
        m = SnowdarXvector(40, 10, extend=False, training=False, extracted_embedding=p)
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        got = m.extract_embedding_ragged([extra, feats[0], feats[1], feats[2]]).numpy()
        assert rel(got[1:], gs["std_{}".format(p)]) < EMB_TOL, p
        assert rel(got[0], m.extract_embedding(extra).numpy()) < ORDER_TOL, p


# ---------------------------------------------------------------- 3. against the per-utterance path
@pytest.mark.parametrize("pos", ["far", "near"])
def test_ragged_matches_per_utterance_extraction(pos):
    m = _xvector(80, 102, pos)
    rng = np.random.RandomState(7)
    lengths = rng.randint(1, 3001, size=45)
    lengths[:4] = [1, 3000, 32, 33]
    utts = [onn.synthetic_feats(1, int(T), 80, 5000 + i)[0] for i, T in enumerate(lengths)]
    single = np.stack([m.extract_embedding(u).numpy() for u in utts])
    got = m.extract_embedding_ragged(utts).numpy()
    x, off = _ragged(utts)
    dev = m.extractor().extract_ragged(x, off).cpu().numpy()
    for i in range(len(utts)):
        assert rel(got[i], single[i]) <= ORDER_TOL, (i, lengths[i])
        assert rel(dev[i], single[i]) <= ORDER_TOL, (i, lengths[i])


# ---------------------------------------------------------------- 4. no leakage, 5. equal lengths
def test_no_leakage_from_workspace_or_companions():
    m = _xvector(80, 102, "near")
    ex = m.extractor()
    long = onn.synthetic_feats(8, 500, 80, 1)
    ex.extract_ragged(*_ragged(list(long)))                       # leaves non-zero data all over the workspace
    u = onn.synthetic_feats(1, 40, 80, 2)[0]
    top = onn.synthetic_feats(1, 128, 80, 3)[0]
    short = [onn.synthetic_feats(1, 5, 80, 10 + i)[0] for i in range(6)]
    longc = [onn.synthetic_feats(1, 120 + i, 80, 20 + i)[0] for i in range(6)]
    a = ex.extract_ragged(*_ragged([u] + short + [top])).clone()  # (B, Tq) = (8, 128) both times
    b = ex.extract_ragged(*_ragged([u] + longc + [top])).clone()
    again = ex.extract_ragged(*_ragged([u] + short + [top])).clone()
    assert torch.equal(a[0], b[0]) and torch.equal(a[-1], b[-1])
    assert torch.equal(a, again)


def test_equal_lengths_are_bit_identical_to_the_batch_path():
    m = _xvector(80, 102, "far")
    feats = onn.synthetic_feats(64, 256, 80, 4)
    want = m.extract_embedding_batch(feats)
    x = torch.from_numpy(feats.reshape(-1, 80)).cuda()
    got = m.extractor().extract_ragged(x, np.arange(65) * 256)
    assert torch.equal(got, want)


# ---------------------------------------------------------------- 6. shard call
def test_ragged_shard_matches_per_batch_calls_in_input_order():
    m = _xvector(23, 101, "far")
    ex = m.extractor()
    rng = np.random.RandomState(11)
    n, batch, max_frames = 1999, 48, 12288
    lengths = rng.randint(1, 2401, size=n)
    lengths[100] = 5000                                            # longer than max_frames: a batch of its own
    feats = (rng.standard_normal((int(lengths.sum()), 23)) * 0.5).astype(np.float32)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    order, batches = ops.ragged_plan(off, batch, max_frames)
    keys = [(len(bt), (int(lengths[bt].max()) + 31) // 32) for bt in batches]
    assert max(len(set(keys[0::2])), len(set(keys[1::2]))) > 64            # more (B, Tq) plans than a lane keeps
    assert [len(bt) for bt in batches].count(1) >= 1 and n % batch != 0
    got = ex.extract_ragged_shard_host(feats, off, batch=batch, max_frames=max_frames)
    want = np.empty_like(got)
    for bt in batches:
        x, o = _ragged([feats[off[i]:off[i + 1]] for i in bt])
        want[bt] = ex.extract_ragged(x, o).cpu().numpy()
    assert np.array_equal(got, want)
    pinned = torch.empty(feats.shape, dtype=torch.float32, pin_memory=True)
    pinned.copy_(torch.from_numpy(feats))
    assert np.array_equal(ex.extract_ragged_shard_host(pinned, off, batch=batch, max_frames=max_frames), want)


# ---------------------------------------------------------------- 7. errors, 8. fallback
def test_ragged_errors():
    m = _xvector(80, 102, "far")
    ex = m.extractor()
    x, off = _ragged([onn.synthetic_feats(1, 20, 80, 1)[0], onn.synthetic_feats(1, 30, 80, 2)[0]])
    with pytest.raises(XvbError):
        ex.extract_ragged(x, [0, 20, 20, 50])                      # a zero-length utterance
    ex.set_fused_pooling(False)
    with pytest.raises(XvbError):
        ex.extract_ragged(x, off)
    ex.set_fused_pooling(True)
    table = torch.zeros(64, 512, device="cuda")
    ptrs = (C.c_void_p * 1)(table.data_ptr())
    ex.set_gather(ptrs, 1, 0, 512)
    try:
        with pytest.raises(XvbError):
            ex.extract_ragged(x, off)
        with pytest.raises(XvbError):
            ex.extract_ragged_shard_host(x.cpu().numpy(), off)
    finally:
        ex.set_gather(None, 0, 0, 0)
    assert ex.extract_ragged(x, off).shape == (2, 512)
    with pytest.raises(ValueError, match="extract_embedding"):
        m.extract_embedding_ragged([onn.synthetic_feats(1, 10001, 80, 3)[0]])


def test_fallback_for_models_without_a_ragged_path():
    from asv_subtools_b200.model.snowdar_xvector import Xvector
    sd = onn.make_state_dict(onn.snowdar_xvector_spec(40, pooling="attentive", pooling_params={}), 311)
    m = Xvector(40, 10, training=False, extracted_embedding="far", pooling="attentive", pooling_params={})
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    lengths = [50, 7, 50, 120, 7, 50]
    utts = [onn.synthetic_feats(1, T, 40, 60 + i)[0] for i, T in enumerate(lengths)]
    got = m.extract_embedding_ragged(utts)
    for T in set(lengths):
        idx = [i for i, t in enumerate(lengths) if t == T]
        want = m.extract_embedding_batch(np.stack([utts[i] for i in idx])).cpu()
        assert torch.equal(got[idx], want), T


# ---------------------------------------------------------------- 9. CLIs
def _write_ark(path, feats):
    with open(path, "wb") as f:
        for k, v in feats.items():
            kaldi_io.write_mat(f, v, key=k)


def test_clis_ragged_match_the_default_path_in_input_order(tmp_path):
    m = _xvector(80, 102, "far")
    rng = np.random.RandomState(3)
    lengths = list(rng.randint(1, 900, size=40)) + [450, 450, 10050]      # 10050 > maxChunk: the chunk rule
    feats = {"u{:03d}".format(39 - i if i < 40 else i): onn.synthetic_feats(1, int(t), 80, 700 + i)[0]
             for i, t in enumerate(lengths)}
    keys = list(feats)
    ark = str(tmp_path / "feats.ark")
    _write_ark(ark, feats)
    sd = onn.make_state_dict(onn.xvector_spec(80), 102)
    torch.save(sd, str(tmp_path / "final.params"))
    blueprint = os.path.join(ROOT, "asv_subtools_b200", "model", "xvector.py")
    (tmp_path / "nnet.config").write_text(
        'model_blueprint;{}\nmodel_creation;Xvector(80,10,training=False,extracted_embedding="far")\n'.format(blueprint))
    outs = {}
    for mode in ("false", "true"):
        out = str(tmp_path / "py_{}.ark".format(mode))
        run = subprocess.run([sys.executable, "-m", "asv_subtools_b200.pipeline.extract_embeddings", "--nnet-config",
                              str(tmp_path / "nnet.config"), "--ragged", mode, str(tmp_path / "final.params"), "ark:" + ark,
                              "ark:" + out], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert run.returncode == 0, run.stdout + run.stderr
        outs["py_" + mode] = list(kaldi_io.read_vec_flt_ark(out))
    model = str(tmp_path / "xv80.xvbm")
    m.extractor().save(model)
    for mode, extra in (("false", []), ("true", ["--ragged"])):
        out = str(tmp_path / "bin_{}.ark".format(mode))
        run = subprocess.run([BIN] + extra + [model, "ark:" + ark, "ark:" + out], capture_output=True, text=True, timeout=600)
        assert run.returncode == 0, run.stdout + run.stderr
        outs["bin_" + mode] = list(kaldi_io.read_vec_flt_ark(out))
    for tool in ("py", "bin"):
        base, rag = dict(outs[tool + "_false"]), outs[tool + "_true"]
        assert [k for k, _ in rag] == keys, tool                        # input order
        assert sorted(base) == sorted(keys)
        for k, v in rag:
            assert rel(v, base[k]) <= ORDER_TOL, (tool, k)


def test_xvb_extract_ragged_rejects_an_ecapa_model(tmp_path):
    from asv_subtools_b200.model.ecapa_tdnn_xvector import ECAPA_TDNN
    canon = dict(training=False, extracted_embedding="near",
                 ecapa_params={"channels": 1024, "embd_dim": 192, "mfa_conv": 1536,
                               "bn_params": {"momentum": 0.5, "affine": True, "track_running_stats": True}},
                 fc2_params={"nonlinearity": "", "bn": True, "bn_params": {"momentum": 0.5, "affine": False, "track_running_stats": True}})
    m = ECAPA_TDNN(80, 10, **canon)
    m.load_state_dict(onn.make_state_dict(onn.ecapa_spec(80), 201), strict=True)
    m.cuda().eval()
    model = str(tmp_path / "ecapa.xvbm")
    m.extractor().save(model)
    ark = str(tmp_path / "feats.ark")
    _write_ark(ark, {"e0": onn.synthetic_feats(1, 50, 80, 1)[0]})
    run = subprocess.run([BIN, "--ragged", model, ark, "ark:" + str(tmp_path / "xv.ark")], capture_output=True, text=True,
                         timeout=300)
    assert run.returncode == 1 and "ERROR" in run.stderr and "ragged" in run.stderr
