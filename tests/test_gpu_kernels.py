"""Parity tests proper: every CUDA kernel, called through the C ABI, against the CPU oracle on the
same seeded inputs.  Needs a B200 (`-m gpu`)."""
import numpy as np
import pytest
import torch

from oracle import nnet as onn

pytestmark = pytest.mark.gpu

# bf16x3 split GEMM: per-product error <= ~3*2^-18; measured as max|d| / max|ref| per tensor.
GEMM_TOL = 3e-5
EMB_TOL = 1e-4  # north-star tolerance for embeddings (fp32, relative to the largest component)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


@pytest.fixture(scope="module")
def ops():
    from asv_subtools_b200 import ops as _ops
    assert torch.cuda.is_available()
    return _ops


def _layer_inputs(B, T, Cin, Cout, context, seed, bn=True):
    rng = np.random.RandomState(seed)
    left, right, tot = onn.context_span(context)
    x = rng.standard_normal((B, T, Cin)).astype(np.float32)
    w = (rng.standard_normal((Cout, Cin, tot)) * np.sqrt(2.0 / (Cin * len(context)))).astype(np.float32)
    b = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    scale = rng.uniform(0.5, 1.5, Cout).astype(np.float32) if bn else None
    shift = (0.1 * rng.standard_normal(Cout)).astype(np.float32) if bn else None
    return x, w, b, scale, shift


def _oracle_layer(x, w, b, scale, shift, context, relu):
    with torch.no_grad():
        y = onn.tdnn_affine(torch.from_numpy(x).transpose(1, 2), torch.from_numpy(w), torch.from_numpy(b), context)
        if relu:
            y = torch.relu(y)
        if scale is not None:
            y = y * torch.from_numpy(scale)[None, :, None] + torch.from_numpy(shift)[None, :, None]
    return y.transpose(1, 2).contiguous().numpy()


def test_split_planes(ops):
    x = torch.randn(37, 23, device="cuda") * 3
    p = ops.split_f32(x)
    assert p.hi.shape == (37, 24) and p.hi.dtype == torch.bfloat16
    back = p.float()
    assert rel(back.cpu().numpy(), x.cpu().numpy()) < 2.0 ** -16
    assert torch.all(p.hi[:, 23] == 0) and torch.all(p.lo[:, 23] == 0)


def test_pack_weight_drops_masked_taps(ops):
    rng = np.random.RandomState(0)
    w = rng.standard_normal((40, 24, 7)).astype(np.float32)  # context [-3,0,3]: taps 1,2,4,5 are garbage
    p = ops.pack_tdnn_weight(torch.from_numpy(w).cuda(), [-3, 0, 3])
    assert p.hi.shape == (40, 3 * 32)  # K index = tap*cin_p16 + c, cin_p16 = 32
    full = (p.hi.float() + p.lo.float()).cpu().numpy().reshape(40, 3, 32)
    want = np.stack([w[:, :, 0], w[:, :, 3], w[:, :, 6]], axis=1)
    assert rel(full[:, :, :24], want) < 2.0 ** -16
    assert np.all(full[:, :, 24:] == 0)


@pytest.mark.parametrize("B,T,Cin,Cout,context,relu", [
    (2, 19, 24, 64, [-2, -1, 0, 1, 2], True),
    (1, 5, 16, 32, [-3, 0, 3], False),
])
def test_simt_layer_vs_oracle(ops, B, T, Cin, Cout, context, relu):
    x, w, b, scale, shift = _layer_inputs(B, T, Cin, Cout, context, 3)
    y = ops.tdnn_affine_simt(torch.from_numpy(x).cuda(), torch.from_numpy(w).cuda(), context,
                             torch.from_numpy(b).cuda(), torch.from_numpy(scale).cuda(),
                             torch.from_numpy(shift).cuda(), relu=relu)
    assert rel(y.cpu().numpy(), _oracle_layer(x, w, b, scale, shift, context, relu)) < 1e-5


GEMM_CASES = [
    # B, T, Cin, Cout, context, relu, f32-out   (M tiles / N tiles / K tails exercised).  These small shapes run the
    # <32,1,1> and <64,1,1> instantiations only; test_gpu_gemm_variants.py reaches the others.
    (2, 50, 24, 512, [-2, -1, 0, 1, 2], True, False),   # tdnn1, 23->24-dim MFCC: partial K step
    (3, 37, 80, 512, [-2, -1, 0, 1, 2], True, False),   # tdnn1, 80-dim fbank: 64+16 channel blocks, ragged T
    (2, 40, 512, 512, [-2, 0, 2], True, False),         # tdnn2: masked taps dropped
    (1, 7, 512, 512, [-3, 0, 3], True, False),          # tdnn3: T < context span, padding dominates
    (5, 16, 512, 512, [0], True, False),                # tdnn4
    (2, 33, 512, 1500, [0], True, True),                # tdnn5 shape, fp32 out: <32,1,1>, N tail 1500 = 46*32+28
    (9, 1, 3000, 512, [0], False, True),                # tdnn6.affine: segment level, M=B rows, narrow N tiles
    (200, 8, 128, 128, [-2, 0, 2], True, False),        # Res2Net-shaped block: 13 M blocks, 52 <32,1,1> tiles, one per CTA
    (16, 200, 512, 512, [-2, 0, 2], True, False),       # Tb=8 x Bb=16 tiling of the BASELINE shape
]


@pytest.mark.parametrize("B,T,Cin,Cout,context,relu,f32out", GEMM_CASES)
def test_tdnn_gemm_vs_oracle(ops, B, T, Cin, Cout, context, relu, f32out):
    x, w, b, scale, shift = _layer_inputs(B, T, Cin, Cout, context, 11)
    xp = ops.split_f32(torch.from_numpy(x).cuda())
    wp = ops.pack_tdnn_weight(torch.from_numpy(w).cuda(), context)
    y, yf = ops.tdnn_affine(xp, wp, Cout, context, torch.from_numpy(b).cuda(), torch.from_numpy(scale).cuda(),
                            torch.from_numpy(shift).cuda(), relu=relu, out_planes=not f32out, out_f32=f32out)
    torch.cuda.synchronize()
    got = (yf if f32out else y.float()).cpu().numpy()
    ref = _oracle_layer(x, w, b, scale, shift, context, relu)
    assert got.shape == ref.shape
    assert np.all(np.isfinite(got))
    assert rel(got, ref) < GEMM_TOL
    # device-side cross-check against the fp32 CUDA-core layer reading the *unpacked* weight
    simt = ops.tdnn_affine_simt(torch.from_numpy(x).cuda(), torch.from_numpy(w).cuda(), context,
                                torch.from_numpy(b).cuda(), torch.from_numpy(scale).cuda(),
                                torch.from_numpy(shift).cuda(), relu=relu).cpu().numpy()
    assert rel(got, simt) < GEMM_TOL


def test_tdnn_gemm_zero_padding_is_exact(ops):
    """Linearity/padding property: frames outside [0,T) contribute exactly nothing, and utterances
    never leak into each other: an all-zero utterance next to a non-zero one stays at relu(bias)."""
    B, T, Cin, Cout, context = 4, 20, 64, 64, [-3, 0, 3]
    x, w, b, _, _ = _layer_inputs(B, T, Cin, Cout, context, 5, bn=False)
    x[1] = 0
    xp = ops.split_f32(torch.from_numpy(x).cuda())
    wp = ops.pack_tdnn_weight(torch.from_numpy(w).cuda(), context)
    _, yf = ops.tdnn_affine(xp, wp, Cout, context, torch.from_numpy(b).cuda(), relu=True, out_planes=False, out_f32=True)
    got = yf.cpu().numpy()
    assert np.array_equal(got[1], np.broadcast_to(np.maximum(b, 0), (T, Cout)))


@pytest.mark.parametrize("B,T,C", [(3, 200, 1500), (2, 1, 1500), (2, 7, 512), (1, 1000, 128), (4, 64, 4)])
def test_stats_pool_vs_oracle(ops, B, T, C):
    rng = np.random.RandomState(21)
    x = (rng.standard_normal((B, T, C)) * rng.uniform(0.1, 3.0, (1, 1, C)) + rng.standard_normal((1, 1, C))).astype(np.float32)
    out, planes = ops.stats_pool(torch.from_numpy(x).cuda(), planes=True)
    with torch.no_grad():
        ref = onn.statistics_pooling(torch.from_numpy(x).transpose(1, 2)).squeeze(2).numpy()
    assert rel(out.cpu().numpy(), ref) < 2e-6
    assert rel(planes.float().cpu().numpy(), ref) < 2.0 ** -16


def test_stats_pool_constant_input_clamps_to_eps(ops):
    x = torch.full((2, 50, 8), 3.25, device="cuda")
    out = ops.stats_pool(x, eps=1e-10).cpu().numpy()
    assert np.allclose(out[:, :8], 3.25) and np.allclose(out[:, 8:], 1e-5, rtol=1e-3)  # sqrt(clamp(0, 1e-10))


# ---------------------------------------------------------------- whole model vs golden fixtures
def _model(dim, seed, pos):
    from asv_subtools_b200.model.xvector import Xvector
    sd = onn.make_state_dict(onn.xvector_spec(dim), seed)
    m = Xvector(dim, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval(), sd


@pytest.mark.parametrize("dim,seed", [(23, 101), (80, 102)])
@pytest.mark.parametrize("pos", ["far", "near"])
def test_xvector_embeddings_match_reference_golden(golden, dim, seed, pos):
    g = golden("xvector")
    m, _ = _model(dim, seed, pos)
    feats = onn.synthetic_feats(4, 200, dim, seed + 1000)
    ref = g["xv{}_{}_emb".format(dim, pos)]
    single = np.stack([m.extract_embedding(feats[i]).numpy() for i in range(4)])
    batch = m.extract_embedding_batch(feats).cpu().numpy()
    assert single.shape == (4, 512) and single.dtype == np.float32
    for i in range(4):
        assert rel(single[i], ref[i]) < EMB_TOL
        assert rel(batch[i], ref[i]) < EMB_TOL
        cos = np.dot(batch[i], ref[i]) / (np.linalg.norm(batch[i]) * np.linalg.norm(ref[i]))
        assert cos > 1 - 1e-6


@pytest.mark.parametrize("dim,seed", [(23, 101), (80, 102)])
def test_xvector_edge_lengths(golden, dim, seed):
    g = golden("xvector")
    m, _ = _model(dim, seed, "far")
    for T in (1, 3, 7):
        f = onn.synthetic_feats(1, T, dim, seed + 3000 + T)[0]
        assert rel(m.extract_embedding(f).numpy(), g["xv{}_far_T{}".format(dim, T)]) < EMB_TOL


def test_xvector_chunked_long_utterance(golden):
    g = golden("xvector")
    m, _ = _model(23, 101, "far")
    f = onn.synthetic_feats(1, 10050, 23, 4242)[0]
    assert rel(m.extract_embedding(f).numpy(), g["xv23_far_T10050"]) < EMB_TOL


def test_xvector_intermediates(golden):
    """Pooled statistics of the native extractor against the reference's own layer outputs."""
    g = golden("xvector")
    m, _ = _model(80, 102, "far")
    feats = onn.synthetic_feats(2, 50, 80, 102 + 2000)
    fused_emb = m.extract_embedding_batch(feats).cpu().numpy()
    fused_stats = m.extractor().debug_f32(-1, (2, 3000)).cpu().numpy()       # pooled in tdnn5's epilogue
    assert rel(fused_stats, g["xv80_inter_stats"][:, :, 0]) < EMB_TOL
    m.extractor().set_fused_pooling(False)                                   # fp32 tensor + standalone pooling kernel
    emb = m.extract_embedding_batch(feats).cpu().numpy()
    stats = m.extractor().debug_f32(-1, (2, 3000)).cpu().numpy()
    assert rel(stats, g["xv80_inter_stats"][:, :, 0]) < EMB_TOL
    last = m.extractor().debug_f32(0, (2, 50, 1500)).cpu().numpy()
    assert rel(last.transpose(0, 2, 1)[:, :8], g["xv80_inter_tdnn5"]) < EMB_TOL
    assert rel(fused_stats, stats) < 2e-6 and rel(fused_emb, emb) < 2e-6


@pytest.mark.parametrize("B,T", [(3, 200), (2, 1), (5, 37), (1, 300), (40, 8)])
def test_fused_pooling_layer_vs_oracle(ops, B, T):
    """tdnn5-shaped layer with the pooling fused into the epilogue (ragged T, Tb in {1,4,8,32})."""
    x, w, b, scale, shift = _layer_inputs(B, T, 512, 1500, [0], 17)
    xp = ops.split_f32(torch.from_numpy(x).cuda())
    wp = ops.pack_tdnn_weight(torch.from_numpy(w).cuda(), [0])
    out = ops.fused_pool_layer(xp, wp, 1500, [0], torch.from_numpy(b).cuda(), torch.from_numpy(scale).cuda(),
                               torch.from_numpy(shift).cuda(), relu=True).cpu().numpy()
    y = _oracle_layer(x, w, b, scale, shift, [0], True)
    with torch.no_grad():
        ref = onn.statistics_pooling(torch.from_numpy(y).transpose(1, 2)).squeeze(2).numpy()
    assert rel(out[:, :1500], ref[:, :1500]) < GEMM_TOL
    assert rel(out[:, 1500:], ref[:, 1500:]) < 1e-4 if T > 1 else np.allclose(out[:, 1500:], 1e-5, rtol=1e-3)


@pytest.mark.parametrize("pos", ["far", "near"])
def test_extended_xvector_matches_reference_golden(golden, pos):
    from asv_subtools_b200.model.extended_xvector import ExtendedXvector
    g = golden("xvector")
    sd = onn.make_state_dict(onn.extended_xvector_spec(80), 103)
    m = ExtendedXvector(80, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    feats = onn.synthetic_feats(3, 150, 80, 1103)
    got = m.extract_embedding_batch(feats).cpu().numpy()
    for i in range(3):
        assert rel(got[i], g["ext80_{}_emb".format(pos)][i]) < EMB_TOL
        assert rel(m.extract_embedding(feats[i]).numpy(), g["ext80_{}_emb".format(pos)][i]) < EMB_TOL


def test_host_buffer_path_matches_device_path():
    m, _ = _model(80, 102, "far")
    feats = onn.synthetic_feats(8, 200, 80, 77)
    a = m.extract_embedding_batch(feats).cpu().numpy()
    b = m.extractor().extract_host(feats)
    assert np.array_equal(a, b)


def test_no_cpu_path():
    from asv_subtools_b200.model.xvector import Xvector
    m = Xvector(23, 10, training=False)
    with pytest.raises(RuntimeError):
        m.extract_embedding(np.zeros((10, 23), dtype=np.float32))
    m.cuda()
    with pytest.raises(TypeError):
        m.extract_embedding(np.zeros((10, 23), dtype=np.float64))


# ---------------------------------------------------------------- BASELINE-size properties
def test_full_size_batch_invariance_and_padding_properties():
    """At the BASELINE shape (256 x 200 x 80) the oracle is too slow to replay, so check
    size-independent properties: (i) an utterance's embedding does not depend on its batch
    neighbours or position (bit-exact: tiles only regroup rows, the K order is fixed);
    (ii) all-zero utterances give the bias-only embedding; (iii) sub-batches agree with the oracle."""
    m, sd = _model(80, 102, "far")
    feats = onn.synthetic_feats(256, 200, 80, 2024)
    feats[7] = 0
    feats[200] = 0
    full = m.extract_embedding_batch(feats).cpu().numpy()
    assert np.all(np.isfinite(full)) and full.shape == (256, 512)
    assert np.array_equal(full[7], full[200])
    perm = np.random.RandomState(0).permutation(256)
    assert np.array_equal(m.extract_embedding_batch(feats[perm]).cpu().numpy(), full[perm])
    assert np.array_equal(m.extract_embedding_batch(feats[:16]).cpu().numpy(), full[:16])
    # a different batch size changes the time blocking of the fused pooling (Chan merge order): ~1 ulp
    assert rel(m.extract_embedding_batch(feats[100:101]).cpu().numpy(), full[100:101]) < 2e-6
    assert rel(m.extract_embedding_batch(feats[:3]).cpu().numpy(), full[:3]) < 2e-6
    with torch.no_grad():
        ref = onn.xvector_forward(sd, torch.from_numpy(feats[[0, 7, 255]]).transpose(1, 2), "far").squeeze(2).numpy()
    for got, want in zip(full[[0, 7, 255]], ref):
        assert rel(got, want) < EMB_TOL


def test_pipelined_host_path_matches():
    m, _ = _model(80, 102, "far")
    ex = m.extractor()
    feats = [torch.from_numpy(onn.synthetic_feats(32, 200, 80, 50 + i)).pin_memory() for i in range(4)]
    outs = [torch.empty(32, 512).pin_memory() for _ in range(4)]
    ex.submit_host(feats[0].data_ptr(), 32, 200, outs[0].data_ptr(), 0)
    for i in range(1, 4):
        ex.submit_host(feats[i].data_ptr(), 32, 200, outs[i].data_ptr(), i % 2)
        ex.wait((i - 1) % 2)
    ex.wait(1)
    for f, o in zip(feats, outs):
        assert np.array_equal(o.numpy(), m.extract_embedding_batch(f.numpy()).cpu().numpy())
    from asv_subtools_b200 import _lib
    ex.submit_host(feats[0].data_ptr(), 32, 200, outs[0].data_ptr(), 0)
    with pytest.raises(_lib.XvbError):                      # slot still in flight
        ex.submit_host(feats[1].data_ptr(), 32, 200, outs[1].data_ptr(), 0)
    ex.wait(0)


def test_im2col_first_layer_and_split_k_are_equivalent_paths(ops, monkeypatch):
    """Two shape-driven fast paths of the extractor against their plain forms:
    (i) the first layer as an im2col view over time-padded planes (7 channel blocks instead of 10 for
        [-2..2] x 80) keeps the K order, so the embeddings are bit-identical;
    (ii) split-K of the segment layer (K = 3000) sums per-slice fp32 partials in a fixed order: equal within the
         rounding of the accumulation order (GEMM_TOL), and bit-reproducible from call to call."""
    feats = onn.synthetic_feats(24, 117, 80, 77)

    def run(im2col, splitk, pos="far"):
        monkeypatch.setenv("XVB_IM2COL", im2col)
        monkeypatch.setenv("XVB_SPLITK", splitk)
        m, _ = _model(80, 102, pos)
        out = m.extract_embedding_batch(feats).cpu().numpy()
        m.invalidate()
        return out

    base = run("0", "0")
    assert np.array_equal(run("1", "0"), base)
    for pos in ("far", "near"):
        a, b = run("1", "1", pos), run("0", "0", pos)
        assert rel(a, b) < GEMM_TOL, pos
        assert np.array_equal(a, run("1", "1", pos)), pos
    # ragged tails: T not a multiple of anything, B = 1
    monkeypatch.setenv("XVB_IM2COL", "1")
    monkeypatch.setenv("XVB_SPLITK", "1")
    m, sd = _model(80, 102, "far")
    for T in (1, 3, 7, 61):
        f = onn.synthetic_feats(1, T, 80, 500 + T)
        with torch.no_grad():
            want = onn.xvector_forward(sd, torch.from_numpy(f).transpose(1, 2), "far").squeeze(2).numpy()
        assert rel(m.extract_embedding_batch(f).cpu().numpy(), want) < EMB_TOL, T


def test_split_frames_pads_with_zero_frames(ops):
    import ctypes as C
    from asv_subtools_b200._lib import check, lib
    x = torch.randn(3, 5, 20, device="cuda")
    hi = torch.full((3, 9, 24), 7, dtype=torch.bfloat16, device="cuda")
    lo = torch.full((3, 9, 24), 7, dtype=torch.bfloat16, device="cuda")
    check(lib.xvb_split_frames(C.c_void_p(x.data_ptr()), 3, 5, 20, C.c_void_p(hi.data_ptr()), C.c_void_p(lo.data_ptr()), 24, 3, 1, None))
    back = hi.float() + lo.float()
    assert torch.equal(back[:, :3], torch.zeros(3, 3, 24, device="cuda")) and torch.equal(back[:, 8:], torch.zeros(3, 1, 24, device="cuda"))
    assert torch.equal(back[:, 3:8, 20:], torch.zeros(3, 5, 4, device="cuda"))
    assert (back[:, 3:8, :20] - x).abs().max() < 1e-5 * x.abs().max()


@pytest.mark.parametrize("cname,extend,seed", [("std", False, 301), ("ext", True, 302)])
def test_snowdar_xvector_matches_reference_golden(golden, cname, extend, seed):
    """model/snowdar_xvector.py (default BatchNorm affine=False; positions far / near_affine / near) against the
    reference blueprint's own outputs (tests/golden/make_golden_snowdar.py)."""
    from asv_subtools_b200.model.snowdar_xvector import Xvector
    g = golden("snowdar")
    sd = onn.make_state_dict(onn.snowdar_xvector_spec(40, extend=extend), seed)
    feats = onn.synthetic_feats(3, 120, 40, seed + 1000)
    for pos in ("far", "near_affine", "near"):
        m = Xvector(40, 10, extend=extend, training=False, extracted_embedding=pos)
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        emb = np.stack([m.extract_embedding(feats[i]).numpy() for i in range(3)])
        assert rel(emb, g["{}_{}".format(cname, pos)]) < EMB_TOL, pos
        assert rel(m.extract_embedding_batch(feats).cpu().numpy(), g["{}_{}".format(cname, pos)]) < EMB_TOL, pos
    with pytest.raises(NotImplementedError):
        Xvector(40, 10, SE=True)


def test_replicated_table_hooks_store_every_batch_into_every_copy():
    """xvb_extractor_set_gather + xvb_scatter_rows on ONE GPU (csrc/peer.cu; the multi-process NVLink form is
    tools/peer_table_check.py under torchrun): two table copies allocated with xvb_ipc_alloc, the shard call (device
    and host-buffer forms, two lanes, ragged tail batch) fills both at the rank's row offset and still returns its own
    rows; turning the hook off stops the stores."""
    import ctypes as C
    from asv_subtools_b200._lib import check, lib
    m, _ = _model(80, 102, "far")
    ex = m.extractor()
    n, t, d, row0, rows = 150, 61, 512, 40, 256
    feats = torch.from_numpy(onn.synthetic_feats(n, t, 80, 919)).cuda()
    want = ex.extract_shard(feats, 64).clone()
    ptrs = (C.c_void_p * 2)()
    for k in range(2):
        p = C.c_void_p()
        check(lib.xvb_ipc_alloc(C.byref(p), rows * d * 4), "xvb_ipc_alloc")
        ptrs[k] = p.value

    def view(k):
        holder = type("_B", (), {})()
        holder.__cuda_array_interface__ = {"shape": (rows, d), "typestr": "<f4", "data": (int(ptrs[k]), False), "version": 3, "strides": None}
        return torch.as_tensor(holder, device="cuda")
    tabs = [view(0), view(1)]
    handle = (C.c_uint8 * 64)()
    check(lib.xvb_ipc_export(C.c_void_p(ptrs[0]), handle), "xvb_ipc_export")       # exportable (opening needs a second process)
    try:
        ex.set_gather(ptrs, 2, row0, d)
        for tb in tabs:
            tb.fill_(-7.0)
        got = ex.extract_shard(feats, 64)
        torch.cuda.synchronize()
        assert torch.equal(got, want)
        for tb in tabs:
            assert torch.equal(tb[row0:row0 + n], want) and bool((tb[:row0] == -7.0).all()) and bool((tb[row0 + n:] == -7.0).all())
        host = torch.empty(n, t, 80, dtype=torch.float32, pin_memory=True)
        host.copy_(feats)
        out = torch.empty(n, d, dtype=torch.float32, pin_memory=True)
        tabs[1].fill_(-7.0)
        ex.extract_shard_host(host.data_ptr(), n, t, out.data_ptr(), 64)
        assert torch.equal(out, want.cpu()) and torch.equal(tabs[1][row0:row0 + n], want)
        ex.set_gather(None, 0, 0, 0)
        tabs[0].fill_(-7.0)
        ex.extract_shard(feats, 64)
        torch.cuda.synchronize()
        assert bool((tabs[0] == -7.0).all())
    finally:
        ex.set_gather(None, 0, 0, 0)
        torch.cuda.synchronize()
        del tabs
        for k in range(2):
            lib.xvb_ipc_free(C.c_void_p(ptrs[k]))


SNOWDAR_POOLING_CASES = {
    "attn1": ("attentive", {}, 311),
    "attn2": ("attentive", {"affine_layers": 2, "hidden_size": 64}, 312),
    "mha_share": ("multi-head", {"num_head": 4}, 313),
    "mha_full": ("multi-head", {"num_head": 4, "share": False, "affine_layers": 2}, 314),
    "mres": ("multi-resolution", {"num_head": 4, "temperature": True, "affine_layers": 2}, 315),
    "lde": ("lde", {"num_head": 12, "num_nodes": 200}, 316),                        # LDEPooling(200, c_num=12): 2400-d encoding
    "xi_mean": ("xi-postmean-softplus2", {"hidden_size": 64, "num_nodes": 200}, 319),  # xi-vector, posterior mean
    "xi_dist": ("xi-postdist-softplus2", {"hidden_size": 64, "num_nodes": 200}, 320),  # ... mean | spread
}


@pytest.mark.parametrize("cname", sorted(SNOWDAR_POOLING_CASES))
def test_snowdar_attention_poolings_match_reference_golden(golden, cname):
    """pooling = attentive / multi-head / multi-resolution of the snowdar blueprint (libs/nnet/pooling.py:214-587 behind
    snowdar_xvector.py:119-136) against the reference's own outputs: grouped attention affines, shared and per-channel
    alphas, head boundaries that are not multiples of four channels (1500 / 4 = 375), per-head temperature."""
    from asv_subtools_b200.model.snowdar_xvector import Xvector
    pooling, pp, seed = SNOWDAR_POOLING_CASES[cname]
    g = golden("snowdar")
    sd = onn.make_state_dict(onn.snowdar_xvector_spec(40, pooling=pooling, pooling_params=pp), seed)
    feats = onn.synthetic_feats(3, 120, 40, seed + 1000)
    for pos in ("far", "near"):
        m = Xvector(40, 10, training=False, extracted_embedding=pos, pooling=pooling, pooling_params=pp)
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        want = g["{}_{}".format(cname, pos)]
        assert rel(m.extract_embedding_batch(feats).cpu().numpy(), want) < EMB_TOL, (cname, pos)
        assert rel(m.extract_embedding(feats[1]).numpy(), want[1]) < EMB_TOL, (cname, pos)
    with pytest.raises(NotImplementedError):
        Xvector(40, 10, pooling="no-such-pooling")


def test_snowdar_bn_relu_order_and_weight_normalisation(golden):
    """tdnn_layer_params={"bn-relu": True} (affine -> BatchNorm -> ReLU, components.py:386-403; folded into weight and bias
    at hand-over) against the reference's own outputs, through the native extractor (statistics pooling) and through the
    op-by-op extractor (attentive pooling, against the oracle); TdnnAffine(norm_w=True) (components.py:139-140) layer
    against the oracle."""
    from asv_subtools_b200 import ops
    from asv_subtools_b200.model.snowdar_xvector import Xvector
    from asv_subtools_b200.nnet import ReluBatchNormTdnnLayer
    from asv_subtools_b200.nnet.components import TdnnAffine
    g = golden("snowdar")
    tlp = {"bn-relu": True, "bn_params": {"momentum": 0.5, "affine": True, "track_running_stats": True}}
    sd = onn.make_state_dict(onn.snowdar_xvector_spec(40, bn_affine=True), 317)
    feats = onn.synthetic_feats(3, 120, 40, 1317)
    for pos in ("far", "near_affine", "near"):
        m = Xvector(40, 10, training=False, extracted_embedding=pos, tdnn_layer_params=tlp)
        m.load_state_dict(sd, strict=True)
        m.cuda().eval()
        assert rel(m.extract_embedding_batch(feats).cpu().numpy(), g["bnrelu_{}".format(pos)]) < EMB_TOL, pos
    pp = {"affine_layers": 2, "hidden_size": 64}
    sd2 = onn.make_state_dict(onn.snowdar_xvector_spec(40, bn_affine=True, pooling="attentive", pooling_params=pp), 318)
    m = Xvector(40, 10, training=False, extracted_embedding="near", tdnn_layer_params=tlp, pooling="attentive", pooling_params=pp)
    m.load_state_dict(sd2, strict=True)
    m.cuda().eval()
    with torch.no_grad():
        ref = onn.snowdar_xvector_forward(sd2, torch.from_numpy(feats).transpose(1, 2), "near", pooling="attentive",
                                          pooling_params=pp, bn_relu=True).squeeze(2).numpy()
    assert rel(m.extract_embedding_batch(feats).cpu().numpy(), ref) < EMB_TOL
    # norm_w
    aff = TdnnAffine(48, 64, context=[-2, 0, 2], norm_w=True)
    torch.manual_seed(5)
    torch.nn.init.normal_(aff.weight, 0.0, 0.3)
    torch.nn.init.normal_(aff.bias, 0.0, 0.1)
    x = torch.randn(2, 48, 37)
    ref = onn.relu_bn_tdnn_layer(x, {"l.affine.weight": aff.weight.detach(), "l.affine.bias": aff.bias.detach()}, "l", [-2, 0, 2],
                                 relu=False, bn=False, norm_w=True).transpose(1, 2).numpy()
    w = ops.pack_tdnn_weight(aff.dense_weight().cuda().contiguous(), [-2, 0, 2])
    xin = ops.split_f32(x.transpose(1, 2).contiguous().cuda())
    _, y = ops.tdnn_affine(xin, w, 64, [-2, 0, 2], bias=aff.bias.detach().cuda(), out_planes=False, out_f32=True)
    assert rel(y.cpu().numpy(), ref) < 3e-5
    with pytest.raises(NotImplementedError):
        TdnnAffine(48, 64, norm_f=True)
    assert isinstance(ReluBatchNormTdnnLayer(8, 8, **tlp).export()[2], type(None))


@pytest.mark.parametrize("B,T,C,K", [(3, 77, 200, 12), (2, 130, 64, 64), (1, 5, 24, 1), (2, 33, 20, 7)])
def test_lde_pool_kernels_vs_oracle(B, T, C, K):
    """xvb_lde_pool against oracle.lde_pooling (LDEPooling.forward, pooling.py:148-159): cluster counts that do and do not
    fill the eight thread groups, more than one 64-frame staging chunk, a strided input view."""
    from asv_subtools_b200 import ops
    rng = np.random.RandomState(C + K)
    x = (rng.standard_normal((B, T, C)) * 0.6).astype(np.float32)
    mu = (rng.standard_normal((C, K)) * 0.6).astype(np.float32)
    s = rng.uniform(0.05, 0.3, K).astype(np.float32)
    xw = torch.zeros(B, T, C + 4, device="cuda")
    xw[..., :C] = torch.from_numpy(x).cuda()
    neg_beta = torch.from_numpy(-(s ** 2 + np.float32(1e-10))).cuda()
    got, planes = ops.lde_pool(xw[..., :C], torch.from_numpy(mu).cuda(), neg_beta, planes=True)
    ref = onn.lde_pooling(torch.from_numpy(x).transpose(1, 2), torch.from_numpy(mu), torch.from_numpy(s)).squeeze(2).numpy()
    assert got.shape == ref.shape and rel(got.cpu().numpy(), ref) < 5e-6
    assert rel(planes.float().view(B, -1)[:, :C * K].cpu().numpy(), ref) < 2e-5


@pytest.mark.parametrize("heads,gdiv_kind,global_heads,unweighted", [(1, "share", False, False), (4, "share", False, True),
                                                                     (4, "full", False, False), (3, "share", True, False),
                                                                     (2, "full", True, False)])
def test_attn_head_stats_pool_kernel_vs_oracle(heads, gdiv_kind, global_heads, unweighted):
    """xvb_attn_head_stats_pool against oracle.attention_pooling for every head map, both std branches (the reference's
    `stddev_attention=False` branch only type-checks for split heads, pooling.py:432-434 vs :507-509), strided inputs."""
    from asv_subtools_b200 import ops
    rng = np.random.RandomState(11)
    B, T, C = 3, 77, 24 * heads if not global_heads else 20
    x = rng.standard_normal((B, T, C)).astype(np.float32) * 1.5 + 0.3
    pooled = C * heads if global_heads else C
    G = heads if gdiv_kind == "share" else pooled
    logits = rng.standard_normal((B, T, G)).astype(np.float32) * 2.0
    gdiv = 1 if gdiv_kind == "full" else (C if global_heads else C // heads)
    xw = torch.zeros(B, T, C + 4, device="cuda")
    xw[..., :C] = torch.from_numpy(x).cuda()
    lw = torch.zeros(B, T, (G + 7) // 8 * 8, device="cuda")
    lw[..., :G] = torch.from_numpy(logits).cuda()
    got, planes = ops.attn_head_stats_pool(lw[..., :G], xw[..., :C], pooled, gdiv, unweighted_var=unweighted, planes=True)
    alpha = torch.softmax(torch.from_numpy(logits).transpose(1, 2), dim=2)              # (B, G, T)
    ref = onn.attention_pooling(torch.from_numpy(x).transpose(1, 2), alpha, heads, global_heads,
                                stddev_attention=not unweighted).squeeze(2).numpy()
    assert got.shape == ref.shape and rel(got.cpu().numpy(), ref) < 2e-6
    assert rel(planes.float().view(B, -1).cpu().numpy(), ref) < 1e-5


@pytest.mark.parametrize("pos", ["far", "near"])
def test_factored_xvector_matches_reference_golden(golden, pos):
    """model/factored_xvector.py (F-TDNN blocks, skip concatenations, bypass) against the reference blueprint's own
    outputs (tests/golden/make_golden_ftdnn.py); ragged lengths against the oracle."""
    from asv_subtools_b200.model.factored_xvector import Xvector
    g = golden("ftdnn")
    sd = onn.make_state_dict(onn.factored_xvector_spec(40), 401)
    feats = onn.synthetic_feats(2, 90, 40, 1401)
    m = Xvector(40, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    emb = np.stack([m.extract_embedding(feats[i]).numpy() for i in range(2)])
    assert rel(emb, g[pos]) < EMB_TOL
    assert rel(m.extract_embedding_batch(feats).cpu().numpy(), g[pos]) < EMB_TOL
    for T in (1, 5, 33):
        f = onn.synthetic_feats(3, T, 40, 1500 + T)
        with torch.no_grad():
            want = onn.factored_xvector_forward(sd, torch.from_numpy(f).transpose(1, 2), pos).squeeze(2).numpy()
        assert rel(m.extract_embedding_batch(f).cpu().numpy(), want) < EMB_TOL, T


@pytest.mark.gpu
@pytest.mark.parametrize("pos", ["far", "near"])
def test_shard_calls_and_cached_launch_plans_equal_per_batch_extraction(pos):
    """xvb_extractor_extract_shard[_host] (the reference's caller loop, extract_embeddings.py:73-83, as one call) and
    the per-(B, T) launch-plan cache: a shard in ragged batches, the same shard through pinned host buffers, and batch
    shapes revisited in a different order all reproduce independent per-batch calls bit for bit ("far": split-K last
    layer, reduce kernel redirected; "near": the last layer's output map re-encoded per destination)."""
    m, _ = _model(80, 102, pos)
    ex = m.extractor()
    n, t = 150, 61
    feats = torch.from_numpy(onn.synthetic_feats(n, t, 80, 909)).cuda()
    want = torch.cat([ex.extract(feats[i:i + 64]).clone() for i in range(0, n, 64)])      # batches of 64, 64, 22
    got = ex.extract_shard(feats, 64)
    assert torch.equal(got, want)
    assert ex.last_launches >= 3 * 8
    other = torch.from_numpy(onn.synthetic_feats(5, 33, 80, 910)).cuda()                  # another shape in between
    w_other = ex.extract(other).clone()
    assert torch.equal(ex.extract_shard(feats, 64), want) and torch.equal(ex.extract(other), w_other)
    m2, _ = _model(80, 102, pos)                                                            # cold extractor, no cached plans
    assert torch.equal(m2.extractor().extract(other), w_other)
    host = torch.empty(n, t, 80, dtype=torch.float32, pin_memory=True)
    host.copy_(feats)
    out = torch.empty(n, ex.embed_dim, dtype=torch.float32, pin_memory=True)
    ex.extract_shard_host(host.data_ptr(), n, t, out.data_ptr(), 64)
    assert torch.equal(out, want.cpu())
    ex.set_profiling(True)                                                                 # events of every batch are kept
    ex.extract_shard(feats, 64)
    times = ex.kernel_times_ms(max_n=256)
    ex.set_profiling(False)
    per_batch = len(times) // 3 + 1
    assert len(times) == 3 * per_batch - 1 and all(x >= 0 for x in times)
