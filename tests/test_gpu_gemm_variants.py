"""Every layer instantiation of the tcgen05 GEMM (csrc/tdnn_gemm.cu: tdnn_gemm_bf16x3_kernel<BLOCK_N, kCta, kNSub, kPool,
kHist, kMask>) against a float64 reference, at shapes that select it.

The host picks the instantiation from m_tiles x ceil(Cout / BLOCK_N) against the SM count, so a small test shape and a
production shape run different code for the same layer.  Each case below names the instantiation it is meant to reach;
torch.profiler reports which kernel really ran, and the test asserts the two agree (on a 148-SM B200).  The paths only
the tuning knobs reach (XVB_GEMM_CTA / WIDE / BN / STORE / BOX64, read once per process) run in subprocesses through
tests/gemm_variant_worker.py.  The trial-histogram instantiation (kHist) is covered by test_trial_histogram.py.

Every output element is checked against an elementwise error bound derived from the arithmetic (see `reference`), not
against a tolerance on the largest value, so a wrong tile of small-magnitude rows cannot hide behind large ones.  The
checker itself is tested on the CPU (test_checker_rejects_defective_outputs)."""
import hashlib
import json
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "gemm_variant_worker.py")
EMB_TOL = 1e-4      # embeddings, relative to the row's largest component (as test_gpu_kernels.py)
SM_COUNT = 148      # the dispatch thresholds in the cases' expected instantiations assume a B200

# ---------------------------------------------------------------- (a) float64 reference and error bound
U24 = 2.0 ** -24    # fp32 unit roundoff
U8 = 2.0 ** -8      # bf16 unit roundoff (8-bit significand, round to nearest: split_bf16, common.cuh)
# A (dropped lo*lo term).  hi = rn(v), lo = rn(v - hi): |lo| <= u8 (1 + u8) |v| and |v| <= |hi + lo| / (1 - u8^2), so
# |lo| <= u8 / (1 - u8) |v_eff| for both operands, and the one product the kernel leaves out is bounded per term by
# u8^2 / (1 - u8)^2 |x_eff| |w_eff|.
BOUND_A = U8 ** 2 / (1.0 - U8) ** 2
# C (fp32 accumulation).  Every bf16 x bf16 product is exact in fp32; the accumulator adds n = 3 K_eff of them (hi*hi,
# lo*hi, hi*lo per K element) and each addition rounds the running sum s_i by at most u |s_i|, u = 2^-24, or 2^-23 if
# the tensor core truncates.  The total is <= u sum_i |s_i|.  With independent signs (every input here is Gaussian)
# E|s_i| <= sqrt(i E[t^2]), and sum_{i<=n} sqrt(i) <= (2/3) n^1.5; relative to sum |t| = n E|t| that is
# (2/3) sqrt(n) sqrt(E t^2) / E|t|, and sqrt(E t^2) / E|t| = pi / 2 for a product of two Gaussians.  So the expected
# error is <= 2u (2/3)(pi/2) sqrt(3 K_eff) sum|t| = 3.63 sqrt(K_eff) 2^-24 sum|t|.  sum_i |s_i| / n^1.5 tends to the
# integral of |W_t| of a Brownian path, mean 0.53; over the ~1e8 elements of a case its largest value stays below
# 3.5 (variance of the integral of W is 1/3: P > 3.5 is e^-18), 6.6x the mean -> a factor 8.  The epilogue's bias
# add rounds once more (u |acc + bias|) and the split-K reduce adds <= 8 slices: both far inside that margin.
BOUND_C = 3.63 * 8
# R (relative to |ref|).  fp32 output: the BN fma and the output itself round (u each); tanhf is within 2 ulp, sigmoid
# 1 / (1 + expf(-x)) within 2 ulp of expf plus two roundings -> 2^-21 covers all.  Split-plane output: hi = rn(y),
# lo = rn(y - hi) leaves |y - hi - lo| <= u8^2 |y| = 2^-16 |y| on top.
BOUND_R_F32 = 2.0 ** -21
BOUND_R_PLANES = 2.0 ** -16 + 2.0 ** -21


def reference(x_eff, w_eff, context, bias=None, scale=None, shift=None, relu=False, act=None, utt_bias=None, x2_eff=None,
              lengths=None, planes=False):
    """float64 reference of one layer and its elementwise error bound.

    y = act(BN(ReLU(bias + utt_bias[b] + sum_src sum_tap x_src[b, t + ctx[tap]] . W[:, tap]))), frames outside [0, T)
    read as zeros (F.pad), rows t >= lengths[b] exactly zero.  x_eff, x2_eff: (B, T, Cin) float64 = hi + lo of the split
    planes the kernel reads; w_eff: (Cout, ntaps, Cin) float64 = hi + lo of the packed weight.  Returns (ref, bound),
    both (B, T, Cout) float64 on the inputs' device:
        bound = (A + C sqrt(K_eff) 2^-24) |scale| (|x_eff| (*) |W_eff| + |bias| + |utt_bias|) + R |ref|
    with K_eff = sources x taps x Cin; masked rows get bound 0 (they must be exact zeros)."""
    B, T, Cin = x_eff.shape
    cout = w_eff.shape[0]
    acc = torch.zeros(B, T, cout, dtype=torch.float64, device=x_eff.device)
    mag = torch.zeros_like(acc)
    srcs = [x_eff] + ([x2_eff] if x2_eff is not None else [])
    for xs in srcs:
        xa = xs.abs()
        for k, c in enumerate(context):
            t0, t1 = max(0, -c), min(T, T - c)
            if t1 <= t0:
                continue
            wk = w_eff[:, k, :].t()
            acc[:, t0:t1] += torch.matmul(xs[:, t0 + c:t1 + c], wk)
            mag[:, t0:t1] += torch.matmul(xa[:, t0 + c:t1 + c], wk.abs())
    if bias is not None:
        acc += bias
        mag += bias.abs()
    if utt_bias is not None:
        acc += utt_bias[:, None, :]
        mag += utt_bias.abs()[:, None, :]
    y = torch.relu(acc) if relu else acc
    if scale is not None:
        y = y * scale + shift
        mag = mag * scale.abs()
    if act == "tanh":
        y = torch.tanh(y)          # Lipschitz 1: the bound on the argument carries over
    elif act == "sigmoid":
        y = torch.sigmoid(y)       # Lipschitz 1/4
    k_eff = len(srcs) * len(context) * Cin
    bound = (BOUND_A + BOUND_C * math.sqrt(k_eff) * U24) * mag + (BOUND_R_PLANES if planes else BOUND_R_F32) * y.abs()
    if lengths is not None:
        keep = (torch.arange(T, device=x_eff.device)[None, :] < lengths.to(x_eff.device).long()[:, None])[..., None]
        y = torch.where(keep, y, torch.zeros_like(y))
        bound = torch.where(keep, bound, torch.zeros_like(bound))
    return y, bound


def bound_ratio(got, ref, bound):
    """Largest |got - ref| / bound over all elements; an element with bound 0 (a masked row) must equal ref exactly,
    a NaN counts as infinitely wrong.  Returns (ratio, index of the worst element)."""
    err = (got.to(torch.float64) - ref).abs()
    ratio = torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                        torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, math.inf), ratio)
    flat = int(torch.argmax(ratio.reshape(-1)))
    return float(ratio.reshape(-1)[flat]), np.unravel_index(flat, tuple(ratio.shape))


# ---------------------------------------------------------------- (b) the checker rejects subtly wrong outputs (CPU)
def _bf16_split(v):
    hi = v.to(torch.float32).to(torch.bfloat16)
    lo = (v.to(torch.float32) - hi.to(torch.float32)).to(torch.bfloat16)
    return hi.to(torch.float64), lo.to(torch.float64)


def test_checker_rejects_defective_outputs():
    """Defects a broken tile schedule, pipeline or epilogue would produce, built from the float64 reference itself; each
    must push error/bound above 1 while the correctly rounded outputs stay below it."""
    g = torch.Generator().manual_seed(3)
    B, T, Cin, Cout, ctx = 16, 48, 256, 160, [-2, 0, 2]
    Tb, Bb = 16, 8                                    # one 128-row M tile = 8 utterances x 16 frames
    scales = 10.0 ** (torch.rand(B, generator=g, dtype=torch.float64) * 4 - 2)
    x = torch.randn(B, T, Cin, generator=g, dtype=torch.float64) * scales[:, None, None]
    w = torch.randn(Cout, len(ctx), Cin, generator=g, dtype=torch.float64) * math.sqrt(2.0 / (Cin * len(ctx)))
    bias = 0.1 * torch.randn(Cout, generator=g, dtype=torch.float64)
    xh, xl = _bf16_split(x)
    wh, wl = _bf16_split(w)
    x_eff, w_eff = xh + xl, wh + wl
    ref, bound = reference(x_eff, w_eff, ctx, bias=bias)

    def ratio(got):
        return bound_ratio(got, ref, bound)[0]

    # correct outputs: the exact value rounded to fp32, and the same split into output planes
    assert ratio(ref.to(torch.float32).to(torch.float64)) <= 1.0
    ref_p, bound_p = reference(x_eff, w_eff, ctx, bias=bias, planes=True)
    yh, yl = _bf16_split(ref_p)
    assert bound_ratio(yh + yl, ref_p, bound_p)[0] <= 1.0

    tile = (slice(Bb, 2 * Bb), slice(Tb, 2 * Tb))    # utterances 8..15, frames 16..31
    defects = {}
    # bf16x2 arithmetic: hi*hi + lo*hi, the hi*lo cross term dropped
    defects["cross term dropped"] = reference(xh + xl, wh, ctx, bias=bias)[0]
    # one 64-channel K block of one tap missing in one tile
    got = ref.clone()
    part, _ = reference(x_eff[..., 64:128].contiguous(), w_eff[:, 1:2, 64:128].contiguous(), [ctx[1]])
    got[tile] -= part[tile]
    defects["K block missing in one tile"] = got
    # a tap offset wrong in one tile: tap -2 read at -1
    got = ref.clone()
    wrong, _ = reference(x_eff, w_eff, [-1, 0, 2], bias=bias)
    got[tile] = wrong[tile]
    defects["tap offset wrong in one tile"] = got
    # one tile holding another tile's values (a stale accumulator stage)
    got = ref.clone()
    got[Bb:2 * Bb, Tb:2 * Tb] = ref[Bb:2 * Bb, 0:Tb]
    defects["stale tile"] = got
    # N-tail columns zeroed (160 = 128 + 32)
    got = ref.clone()
    got[..., 128:] = 0
    defects["N tail zeroed"] = got
    for name, got in defects.items():
        assert ratio(got.to(torch.float32).to(torch.float64)) > 1.0, name
    # a masked row that is not exactly zero
    lengths = torch.randint(1, T + 1, (B,), generator=g, dtype=torch.int32)
    lengths[0] = T - 3
    ref_m, bound_m = reference(x_eff, w_eff, ctx, bias=bias, lengths=lengths)
    got = ref_m.to(torch.float32).to(torch.float64)
    assert bound_ratio(got, ref_m, bound_m)[0] <= 1.0
    got[0, T - 3, 5] = 1e-30
    assert bound_ratio(got, ref_m, bound_m)[0] == math.inf


# ---------------------------------------------------------------- (c, d) the cases
def _c(name, B, T, Cin, Cout, ctx, inst, out="planes", bias=True, bn=True, relu=True, act=None, utt_bias=False,
       x2=False, slice_=None, lengths=False, garbage=False, sub=3, seed=None):
    """inst: (BLOCK_N, kCta, kNSub) the default dispatch is expected to pick on 148 SMs; out: planes | f32 | both;
    slice_: (c0, width): write channels [c0, c0 + Cout) of a `width`-channel buffer; lengths: a ragged batch (kMask);
    garbage: non-zero input past each utterance's length; sub: re-run this many utterances (<= 3) as a batch of their
    own, small enough to select <32,1,1>."""
    return dict(name=name, B=B, T=T, Cin=Cin, Cout=Cout, ctx=ctx, inst=tuple(inst), out=out, bias=bias, bn=bn, relu=relu,
                act=act, utt_bias=utt_bias, x2=x2, slice_=slice_, lengths=lengths, garbage=garbage, sub=sub,
                seed=seed if seed is not None else (sum(map(ord, name)) * 7919) % 100003)


_BASE = [
    # up to 9 tiles per CTA: both TMEM accumulator stages, several phase flips; N tail 96 = 64 + 32; box64 store
    _c("n64_persistent", 384, 200, 512, 96, [-2, 0, 2], (64, 1, 1)),
    # CTA pairs with 128-wide tiles, 9 tiles per pair, N tail 192 = 128 + 64; fp32 only, no bias / BN / ReLU
    _c("n128_pairs_f32", 256, 300, 1024, 192, [0], (128, 2, 1), out="f32", bias=False, bn=False, relu=False),
    # odd M-block count (169): the last pair's second CTA has no rows; N tail 72; both outputs (32-column path);
    # per-utterance bias + tanh, as ECAPA's attention hidden layer
    _c("n128_odd_uttbias_tanh", 100, 200, 512, 200, [-3, 0, 3], (128, 2, 1), out="both", bn=False, relu=False,
       act="tanh", utt_bias=True),
    # the benchmark's tdnn2: 6 tiles per pair
    _c("n256_production", 256, 200, 512, 512, [-2, 0, 2], (256, 2, 1)),
    # odd M-block count (75); a second source (W.(x + x2)) written into a channel slice of a wider buffer (ECAPA)
    _c("n256_odd_x2_slice", 48, 200, 512, 512, [-3, 0, 3], (256, 2, 1), x2=True, slice_=(256, 1024)),
    # Tb = 32, 5 tiles per pair, N tail 220 in a 256 tile, Cout % 8 != 0; sigmoid
    _c("n256_tail_sigmoid", 61, 224, 512, 1500, [0], (256, 2, 1), bn=False, relu=False, act="sigmoid", sub=1),
    # 3 column tiles, the wide-tile shape with a last sub-block past Cout (XVB_GEMM_WIDE)
    _c("n256_cout768", 256, 200, 512, 768, [0], (256, 2, 1), out="both"),
    # split-K at the extractor's segment-layer batch sizes: 7 slices, reduce kernel epilogue; 1000 = 7 x 128 + 104
    _c("splitk_b256", 256, 1, 3000, 512, [0], (64, 1, 1), out="both"),
    _c("splitk_b1000", 1000, 1, 3000, 512, [0], (128, 2, 1), out="f32", relu=False),
]
CASES = {c["name"]: c for c in _BASE}
for _b in _BASE:
    if _b["T"] > 1:         # a T == 1 layer has one row per utterance: nothing to mask (split-K drops the lengths)
        _m = dict(_b, name=_b["name"] + "_len", lengths=True, garbage=_b["name"] == "n256_production")
        CASES[_m["name"]] = _m
# fused statistics pooling (kPool): checked through its per-block partials, see test_pool_partials_vs_float64
POOL_CASES = {
    "pool_tdnn5": dict(B=256, T=200, Cin=512, Cout=1500, lengths=False, seed=71),
    "pool_tdnn5_len": dict(B=256, T=200, Cin=512, Cout=1500, lengths=True, seed=72),
    "pool_tb32_len": dict(B=61, T=224, Cin=512, Cout=1500, lengths=True, seed=73),
}

BF16_FILL = 0x7FA5            # NaN bit patterns the outputs are pre-filled with
F32_FILL = 0x7FA5A5A5
_RE_INST = re.compile(r"tdnn_gemm_bf16x3_kernel<\s*(\d+),\s*(\d+),\s*(\d+),\s*(true|false),\s*(true|false),\s*(true|false)\s*>")


def _ops():
    from asv_subtools_b200 import ops
    assert torch.cuda.is_available(), "needs a CUDA device"
    return ops


def inst_name(inst):
    """(BLOCK_N, kCta, kNSub, kPool, kHist, kMask) -> '<256,2,1,kPool,kMask>'"""
    flags = [f for f, on in zip(("kPool", "kHist", "kMask"), inst[3:]) if on]
    return "<" + ",".join([str(v) for v in inst[:3]] + flags) + ">"


def observe_gemm(fn):
    """Run fn under torch.profiler (CUDA activity) and return the GEMM instantiations that ran, as
    (BLOCK_N, kCta, kNSub, kPool, kHist, kMask) tuples.  No kernel recorded at all is an error, not a skip."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    assert kernels, "torch.profiler recorded no CUDA kernel"
    found = []
    for k in kernels:
        m = _RE_INST.search(k)
        if m:
            found.append(tuple(int(v) for v in m.groups()[:3]) + tuple(v == "true" for v in m.groups()[3:]))
    assert found, "no tdnn_gemm_bf16x3_kernel among the recorded kernels: {}".format(sorted(set(kernels))[:8])
    return found


def _lengths_for(B, T, Tb, gen):
    """Lengths +-1 around multiples of the tile's frame count Tb, 1 and T, the rest random."""
    special = [1, T, T - 1]
    for k in (1, 2, 3, T // Tb - 1, T // Tb):
        special += [k * Tb - 1, k * Tb, k * Tb + 1]
    special = [v for v in special if 1 <= v <= T]
    lens = torch.randint(1, T + 1, (B,), generator=gen, dtype=torch.int32)
    lens[:len(special)] = torch.tensor(special[:B], dtype=torch.int32)
    return lens


def _tile_frames(B, T):
    import ctypes as C
    from asv_subtools_b200._lib import lib
    tb = C.c_int()
    nblk = lib.xvb_pool_partial_blocks(B, T, C.byref(tb))
    return nblk, tb.value


def _inputs(case):
    """Seeded inputs on the GPU: per-utterance scales 1e-2 .. 1e2, a packed weight and the epilogue parameters."""
    ops = _ops()
    B, T, Cin, Cout, ctx = case["B"], case["T"], case["Cin"], case["Cout"], case["ctx"]
    gen = torch.Generator().manual_seed(case["seed"])
    left, right, tot = ops.context_span(ctx)

    def randn(*shape):
        return torch.randn(*shape, generator=gen).cuda()

    scales = (10.0 ** (torch.rand(B, generator=gen) * 4 - 2)).cuda()
    d = dict(x=randn(B, T, Cin) * scales[:, None, None])
    d["x2"] = randn(B, T, Cin) * scales[:, None, None] if case["x2"] else None
    d["w"] = randn(Cout, Cin, tot) * math.sqrt(2.0 / (Cin * len(ctx)))
    d["bias"] = 0.1 * randn(Cout) if case["bias"] else None
    d["scale"] = (torch.rand(Cout, generator=gen) + 0.5).cuda() if case["bn"] else None
    d["shift"] = 0.1 * randn(Cout) if case["bn"] else None
    d["utt_bias"] = randn(B, Cout) * 0.3 if case["utt_bias"] else None
    d["lengths"] = None
    if case["lengths"]:
        _, tb = _tile_frames(B, T)
        d["lengths"] = _lengths_for(B, T, tb, gen).cuda()
        if not case["garbage"]:       # what the previous masked layer leaves: zeros past each length
            keep = torch.arange(T, device="cuda")[None, :] < d["lengths"].long()[:, None]
            d["x"] *= keep[..., None]
            if d["x2"] is not None:
                d["x2"] *= keep[..., None]
    return d


def _alloc_outputs(case, B):
    """Pre-filled (NaN bit pattern) output buffers with a row pitch larger than Cout, or a wider buffer for a slice."""
    Cout = case["Cout"]
    T = case["T"]
    c0, width = case["slice_"] or (0, Cout)
    ld = (width + 7) // 8 * 8 + 24
    bufs = {}
    if case["out"] in ("planes", "both"):
        bufs["hi"] = torch.full((B, T, ld), BF16_FILL, dtype=torch.int16, device="cuda").view(torch.bfloat16)
        bufs["lo"] = torch.full((B, T, ld), BF16_FILL, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    if case["out"] in ("f32", "both"):
        bufs["f32"] = torch.full((B, T, ld), F32_FILL, dtype=torch.int32, device="cuda").view(torch.float32)
    return bufs, c0


def _call(case, d, bufs, c0, rows=None):
    ops = _ops()
    Cout = case["Cout"]

    def pick(t):
        return None if t is None else (t if rows is None else t[rows].contiguous())

    xp = ops.split_f32(pick(d["x"]), ld=(case["Cin"] + 7) // 8 * 8 + 8)
    x2p = ops.split_f32(pick(d["x2"])) if d["x2"] is not None else None
    y = ops.SplitPlanes(bufs["hi"][..., c0:c0 + Cout], bufs["lo"][..., c0:c0 + Cout], Cout) if "hi" in bufs else None
    yf = bufs["f32"][..., c0:c0 + Cout] if "f32" in bufs else None

    def run():
        ops.tdnn_affine_ex(xp, d["wp"], Cout, case["ctx"], x2=x2p, bias=d["bias"], bn_scale=d["scale"], bn_shift=d["shift"],
                           utt_bias=pick(d["utt_bias"]), relu=case["relu"], tanh=case["act"] == "tanh",
                           sigmoid=case["act"] == "sigmoid", y=y, y_f32=yf, lengths=pick(d["lengths"]))
    return run, xp, x2p


def _eff(p, channels):
    return (p.hi.to(torch.float64) + p.lo.to(torch.float64))[..., :channels]


def _bits(bufs):
    return {k: v.view(torch.int16 if v.dtype == torch.bfloat16 else torch.int32) for k, v in bufs.items()}


def digest(bufs):
    h = hashlib.sha256()
    for k in sorted(bufs):
        h.update(k.encode())
        h.update(_bits(bufs)[k].cpu().numpy().tobytes())
    return h.hexdigest()


def run_case(case, sub_batch=True, expect_default=True):
    """Run one layer case: observed instantiation, largest error/bound, sentinel / mask / repeat checks, a digest of the
    output bits and (sub_batch) bit-identity of a few utterances re-run on their own.  Returns a JSON-able dict;
    `failures` lists every check that did not hold.  expect_default: the instantiation must be the case's default one
    (off under a tiling knob: the caller checks what ran)."""
    ops = _ops()
    B, T, Cin, Cout, ctx = case["B"], case["T"], case["Cin"], case["Cout"], case["ctx"]
    d = _inputs(case)
    d["wp"] = ops.pack_tdnn_weight(d["w"], ctx)
    res = dict(name=case["name"], failures=[])
    bufs, c0 = _alloc_outputs(case, B)
    run, xp, x2p = _call(case, d, bufs, c0)
    insts = observe_gemm(run)
    res["observed"] = [list(i) for i in insts]
    want = tuple(case["inst"]) + (False, False, bool(case["lengths"]))
    res["expected"] = list(want)
    if expect_default and torch.cuda.get_device_properties(0).multi_processor_count == SM_COUNT and set(insts) != {want}:
        res["failures"].append("ran {} instead of {}".format([inst_name(i) for i in insts], inst_name(want)))
    torch.cuda.synchronize()

    # values against float64
    ntaps = len(ctx)
    w_eff = (d["wp"].hi.to(torch.float64) + d["wp"].lo.to(torch.float64)).view(Cout, ntaps, -1)[:, :, :Cin]
    f64 = (lambda t: None if t is None else t.to(torch.float64))
    ratios = {}
    for form in [f for f, k in (("planes", "hi"), ("f32", "f32")) if k in bufs]:
        ref, bound = reference(_eff(xp, Cin), w_eff, ctx, f64(d["bias"]), f64(d["scale"]), f64(d["shift"]), case["relu"],
                               case["act"], f64(d["utt_bias"]), _eff(x2p, Cin) if x2p is not None else None, d["lengths"],
                               planes=form == "planes")
        if form == "planes":
            got = bufs["hi"][..., c0:c0 + Cout].to(torch.float64) + bufs["lo"][..., c0:c0 + Cout].to(torch.float64)
        else:
            got = bufs["f32"][..., c0:c0 + Cout].to(torch.float64)
        r, idx = bound_ratio(got, ref, bound)
        ratios[form] = r
        if not r <= 1.0:
            res["failures"].append("{}: max error/bound {:.3g} at {} (got {!r}, ref {!r}, bound {:.3g})".format(
                form, r, tuple(int(i) for i in idx), float(got[idx]), float(ref[idx]), float(bound[idx])))
        del ref, bound, got
    res["ratio"] = max(ratios.values())
    res["ratios"] = ratios

    # sentinels outside the written channels, exact (+0) zeros in masked rows.  A row's last 16-byte group is stored
    # whole: its columns past Cout must hold +0 (the pad split_f32 leaves), everything beyond it the sentinel.
    bits = _bits(bufs)
    for k, v in bits.items():
        fill = BF16_FILL if k != "f32" else F32_FILL
        group = 8 if k != "f32" else 4
        pad = slice(c0 + Cout, c0 + (Cout + group - 1) // group * group)
        if not bool((v[..., pad] == 0).all()):
            res["failures"].append("{}: columns [{}, {}) of the last 16-byte group are not +0.0".format(k, pad.start, pad.stop))
        outside = torch.ones(v.shape[-1], dtype=torch.bool, device="cuda")
        outside[c0:pad.stop] = False
        bad = (v[..., outside] != fill).nonzero()
        if len(bad):
            cols = torch.nonzero(outside).view(-1)[bad[:, -1]].unique().tolist()
            res["failures"].append("{}: columns {} outside [{}, {}) were written".format(k, cols[:16], c0, c0 + Cout))
        if d["lengths"] is not None:
            masked = torch.arange(T, device="cuda")[None, :] >= d["lengths"].long()[:, None]
            if not bool((v[..., c0:c0 + Cout][masked] == 0).all()):
                res["failures"].append("{}: a row t >= lengths[b] is not +0.0".format(k))
    # two identical calls, identical bits
    res["digest"] = digest(bufs)
    again, _ = _alloc_outputs(case, B)
    _call(case, d, again, c0)[0]()
    torch.cuda.synchronize()
    if digest(again) != res["digest"]:
        res["failures"].append("a second identical call gave different bits")
    del again

    # a few utterances on their own select <32,1,1>; tiles only regroup rows, so the bits must not change
    if sub_batch and case["sub"]:
        rows = torch.tensor([0, B // 2, B - 1][-case["sub"]:], device="cuda")
        sb, _ = _alloc_outputs(case, len(rows))
        run_sub = _call(case, d, sb, c0, rows=rows)[0]
        sub_insts = observe_gemm(run_sub)
        res["sub_observed"] = [list(i) for i in sub_insts]
        sub_want = (32, 1, 1, False, False, bool(case["lengths"]))
        if torch.cuda.get_device_properties(0).multi_processor_count == SM_COUNT and set(sub_insts) != {sub_want}:
            res["failures"].append("sub-batch ran {} instead of {}".format([inst_name(i) for i in sub_insts],
                                                                           inst_name(sub_want)))
        full = _bits(bufs)
        for k, v in _bits(sb).items():
            if not torch.equal(v, full[k][rows]):
                res["failures"].append("{}: utterances re-run as a batch of 3 differ in bits from the full batch".format(k))
    torch.cuda.synchronize()
    return res


# ---------------------------------------------------------------- results shared by the tests of this module
_RESULTS = {}


def case_result(name):
    if name not in _RESULTS:
        _RESULTS[name] = run_case(CASES[name])
    return _RESULTS[name]


def _report(res):
    return "{}: observed {}, max error/bound {:.3g}".format(res["name"], [inst_name(i) for i in res["observed"]], res["ratio"])


def _require_148():
    n = torch.cuda.get_device_properties(0).multi_processor_count
    if n != SM_COUNT:
        pytest.skip("values checked; the expected instantiations assume {} SMs, this device has {}".format(SM_COUNT, n))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_gemm_variant_vs_float64(name):
    res = case_result(name)
    print(_report(res))
    assert not res["failures"], (_report(res), res["failures"])
    _require_148()


# ---------------------------------------------------------------- (e) kPool partials, without the finalize step
def run_pool_case(name):
    ops = _ops()
    pc = POOL_CASES[name]
    case = _c(name, pc["B"], pc["T"], pc["Cin"], pc["Cout"], [0], (256, 2, 1), lengths=pc["lengths"], seed=pc["seed"])
    B, T, Cin, Cout = case["B"], case["T"], case["Cin"], case["Cout"]
    d = _inputs(case)
    wp = ops.pack_tdnn_weight(d["w"], [0])
    nblk, tb = _tile_frames(B, T)
    partial = torch.full((nblk, B, 2 * Cout), F32_FILL, dtype=torch.int32, device="cuda").view(torch.float32)
    xp = ops.split_f32(d["x"])
    insts = observe_gemm(lambda: ops.tdnn_affine_ex(xp, wp, Cout, [0], bias=d["bias"], bn_scale=d["scale"],
                                                    bn_shift=d["shift"], relu=True, pool_partial=partial,
                                                    lengths=d["lengths"]))
    want = (256, 2, 1, True, False, bool(pc["lengths"]))
    res = dict(name=name, observed=[list(i) for i in insts], expected=list(want), failures=[])
    if set(insts) != {want}:      # kPool is chosen by the call, not by the shape: independent of the SM count
        res["failures"].append("ran {} instead of {}".format([inst_name(i) for i in insts], inst_name(want)))
    w_eff = (wp.hi.to(torch.float64) + wp.lo.to(torch.float64)).view(Cout, 1, -1)[:, :, :Cin]
    y, beta = reference(_eff(xp, Cin), w_eff, [0], d["bias"].double(), d["scale"].double(), d["shift"].double(), True)
    y = y.view(B, T, Cout)
    lens = d["lengths"].long() if d["lengths"] is not None else torch.full((B,), T, device="cuda", dtype=torch.long)
    # per block of tb frames: n valid frames; mean and M2 = sum (y - mean)^2 over them
    pad = nblk * tb - T
    yb = torch.nn.functional.pad(y, (0, 0, 0, pad)).view(B, nblk, tb, Cout)
    bb = torch.nn.functional.pad(beta, (0, 0, 0, pad)).view(B, nblk, tb, Cout)
    t = torch.arange(nblk * tb, device="cuda").view(nblk, tb)
    valid = (t[None] < lens[:, None, None]).to(torch.float64)[..., None]                 # (B, nblk, tb, 1)
    n = valid.sum(2)                                                                      # (B, nblk, 1)
    nz = n.clamp(min=1)
    mean = (yb * valid).sum(2) / nz
    dev = (yb - mean[:, :, None]) * valid
    m2 = (dev ** 2).sum(2)
    # bounds: each frame value is off by <= beta (the layer's bound, fp32 output); fp32 block sums over <= tb values
    # (two passes, Chan merges of 16-frame groups past 16) add <= (tb + 4) u relative roundings
    bmax = (bb * valid).amax(2)
    ymax = (yb.abs() * valid).amax(2)
    k = (tb + 4) * U24
    b_mean = (bb * valid).sum(2) / nz + k * (yb.abs() * valid).sum(2) / nz
    b_m2 = 4 * bmax * dev.abs().sum(2) + n * (2 * bmax + k * ymax) ** 2 + 2 * k * m2
    got = partial.view(nblk, B, 2, Cout).permute(1, 0, 2, 3).to(torch.float64)           # (B, nblk, 2, Cout)
    has = (n[..., 0] > 0)
    ratios = []
    for j, (want_v, bnd) in enumerate(((mean, b_mean), (m2, b_m2))):
        r, idx = bound_ratio(got[:, :, j][has], want_v[has], bnd[has])
        ratios.append(r)
        if not r <= 1.0:
            res["failures"].append("{}: max error/bound {:.3g}".format(("mean", "M2")[j], r))
    res["ratio"] = max(ratios)
    empty_bits = partial.view(torch.int32).view(nblk, B, 2 * Cout).permute(1, 0, 2)[~has]
    res["empty_blocks"] = int((~has).sum())
    if not bool((empty_bits == F32_FILL).all()):
        res["failures"].append("a block past ceil(L_b / Tb) was written")
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(POOL_CASES))
def test_pool_partials_vs_float64(name):
    if name not in _RESULTS:
        _RESULTS[name] = run_pool_case(name)
    res = _RESULTS[name]
    print(_report(res), "blocks left unwritten:", res["empty_blocks"])
    assert not res["failures"], (_report(res), res["failures"])
    if POOL_CASES[name]["lengths"]:
        assert res["empty_blocks"] > 0


# ---------------------------------------------------------------- (f) the whole x-vector at the benchmark batch
@pytest.mark.gpu
@pytest.mark.parametrize("pos", ["far", "near"])
def test_xvector_benchmark_batch_vs_float64_oracle(pos):
    """256 x 200 x 80 through the native extractor (tdnn2-4 on <256,2,1>, tdnn5 on the fused pooling), every row against
    the oracle evaluated in float64 on the GPU."""
    from asv_subtools_b200.model.xvector import Xvector
    from oracle import nnet as onn
    sd = onn.make_state_dict(onn.xvector_spec(80), 102)
    m = Xvector(80, 10, training=False, extracted_embedding=pos)
    m.load_state_dict(sd, strict=True)
    m.cuda().eval()
    feats = onn.synthetic_feats(256, 200, 80, 2024)
    got = m.extract_embedding_batch(feats).cpu().numpy().astype(np.float64)
    sd64 = {k: v.to("cuda", torch.float64) for k, v in sd.items()}
    with torch.no_grad(), torch.device("cuda"):       # the oracle builds its tap masks with torch.tensor
        ref = onn.xvector_forward(sd64, torch.from_numpy(feats).to("cuda", torch.float64).transpose(1, 2), pos)
    ref = ref.squeeze(2).cpu().numpy()
    errs = np.abs(got - ref).max(axis=1) / np.abs(ref).max(axis=1)
    print("{}: worst row {} rel err {:.3g}".format(pos, int(errs.argmax()), float(errs.max())))
    assert float(errs.max()) < EMB_TOL, (int(errs.argmax()), float(errs.max()))


# ---------------------------------------------------------------- 2. the knob-only paths, in subprocesses
# env -> (cases, the instantiation each one must select, or None for the default one).  Store-path knobs change only
# how values are stored; tiling knobs change which rows a CTA owns and the N width of its MMAs, not the K order.  So
# every knob run must reproduce the default run's bits.
KNOB_RUNS = {
    "cta1": ({"XVB_GEMM_CTA": "1"}, {"n256_production": (256, 1, 1), "n128_pairs_f32": (128, 1, 1),
                                     "n128_odd_uttbias_tanh": (128, 1, 1), "n256_production_len": (256, 1, 1),
                                     "n128_pairs_f32_len": (128, 1, 1), "splitk_b1000": (128, 1, 1)}),
    "wide": ({"XVB_GEMM_WIDE": "1"}, {"n256_production": (256, 2, 2), "n256_cout768": (256, 2, 2),
                                      "n256_tail_sigmoid": (256, 2, 2), "n256_production_len": (256, 2, 2),
                                      "n256_cout768_len": (256, 2, 2)}),
    "bn128": ({"XVB_GEMM_BN": "128"}, {"n256_production": (128, 2, 1), "n256_odd_x2_slice": (128, 2, 1),
                                       "n256_production_len": (128, 2, 1)}),
    "store_direct": ({"XVB_GEMM_STORE": "direct"}, {"n256_production": None, "n128_pairs_f32": None,
                                                     "n128_odd_uttbias_tanh": None, "n256_cout768": None,
                                                     "n256_production_len": None, "n128_odd_uttbias_tanh_len": None}),
    "store_reg": ({"XVB_GEMM_STORE": "reg"}, {"n256_production": None, "n128_pairs_f32": None,
                                               "n128_odd_uttbias_tanh": None, "n256_cout768": None,
                                               "n256_production_len": None, "n128_odd_uttbias_tanh_len": None}),
    "box64_off": ({"XVB_GEMM_BOX64": "0"}, {"n256_production": None, "n64_persistent": None,
                                            "n256_tail_sigmoid": None, "n256_production_len": None,
                                            "n64_persistent_len": None}),
}


def knob_result(knob, tmp_dir):
    key = "knob:" + knob
    if key not in _RESULTS:
        env_add, cases = KNOB_RUNS[knob]
        env = dict(os.environ, **env_add)
        out = os.path.join(str(tmp_dir), knob + ".json")
        run = subprocess.run([sys.executable, WORKER, "--out", out] + list(cases), env=env, cwd=ROOT,
                             capture_output=True, text=True, timeout=900)
        assert run.returncode == 0, run.stdout[-4000:] + run.stderr[-4000:]
        with open(out) as f:
            _RESULTS[key] = json.load(f)
    return _RESULTS[key]


@pytest.mark.gpu
@pytest.mark.parametrize("knob", list(KNOB_RUNS))
def test_knob_paths_in_subprocess(knob, tmp_path):
    env_add, cases = KNOB_RUNS[knob]
    results = knob_result(knob, tmp_path)
    assert sorted(results) == sorted(cases)
    problems = []
    for name, inst in cases.items():
        res = results[name]
        print("{} {}".format(knob, _report(res)))
        problems += ["{}: {}".format(name, f) for f in res["failures"]]
        want = tuple(inst if inst is not None else CASES[name]["inst"]) + (False, False, bool(CASES[name]["lengths"]))
        if torch.cuda.get_device_properties(0).multi_processor_count == SM_COUNT and \
                {tuple(i) for i in res["observed"]} != {want}:
            problems.append("{}: ran {} instead of {}".format(name, [inst_name(i) for i in res["observed"]], inst_name(want)))
        if res["digest"] != case_result(name)["digest"]:
            problems.append("{}: output bits differ from the default run".format(name))
    assert not problems, problems
    _require_148()


@pytest.mark.gpu
def test_every_layer_instantiation_ran_and_matched(tmp_path):
    """The union of what the cases above observed covers all 16 layer instantiations in the dispatch (17 are compiled;
    the 17th, kHist, belongs to test_trial_histogram.py), and every one of them passed its float64 check."""
    _require_148()
    seen = {}
    for name in CASES:
        res = case_result(name)
        for i in res["observed"] + res.get("sub_observed", []):
            seen.setdefault(tuple(i), []).append((name, not res["failures"]))
    for name in POOL_CASES:
        if name not in _RESULTS:
            _RESULTS[name] = run_pool_case(name)
        for i in _RESULTS[name]["observed"]:
            seen.setdefault(tuple(i), []).append((name, not _RESULTS[name]["failures"]))
    for knob in KNOB_RUNS:
        for name, res in knob_result(knob, tmp_path).items():
            for i in res["observed"]:
                seen.setdefault(tuple(i), []).append((knob + ":" + name, not res["failures"]))
    layer = {(n, c, s, p, False, m) for (n, c, s, p) in [(32, 1, 1, False), (64, 1, 1, False), (128, 1, 1, False),
                                                          (256, 1, 1, False), (128, 2, 1, False), (256, 2, 1, False),
                                                          (256, 2, 2, False), (256, 2, 1, True)] for m in (False, True)}
    assert len(layer) == 16
    missing = sorted(inst_name(i) for i in layer - set(seen))
    assert not missing, "never ran: {}".format(missing)
    unchecked = sorted(inst_name(i) for i in layer if not any(ok for _, ok in seen[i]))
    assert not unchecked, "ran but never passed: {}".format(unchecked)
    for i in sorted(layer):
        print(inst_name(i), sorted({n for n, _ in seen[i]}))
