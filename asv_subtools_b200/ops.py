"""Thin Python wrappers over the C ABI for torch CUDA tensors (device memory + streams are the
only things torch is used for).  Frame matrices are channel-contiguous ``(B, T, C)``."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import BN, RELU, SIGMOID, TANH, TdnnArgs, check, int_array, lib  # noqa: F401


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _req(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise TypeError("{} must be a contiguous CUDA tensor of dtype {}".format(name, dtype))
    return t


class SplitPlanes:
    """fp32 tensor stored as two bf16 planes hi = bf16(x), lo = bf16(x - hi); last dim padded to `ld`."""

    def __init__(self, hi, lo, channels):
        self.hi, self.lo, self.channels = hi, lo, channels

    @property
    def ld(self):
        """Row pitch in elements (a channel slice keeps the pitch of the tensor it was cut from)."""
        return self.hi.stride(-2) if self.hi.dim() >= 2 else self.hi.shape[-1]

    def float(self):
        return (self.hi.float() + self.lo.float())[..., :self.channels]

    def slice(self, c0, c1):
        """Channel slice [c0, c1) as a view (c0 must keep 16-byte alignment: c0 % 8 == 0)."""
        if c0 % 8:
            raise ValueError("channel slices must start at a multiple of 8")
        return SplitPlanes(self.hi[..., c0:c1], self.lo[..., c0:c1], c1 - c0)

    @staticmethod
    def empty(shape, device):
        return SplitPlanes(torch.empty(shape, dtype=torch.bfloat16, device=device),
                           torch.empty(shape, dtype=torch.bfloat16, device=device), shape[-1])


def split_f32(x, ld=None):
    """(rows..., C) fp32 -> SplitPlanes with row pitch ld (default round_up(C, 8))."""
    x = _req(x, torch.float32, "x")
    c = x.shape[-1]
    ld = ld or (c + 7) // 8 * 8
    rows = x.numel() // c
    hi = torch.empty(x.shape[:-1] + (ld,), dtype=torch.bfloat16, device=x.device)
    lo = torch.empty_like(hi)
    check(lib.xvb_split_f32(_ptr(x), rows, c, c, _ptr(hi), _ptr(lo), ld, _stream()), "xvb_split_f32")
    return SplitPlanes(hi, lo, c)


def context_span(context):
    """left/right/total context as TdnnAffine.__init__ (components.py:50-53)."""
    left = context[0] if context[0] < 0 else 0
    right = context[-1] if context[-1] > 0 else 0
    return left, right, right - left + 1


def pack_tdnn_weight(weight, context):
    """Reference weight (Cout, Cin, tot_context) fp32 CUDA -> packed K-major SplitPlanes."""
    weight = _req(weight, torch.float32, "weight")
    cout, cin, tot = weight.shape
    left, _, tot_expected = context_span(context)
    if tot != tot_expected:
        raise ValueError("weight kernel size {} does not match context {}".format(tot, context))
    n = lib.xvb_packed_weight_elems(cout, cin, len(context))
    hi = torch.empty(n, dtype=torch.bfloat16, device=weight.device)
    lo = torch.empty_like(hi)
    check(lib.xvb_pack_tdnn_weight(_ptr(weight), cout, cin, tot, left, int_array(context), len(context), _ptr(hi),
                                   _ptr(lo), _stream()), "xvb_pack_tdnn_weight")
    return SplitPlanes(hi.view(cout, -1), lo.view(cout, -1), cin)


def tdnn_affine(x, w, cout, context, bias=None, bn_scale=None, bn_shift=None, relu=False, out_planes=True,
                out_f32=False):
    """x: SplitPlanes (B, T, ld).  Returns (SplitPlanes | None, fp32 tensor | None)."""
    b, t, ldx = x.hi.shape
    flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0)
    dev = x.hi.device
    y = None
    yf = None
    if out_planes:
        y = SplitPlanes(torch.empty(b, t, cout, dtype=torch.bfloat16, device=dev),
                        torch.empty(b, t, cout, dtype=torch.bfloat16, device=dev), cout)
    if out_f32:
        yf = torch.empty(b, t, cout, dtype=torch.float32, device=dev)
    check(lib.xvb_tdnn_affine(_ptr(x.hi), _ptr(x.lo), ldx, _ptr(w.hi), _ptr(w.lo), _ptr(bias), _ptr(bn_scale),
                              _ptr(bn_shift), flags, int_array(context), len(context),
                              _ptr(y.hi) if y else None, _ptr(y.lo) if y else None, cout, _ptr(yf), cout,
                              b, t, x.channels, cout, _stream()), "xvb_tdnn_affine")
    return y, yf


def fused_pool_layer(x, w, cout, context, bias=None, bn_scale=None, bn_shift=None, relu=True, eps=1e-10, mode=0, planes=False):
    """TDNN layer whose epilogue pools over time (no (B,T,C) output) + the Chan merge: -> (B, 2*cout) fp32
    [, the same as SplitPlanes (B,1,2*cout) for a following segment-level GEMM]."""
    b, t = x.hi.shape[0], x.hi.shape[1]
    tb = C.c_int()
    nblk = lib.xvb_pool_partial_blocks(b, t, C.byref(tb))
    partial = torch.empty(nblk, b, 2 * cout, dtype=torch.float32, device=x.hi.device)
    tdnn_affine_ex(x, w, cout, context, bias=bias, bn_scale=bn_scale, bn_shift=bn_shift, relu=relu, pool_partial=partial)
    out = torch.empty(b, 2 * cout, dtype=torch.float32, device=x.hi.device)
    op = SplitPlanes.empty((b, 1, 2 * cout), x.hi.device) if planes else None
    check(lib.xvb_pool_finalize(_ptr(partial), nblk, tb.value, b, t, cout, eps, mode, _ptr(out),
                                op.hi.data_ptr() if op else None, op.lo.data_ptr() if op else None, 2 * cout if op else 0,
                                _stream()), "xvb_pool_finalize")
    return (out, op) if planes else out


def tdnn_affine_ex(x, w, cout, context, x2=None, bias=None, bn_scale=None, bn_shift=None, utt_bias=None, row_bias=None,
                   relu=False, tanh=False, sigmoid=False, y=None, y_f32=None, pool_partial=None, lengths=None):
    """Full form of the tcgen05 layer (xvb_tdnn_affine_ex).  x / x2: SplitPlanes (B,T,*) (views
    allowed); y: SplitPlanes to write (view allowed) and/or y_f32: fp32 (B,T,>=cout) tensor.  lengths: (B,) int32
    CUDA tensor of valid frames per utterance (ragged batch: rows t >= lengths[b] come out as exact zeros)."""
    b, t = x.hi.shape[0], x.hi.shape[1]
    a = TdnnArgs()
    a.x_hi, a.x_lo, a.ldx = x.hi.data_ptr(), x.lo.data_ptr(), x.ld
    if x2 is not None:
        a.x2_hi, a.x2_lo, a.ldx2 = x2.hi.data_ptr(), x2.lo.data_ptr(), x2.ld
    a.w_hi, a.w_lo = w.hi.data_ptr(), w.lo.data_ptr()
    keep = []
    for name, v in (("bias", bias), ("bn_scale", bn_scale), ("bn_shift", bn_shift), ("row_bias", row_bias)):
        if v is not None:
            setattr(a, name, _req(v, torch.float32, name).data_ptr())
    if utt_bias is not None:
        a.utt_bias, a.ld_utt_bias = _req(utt_bias, torch.float32, "utt_bias").data_ptr(), utt_bias.shape[-1]
    a.flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0) | (TANH if tanh else 0) | \
        (SIGMOID if sigmoid else 0)
    ctx = int_array(context)
    keep.append(ctx)
    a.context_host, a.ntaps = ctx, len(context)
    if y is not None:
        a.y_hi, a.y_lo, a.ldy = y.hi.data_ptr(), y.lo.data_ptr(), y.ld
    if y_f32 is not None:
        if y_f32.dtype != torch.float32 or not y_f32.is_cuda:
            raise TypeError("y_f32 must be a CUDA float32 tensor")
        a.y_f32, a.ldyf = y_f32.data_ptr(), y_f32.stride(-2)
    if pool_partial is not None:
        a.pool_partial = pool_partial.data_ptr()
    if lengths is not None:
        a.lengths = _req(lengths, torch.int32, "lengths").data_ptr()
    a.B, a.T, a.Cin, a.Cout = b, t, x.channels, cout
    check(lib.xvb_tdnn_affine_ex(C.byref(a), _stream()), "xvb_tdnn_affine_ex")


def plane_mean(x, planes=True):
    """Mean over T of SplitPlanes (B,T,C) -> (fp32 (B,C), SplitPlanes (B,1,C) | None)."""
    b, t, c = x.hi.shape[0], x.hi.shape[1], x.channels
    out = torch.empty(b, c, dtype=torch.float32, device=x.hi.device)
    op = SplitPlanes.empty((b, 1, c), x.hi.device) if planes else None
    check(lib.xvb_plane_mean(x.hi.data_ptr(), x.lo.data_ptr(), x.ld, b, t, c, _ptr(out),
                             op.hi.data_ptr() if op else None, op.lo.data_ptr() if op else None, c, _stream()),
          "xvb_plane_mean")
    return out, op


def res2net_block(x, w_hi, w_lo, bias, scale, shift, dilation, nscale, y):
    """One-kernel Res2Net block: x, y SplitPlanes (B,T,nscale*128); stacked packed weights/params."""
    b, t = x.hi.shape[0], x.hi.shape[1]
    check(lib.xvb_res2net_block(x.hi.data_ptr(), x.lo.data_ptr(), x.ld, _ptr(w_hi), _ptr(w_lo), _ptr(bias), _ptr(scale),
                                _ptr(shift), int(dilation), int(nscale), y.hi.data_ptr(), y.lo.data_ptr(), y.ld, b, t,
                                _stream()), "xvb_res2net_block")


def copy_planes(src, dst):
    """dst[...] = src[...] for two SplitPlanes views of equal shape (B,T,c), c % 8 == 0."""
    rows = src.hi.shape[0] * src.hi.shape[1]
    for s, d in ((src.hi, dst.hi), (src.lo, dst.lo)):
        check(lib.xvb_copy_rows(s.data_ptr(), s.stride(-2) * 2, d.data_ptr(), d.stride(-2) * 2, rows, src.channels * 2,
                                _stream()), "xvb_copy_rows")


def se_apply(z, xin, gate, out, nxt=None):
    """out = z * gate[b] + xin ; nxt = xin + out   (all SplitPlanes (B,T,C), views allowed)."""
    b, t, c = z.hi.shape[0], z.hi.shape[1], z.channels
    gate = _req(gate, torch.float32, "gate")
    check(lib.xvb_se_apply(z.hi.data_ptr(), z.lo.data_ptr(), z.ld, xin.hi.data_ptr(), xin.lo.data_ptr(), xin.ld,
                           _ptr(gate), out.hi.data_ptr(), out.lo.data_ptr(), out.ld,
                           nxt.hi.data_ptr() if nxt else None, nxt.lo.data_ptr() if nxt else None,
                           nxt.ld if nxt else 0, b, t, c, _stream()), "xvb_se_apply")


def stats_pool_ex(x, eps, mode, planes=False):
    """mode 0: StatisticsPooling; mode 1: ECAPA global context (unbiased var + eps)."""
    x = _req(x, torch.float32, "x")
    b, t, c = x.shape
    out = torch.empty(b, 2 * c, dtype=torch.float32, device=x.device)
    op = SplitPlanes.empty((b, 1, 2 * c), x.device) if planes else None
    check(lib.xvb_stats_pool_ex(_ptr(x), c, b, t, c, eps, mode, _ptr(out), op.hi.data_ptr() if op else None,
                                op.lo.data_ptr() if op else None, 2 * c, _stream()), "xvb_stats_pool_ex")
    return (out, op) if planes else out


def attn_stats_pool(logits, x, floor=1e-5, planes=False):
    """softmax over T of logits (B,T,C) -> weighted mean/std of x (B,T,C): (B,2C)."""
    logits = _req(logits, torch.float32, "logits")
    x = _req(x, torch.float32, "x")
    b, t, c = x.shape
    out = torch.empty(b, 2 * c, dtype=torch.float32, device=x.device)
    op = SplitPlanes.empty((b, 1, 2 * c), x.device) if planes else None
    check(lib.xvb_attn_stats_pool(_ptr(logits), c, _ptr(x), c, b, t, c, floor, _ptr(out),
                                  op.hi.data_ptr() if op else None, op.lo.data_ptr() if op else None, 2 * c, _stream()),
          "xvb_attn_stats_pool")
    return (out, op) if planes else out


def lde_pool(x, mu, neg_beta, planes=False):
    """LDE pooling (xvb_lde_pool): x (B,T,C) fp32 (row stride may exceed C), mu (C,K) fp32, neg_beta (K,) fp32
    -> (B, C*K) fp32 [, SplitPlanes (B,1,round_up(C*K,8))]."""
    if x.dtype != torch.float32 or not x.is_cuda or x.dim() != 3 or x.stride(-1) != 1 or x.stride(0) != x.shape[1] * x.stride(1):
        raise TypeError("x must be a (B,T,C) CUDA float32 tensor with contiguous rows")
    mu = _req(mu, torch.float32, "mu")
    neg_beta = _req(neg_beta, torch.float32, "neg_beta")
    b, t, c = x.shape
    k = mu.shape[1]
    out = torch.empty(b, c * k, dtype=torch.float32, device=x.device)
    w = torch.empty(b * t, k, dtype=torch.float32, device=x.device)
    op = None
    if planes:
        op = SplitPlanes.empty((b, 1, (c * k + 7) // 8 * 8), x.device)
        if op.ld != c * k:
            op.hi.zero_()
            op.lo.zero_()
            op.channels = c * k
    check(lib.xvb_lde_pool(_ptr(x), x.stride(-2), b, t, c, _ptr(mu), k, _ptr(neg_beta), _ptr(w), _ptr(out),
                           op.hi.data_ptr() if op else None, op.lo.data_ptr() if op else None, op.ld if op else 0, _stream()),
          "xvb_lde_pool")
    return (out, op) if planes else out


def small_affine(x, w, bias=None, bn_scale=None, bn_shift=None, relu=False, sigmoid=False, tanh=False, planes=False):
    """Segment-level fp32 affine on CUDA cores (xvb_small_affine): x (B, K) fp32, w (N, K) fp32 -> (B, N) fp32
    [, the same as SplitPlanes (B, 1, N)]."""
    x = _req(x, torch.float32, "x")
    w = _req(w, torch.float32, "w")
    b, k = x.shape
    n = w.shape[0]
    y = torch.empty(b, n, dtype=torch.float32, device=x.device)
    op = SplitPlanes.empty((b, 1, (n + 7) // 8 * 8), x.device) if planes else None
    flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0) | (TANH if tanh else 0) | (SIGMOID if sigmoid else 0)
    check(lib.xvb_small_affine(_ptr(x), k, _ptr(w), b, k, n, _ptr(bias), _ptr(bn_scale), _ptr(bn_shift), flags, _ptr(y), n,
                               op.hi.data_ptr() if op else None, op.lo.data_ptr() if op else None, op.ld if op else 0, _stream()),
          "xvb_small_affine")
    return (y, op) if planes else y


def attn_head_stats_pool(logits, x, out_channels, gdiv, floor=1e-10, unweighted_var=False, planes=False, prior_logit=None,
                         prior_x=None, softplus2log=False):
    """Attention pooling with a head map (xvb_attn_head_stats_pool): logits (B,T,G) fp32 (any row pitch >= G), x (B,T,C)
    fp32; output channel o pools x[..., o % C] with softmax_T(logits[..., o // gdiv]).  -> (B, 2*out_channels).
    prior_logit / prior_x (C,) + softplus2log: the xi-vector form (a prior element in the softmax, logits = 2 log softplus)."""
    for name, v in (("logits", logits), ("x", x)):       # channel-slice views of wider buffers are fine: rows stay contiguous
        if v.dtype != torch.float32 or not v.is_cuda or v.dim() != 3 or v.stride(-1) != 1 or v.stride(0) != v.shape[1] * v.stride(1):
            raise TypeError("{} must be a (B,T,*) CUDA float32 tensor with contiguous rows".format(name))
    b, t, c = x.shape
    g = logits.shape[-1]
    out = torch.empty(b, 2 * out_channels, dtype=torch.float32, device=x.device)
    op = SplitPlanes.empty((b, 1, 2 * out_channels), x.device) if planes else None
    check(lib.xvb_attn_head_stats_pool_prior(_ptr(logits), logits.stride(-2), g, _ptr(x), x.stride(-2), b, t, c, out_channels,
                                             int(gdiv), floor, 1 if unweighted_var else 0, _ptr(prior_logit), _ptr(prior_x),
                                             1 if softplus2log else 0, _ptr(out), op.hi.data_ptr() if op else None,
                                             op.lo.data_ptr() if op else None, 2 * out_channels, _stream()),
          "xvb_attn_head_stats_pool")
    return (out, op) if planes else out


def tdnn_affine_simt(x, weight, context, bias=None, bn_scale=None, bn_shift=None, relu=False):
    """fp32 CUDA-core cross-check: x (B,T,Cin) fp32, weight (Cout,Cin,tot) as in the reference."""
    x = _req(x, torch.float32, "x")
    weight = _req(weight, torch.float32, "weight")
    b, t, cin = x.shape
    cout, _, tot = weight.shape
    left, _, _ = context_span(context)
    flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0)
    y = torch.empty(b, t, cout, dtype=torch.float32, device=x.device)
    check(lib.xvb_tdnn_affine_simt(_ptr(x), cin, _ptr(weight), tot, left, _ptr(bias), _ptr(bn_scale), _ptr(bn_shift),
                                   flags, int_array(context), len(context), _ptr(y), cout, b, t, cin, cout, _stream()),
          "xvb_tdnn_affine_simt")
    return y


def stats_pool(x, eps=1e-10, planes=False):
    """x (B,T,C) fp32 -> (B,2C) fp32 [, SplitPlanes]  (pooling.py:58-67)."""
    x = _req(x, torch.float32, "x")
    b, t, c = x.shape
    out = torch.empty(b, 2 * c, dtype=torch.float32, device=x.device)
    hi = lo = None
    if planes:
        hi = torch.empty(b, 2 * c, dtype=torch.bfloat16, device=x.device)
        lo = torch.empty_like(hi)
    check(lib.xvb_stats_pool(_ptr(x), c, b, t, c, eps, _ptr(out), _ptr(hi), _ptr(lo), 2 * c, _stream()),
          "xvb_stats_pool")
    return (out, SplitPlanes(hi, lo, 2 * c)) if planes else out


# ------------------------------------------------------------------ scoring
def center_length_norm(x, mean=None):
    x = _req(x, torch.float32, "x")
    y = torch.empty_like(x)
    check(lib.xvb_center_length_norm(_ptr(x), _ptr(mean), _ptr(y), x.shape[0], x.shape[1], _stream()),
          "xvb_center_length_norm")
    return y


def column_mean(x):
    x = _req(x, torch.float32, "x")
    m = torch.empty(x.shape[1], dtype=torch.float32, device=x.device)
    check(lib.xvb_column_mean(_ptr(x), x.shape[0], x.shape[1], _ptr(m), _stream()), "xvb_column_mean")
    return m


def cosine_trials(enroll, test, trial_e, trial_t):
    enroll = _req(enroll, torch.float32, "enroll")
    test = _req(test, torch.float32, "test")
    trial_e = _req(trial_e, torch.int32, "trial_e")
    trial_t = _req(trial_t, torch.int32, "trial_t")
    s = torch.empty(trial_e.shape[0], dtype=torch.float32, device=enroll.device)
    check(lib.xvb_cosine_trials(_ptr(enroll), _ptr(test), enroll.shape[1], _ptr(trial_e), _ptr(trial_t),
                                trial_e.shape[0], _ptr(s), _stream()), "xvb_cosine_trials")
    return s


def speaker_mean(x, spk2rows):
    """x (N,D) fp32 CUDA; spk2rows: list of row-index lists (spk2utt order) -> ((S,D) means, num_utts)."""
    x = _req(x, torch.float32, "x")
    counts = np.array([len(r) for r in spk2rows], dtype=np.int32)
    offsets = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)).to(x.device)
    members = torch.from_numpy(np.concatenate([np.asarray(r, dtype=np.int32) for r in spk2rows])).to(x.device)
    out = torch.empty(len(spk2rows), x.shape[1], dtype=torch.float32, device=x.device)
    check(lib.xvb_speaker_mean(_ptr(x), x.shape[1], _ptr(offsets), _ptr(members), len(spk2rows), _ptr(out), _stream()),
          "xvb_speaker_mean")
    return out, counts


def topn_mean_std(S, top_n=0, ddof=1):
    """Per row of a cohort score matrix: mean / std of the top_n largest entries (0 = all); ddof = 1 is pandas'
    .std() (score/ScoreNormalization.py), ddof = 0 np.std (subtools2/egrecho/score/asnorm.py)."""
    S = _req(S, torch.float32, "S")
    m = torch.empty(S.shape[0], dtype=torch.float32, device=S.device)
    sd = torch.empty_like(m)
    check(lib.xvb_topn_mean_std_ddof(_ptr(S), S.shape[1], S.shape[0], S.shape[1], int(top_n), int(ddof), _ptr(m), _ptr(sd),
                                     _stream()), "xvb_topn_mean_std")
    return m, sd


def snorm_trials(scores, trial_e, trial_t, mean_e, std_e, mean_t, std_t):
    scores = _req(scores, torch.float32, "scores")
    out = torch.empty_like(scores)
    check(lib.xvb_snorm_trials(_ptr(scores), _ptr(_req(trial_e, torch.int32, "trial_e")),
                               _ptr(_req(trial_t, torch.int32, "trial_t")), scores.shape[0], _ptr(mean_e), _ptr(std_e),
                               _ptr(mean_t), _ptr(std_t), _ptr(out), _stream()), "xvb_snorm_trials")
    return out


def bilinear_trials(enroll, test, trial_e, trial_t, row_term=None, col_term=None):
    enroll = _req(enroll, torch.float32, "enroll")
    test = _req(test, torch.float32, "test")
    trial_e = _req(trial_e, torch.int32, "trial_e")
    trial_t = _req(trial_t, torch.int32, "trial_t")
    s = torch.empty(trial_e.shape[0], dtype=torch.float32, device=enroll.device)
    check(lib.xvb_bilinear_trials(_ptr(enroll), _ptr(test), enroll.shape[1], _ptr(trial_e), _ptr(trial_t),
                                  trial_e.shape[0], _ptr(row_term), _ptr(col_term), _ptr(s), _stream()),
          "xvb_bilinear_trials")
    return s


def project(x, m):
    """x (rows, D) . m^T with m (Dout, D) -> (rows, Dout)."""
    x = _req(x, torch.float32, "x")
    m = _req(m, torch.float32, "m")
    y = torch.empty(x.shape[0], m.shape[0], dtype=torch.float32, device=x.device)
    check(lib.xvb_project(_ptr(x), x.shape[0], x.shape[1], _ptr(m), m.shape[0], _ptr(y), _stream()), "xvb_project")
    return y


def cosine_matrix(enroll, test):
    enroll = _req(enroll, torch.float32, "enroll")
    test = _req(test, torch.float32, "test")
    s = torch.empty(enroll.shape[0], test.shape[0], dtype=torch.float32, device=enroll.device)
    check(lib.xvb_cosine_matrix(_ptr(enroll), enroll.shape[0], _ptr(test), test.shape[0], enroll.shape[1], _ptr(s),
                                test.shape[0], _stream()), "xvb_cosine_matrix")
    return s


def plda_terms(x, gamma, c):
    x = _req(x, torch.float32, "x")
    term = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
    check(lib.xvb_plda_terms(_ptr(x), x.shape[0], x.shape[1], _ptr(_req(gamma, torch.float32, "gamma")),
                             _ptr(_req(c, torch.float32, "c")), _ptr(term), _stream()), "xvb_plda_terms")
    return term


def plda_matrix(enroll, test, l2, row, col):
    enroll = _req(enroll, torch.float32, "enroll")
    test = _req(test, torch.float32, "test")
    s = torch.empty(enroll.shape[0], test.shape[0], dtype=torch.float32, device=enroll.device)
    check(lib.xvb_plda_matrix(_ptr(enroll), enroll.shape[0], _ptr(test), test.shape[0], enroll.shape[1],
                              _ptr(_req(l2, torch.float32, "l2")), _ptr(row), _ptr(col), _ptr(s), test.shape[0],
                              _stream()), "xvb_plda_matrix")
    return s


def topn_indices(S, top_n):
    """(rows, top_n) int32: cohort indices of every row's top_n scores, best first."""
    S = _req(S, torch.float32, "S")
    top_n = min(int(top_n), S.shape[1])   # groupby().head(top_n): a cohort smaller than top_n is used whole
    idx = torch.empty(S.shape[0], top_n, dtype=torch.int32, device=S.device)
    check(lib.xvb_topn_indices(_ptr(S), S.shape[1], S.shape[0], S.shape[1], int(top_n), _ptr(idx), _stream()), "xvb_topn_indices")
    return idx


def snorm_cross_trials(scores, trial_e, trial_t, enroll_cohort, test_cohort, top_enroll, top_test):
    scores = _req(scores, torch.float32, "scores")
    out = torch.empty_like(scores)
    check(lib.xvb_snorm_cross_trials(_ptr(scores), _ptr(_req(trial_e, torch.int32, "trial_e")), _ptr(_req(trial_t, torch.int32, "trial_t")),
                                     scores.shape[0], _ptr(_req(enroll_cohort, torch.float32, "enroll_cohort")), enroll_cohort.shape[1],
                                     _ptr(_req(test_cohort, torch.float32, "test_cohort")), test_cohort.shape[1],
                                     _ptr(_req(top_enroll, torch.int32, "top_enroll")), _ptr(_req(top_test, torch.int32, "top_test")),
                                     top_enroll.shape[1], _ptr(out), _stream()), "xvb_snorm_cross_trials")
    return out


def matmul_nt(a, b, row_bias=None, col_bias=None):
    """a (M,K) . b (N,K)^T + row_bias[i] + col_bias[j] -> (M,N) fp32 on the tcgen05 layer (N % 4 == 0)."""
    a = _req(a, torch.float32, "a")
    b = a if b is a else _req(b, torch.float32, "b")
    out = torch.empty(a.shape[0], b.shape[0], dtype=torch.float32, device=a.device)
    check(lib.xvb_matmul_nt(_ptr(a), a.shape[0], _ptr(b), b.shape[0], a.shape[1], _ptr(row_bias), _ptr(col_bias), _ptr(out),
                            b.shape[0], _stream()), "xvb_matmul_nt")
    return out


def center_rows_transposed(x, spk, means, sqrt_weight=None):
    """-> (D, N): column i = sqrt_weight[spk[i]] * (x[i] - means[spk[i]])."""
    x = _req(x, torch.float32, "x")
    spk = _req(spk, torch.int32, "spk")
    means = _req(means, torch.float32, "means")
    out = torch.empty(x.shape[1], x.shape[0], dtype=torch.float32, device=x.device)
    check(lib.xvb_center_rows_transposed(_ptr(x), _ptr(spk), _ptr(means), _ptr(sqrt_weight), x.shape[0], x.shape[1], _ptr(out),
                                         x.shape[0], _stream()), "xvb_center_rows_transposed")
    return out


def plda_em_rows(u, n, weight, psi):
    """-> (what_T, resid_T), both (D, S); see include/xvb200.h."""
    u = _req(u, torch.float32, "u")
    s, d = u.shape
    what = torch.empty(d, s, dtype=torch.float32, device=u.device)
    resid = torch.empty(d, s, dtype=torch.float32, device=u.device)
    check(lib.xvb_plda_em_rows(_ptr(u), _ptr(_req(n, torch.float32, "n")), _ptr(weight), _ptr(_req(psi, torch.float32, "psi")),
                               s, d, _ptr(what), _ptr(resid), s, _stream()), "xvb_plda_em_rows")
    return what, resid


def plda_normalize_rows(u, psi, num_examples=None, simple=False):
    """In place: u[r] *= sqrt(D / sum_d u_d^2 / (psi_d + 1/n_r))  (simple: sqrt(D) / ||u[r]||)."""
    u = _req(u, torch.float32, "u")
    check(lib.xvb_plda_normalize_rows(_ptr(u), _ptr(_req(psi, torch.float32, "psi")), _ptr(num_examples), u.shape[0], u.shape[1],
                                      int(bool(simple)), _stream()), "xvb_plda_normalize_rows")
    return u


def plda_llr_operands(u, psi, num_examples, side):
    """-> ((rows, 2D) operand, (rows,) term) of the Kaldi-style PLDA LLR; side 0 = enroll, 1 = test."""
    u = _req(u, torch.float32, "u")
    a = torch.empty(u.shape[0], 2 * u.shape[1], dtype=torch.float32, device=u.device)
    term = torch.empty(u.shape[0], dtype=torch.float32, device=u.device)
    check(lib.xvb_plda_llr_operands(_ptr(u), _ptr(_req(psi, torch.float32, "psi")), _ptr(num_examples), u.shape[0], u.shape[1],
                                    int(side), _ptr(a), _ptr(term), _stream()), "xvb_plda_llr_operands")
    return a, term


def trial_histogram(enroll, enroll_spk, test, test_spk, lo, hi, nbins=2048, row_term=None, col_term=None,
                    symmetric=False, unit_first=0, unit_stride=1, out=None):
    """(2, nbins) int64 histogram [nontarget | target] of enroll.test^T (+ terms) -- scores are never
    stored.  `out` is accumulated into when given."""
    enroll = _req(enroll, torch.float32, "enroll")
    test = enroll if test is enroll else _req(test, torch.float32, "test")
    enroll_spk = _req(enroll_spk, torch.int32, "enroll_spk")
    test_spk = enroll_spk if test_spk is enroll_spk else _req(test_spk, torch.int32, "test_spk")
    if enroll_spk.shape[0] != enroll.shape[0] or test_spk.shape[0] != test.shape[0] or enroll.shape[1] != test.shape[1]:
        raise ValueError("trial_histogram: shape mismatch")
    if out is None:
        out = torch.zeros(2, nbins, dtype=torch.int64, device=enroll.device)
    elif out.dtype != torch.int64 or tuple(out.shape) != (2, nbins) or not out.is_contiguous() or out.device != enroll.device:
        raise ValueError("trial_histogram: out must be a contiguous (2, nbins) int64 tensor on the embeddings' device")
    check(lib.xvb_trial_histogram(_ptr(enroll), enroll.shape[0], _ptr(enroll_spk), _ptr(test), test.shape[0],
                                  _ptr(test_spk), enroll.shape[1], _ptr(row_term), _ptr(col_term), int(bool(symmetric)),
                                  int(unit_first), int(unit_stride), float(lo), float(hi), int(nbins), _ptr(out),
                                  _stream()), "xvb_trial_histogram")
    return out


# ------------------------------------------------------------------ ragged batching policy (host only)
def ragged_plan(offsets, batch=256, max_frames=0):
    """xvb_ragged_plan: offsets (N+1,) -> (order (N,) int32, list of per-batch index arrays into order).  Stable sort by
    length, then batches of <= batch utterances with B * round_up(max L, 32) <= max_frames (<= 0: 262144)."""
    off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64))
    n = off.size - 1
    if off.ndim != 1 or n < 1:
        raise ValueError("ragged_plan: need (N+1,) offsets with N >= 1")
    order = np.empty(n, dtype=np.int32)
    first = np.empty(n + 1, dtype=np.int64)
    nb = C.c_int64()
    check(lib.xvb_ragged_plan(off.ctypes.data_as(C.c_void_p), n, int(batch), int(max_frames), order.ctypes.data_as(C.c_void_p),
                              first.ctypes.data_as(C.c_void_p), C.byref(nb)), "xvb_ragged_plan")
    first = first[:nb.value + 1]
    return order, [order[first[k]:first[k + 1]] for k in range(nb.value)]


# ------------------------------------------------------------------ whole-model extractor
class Extractor:
    """Owner of a native xvb_extractor_t (packed weights + workspace on the current device)."""

    def __init__(self, feat_dim):
        self._h = C.c_void_p()
        check(lib.xvb_extractor_create(C.byref(self._h), int(feat_dim)), "xvb_extractor_create")
        self.feat_dim = int(feat_dim)
        self._keep = []
        self._layers = []      # (kind, context, w, b, scale, shift, flags): what save() writes
        self._eps = None

    @staticmethod
    def _np(a):
        if a is None:
            return None, None
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
        return a, a.ctypes.data_as(C.c_void_p)

    def add_frame_layer(self, weight, bias, context, bn_scale=None, bn_shift=None, relu=True):
        w, wp = self._np(weight)
        b, bp = self._np(bias)
        s, sp = self._np(bn_scale)
        t, tp = self._np(bn_shift)
        flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0)
        check(lib.xvb_extractor_add_frame_layer(self._h, w.shape[0], int_array(context), len(context), wp, bp, sp, tp,
                                                flags), "xvb_extractor_add_frame_layer")
        self._layers.append(("frame", [int(c) for c in context], w, b, s, t, flags))

    def add_segment_layer(self, weight, bias, bn_scale=None, bn_shift=None, relu=False):
        w, wp = self._np(weight)
        b, bp = self._np(bias)
        s, sp = self._np(bn_scale)
        t, tp = self._np(bn_shift)
        flags = (RELU if relu else 0) | (BN if bn_scale is not None else 0)
        check(lib.xvb_extractor_add_segment_layer(self._h, w.shape[0], wp, bp, sp, tp, flags),
              "xvb_extractor_add_segment_layer")
        self._layers.append(("segment", [0], w, b, s, t, flags))

    def finalize(self, pooling_eps=1e-10):
        check(lib.xvb_extractor_finalize(self._h, pooling_eps), "xvb_extractor_finalize")
        self.embed_dim = lib.xvb_extractor_embed_dim(self._h)
        self._eps = float(pooling_eps)

    def save(self, path):
        """Write the layer list as an .xvbm file (csrc/model_file.cpp) for xvb_extractor_load /
        the Python-free `bin/xvb-extract`."""
        import struct
        if self._eps is None:
            raise RuntimeError("Extractor.save: finalize() first")
        frames = [l for l in self._layers if l[0] == "frame"]
        segs = [l for l in self._layers if l[0] == "segment"]
        with open(path, "wb") as f:
            f.write(b"XVBM0001" + struct.pack("<ifii", self.feat_dim, self._eps, len(frames), len(segs)))
            for _, ctx, w, b, s, t, flags in frames + segs:
                w3 = w.reshape(w.shape[0], w.shape[1], -1)
                f.write(struct.pack("<7i", w3.shape[0], w3.shape[1], len(ctx), w3.shape[2], flags, int(b is not None),
                                    int(s is not None)))
                f.write(struct.pack("<%di" % len(ctx), *ctx))
                f.write(np.ascontiguousarray(w3, dtype="<f4").tobytes())
                if b is not None:
                    f.write(np.ascontiguousarray(b, dtype="<f4").tobytes())
                if s is not None:
                    f.write(np.ascontiguousarray(s, dtype="<f4").tobytes() + np.ascontiguousarray(t, dtype="<f4").tobytes())

    @classmethod
    def load(cls, path):
        """An extractor straight from an .xvbm file (no Python-side layer objects)."""
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        check(lib.xvb_extractor_load(C.byref(self._h), str(path).encode()), "xvb_extractor_load")
        self.feat_dim = lib.xvb_extractor_feat_dim(str(path).encode())
        self.embed_dim = lib.xvb_extractor_embed_dim(self._h)
        self._keep, self._layers, self._eps = [], [], None
        return self

    def extract(self, feats):
        """feats (B,T,F) fp32 CUDA -> (B,D) fp32 CUDA, asynchronous on the current stream."""
        feats = _req(feats, torch.float32, "feats")
        b, t, f = feats.shape
        if f != self.feat_dim:
            raise ValueError("expected feature dim {}, got {}".format(self.feat_dim, f))
        emb = torch.empty(b, self.embed_dim, dtype=torch.float32, device=feats.device)
        check(lib.xvb_extractor_extract(self._h, _ptr(feats), b, t, _ptr(emb), _stream()), "xvb_extractor_extract")
        return emb

    def extract_host(self, feats_np):
        """feats (B,T,F) float32 host array -> (B,D) float32 host array (H2D + D2H inside the call)."""
        feats_np = np.ascontiguousarray(feats_np, dtype=np.float32)
        b, t, f = feats_np.shape
        if f != self.feat_dim:
            raise ValueError("expected feature dim {}, got {}".format(self.feat_dim, f))
        emb = np.empty((b, self.embed_dim), dtype=np.float32)
        check(lib.xvb_extractor_extract_host(self._h, feats_np.ctypes.data_as(C.c_void_p), b, t,
                                             emb.ctypes.data_as(C.c_void_p), _stream()), "xvb_extractor_extract_host")
        return emb

    def submit_host(self, feats_ptr, b, t, emb_ptr, slot):
        """Pipelined host path: queue batch `slot` (0/1); pair with wait(slot)."""
        check(lib.xvb_extractor_submit_host(self._h, C.c_void_p(feats_ptr), b, t, C.c_void_p(emb_ptr), slot, _stream()),
              "xvb_extractor_submit_host")

    def wait(self, slot):
        check(lib.xvb_extractor_wait(self._h, slot), "xvb_extractor_wait")

    def extract_shard(self, feats, batch=256, out=None):
        """feats (N,T,F) fp32 CUDA -> (N,D) fp32 CUDA: the whole shard in `batch`-utterance batches, one C call
        (extract_embeddings.py:73-83's loop), asynchronous on the current stream."""
        feats = _req(feats, torch.float32, "feats")
        n, t, f = feats.shape
        if f != self.feat_dim:
            raise ValueError("expected feature dim {}, got {}".format(self.feat_dim, f))
        emb = out if out is not None else torch.empty(n, self.embed_dim, dtype=torch.float32, device=feats.device)
        if out is not None:
            _req(out, torch.float32, "out")
            if tuple(out.shape) != (n, self.embed_dim):
                raise ValueError("out must be ({}, {})".format(n, self.embed_dim))
        check(lib.xvb_extractor_extract_shard(self._h, _ptr(feats), n, t, int(batch), _ptr(emb), _stream()),
              "xvb_extractor_extract_shard")
        return emb

    def extract_shard_host(self, feats_ptr, n, t, emb_ptr, batch=256):
        """Host-buffer shard call (pinned feats in, embeddings out, copies overlapped with the stack)."""
        check(lib.xvb_extractor_extract_shard_host(self._h, C.c_void_p(feats_ptr), int(n), int(t), int(batch),
                                                   C.c_void_p(emb_ptr), _stream()), "xvb_extractor_extract_shard_host")

    def set_gather(self, pointers, ntables, row0, ld):
        """Replicated-table form of the shard calls (parallel.PeerTable.attach): every batch's embeddings also go to
        `ntables` table copies at row0 + row; ntables = 0 turns it off."""
        check(lib.xvb_extractor_set_gather(self._h, pointers, int(ntables), int(row0), int(ld)), "xvb_extractor_set_gather")

    def extract_ragged(self, feats, offsets):
        """Ragged batch: feats (sum_T, F) fp32 CUDA, utterance b = rows offsets[b] .. offsets[b+1] (host ints, B+1)
        -> (B, D) fp32 CUDA, asynchronous on the current stream."""
        feats = _req(feats, torch.float32, "feats")
        if feats.dim() != 2 or feats.shape[1] != self.feat_dim:
            raise ValueError("expected (sum_T, {}) features, got {}".format(self.feat_dim, tuple(feats.shape)))
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64))
        if off.ndim != 1 or off.size < 2 or off[-1] > feats.shape[0] or off.max() > np.iinfo(np.int32).max:
            raise ValueError("offsets must be (B+1,) row indices into feats")
        off = off.astype(np.int32)
        b = off.size - 1
        emb = torch.empty(b, self.embed_dim, dtype=torch.float32, device=feats.device)
        check(lib.xvb_extractor_extract_ragged(self._h, _ptr(feats), off.ctypes.data_as(C.c_void_p), b, _ptr(emb), _stream()),
              "xvb_extractor_extract_ragged")
        return emb

    def extract_ragged_shard_host(self, feats, offsets, batch=256, max_frames=0):
        """N utterances of any lengths in host memory: feats (sum_T, F) float32 (ndarray or CPU tensor; staged through
        pinned memory unless it is a pinned tensor already), offsets (N+1,) -> (N, D) float32 ndarray in input order.
        Batches as xvb_ragged_plan cuts them (max_frames <= 0: 262144 padded frames per batch)."""
        if isinstance(feats, torch.Tensor) and feats.is_pinned() and feats.dtype == torch.float32 and feats.is_contiguous():
            host = feats
        else:
            src = torch.as_tensor(np.ascontiguousarray(feats, dtype=np.float32))
            if src.dim() != 2:
                raise ValueError("expected (sum_T, {}) features, got {}".format(self.feat_dim, tuple(src.shape)))
            host = self.staging_buffer(src.shape[0])
            host.copy_(src)
        if host.dim() != 2 or host.shape[1] != self.feat_dim:
            raise ValueError("expected (sum_T, {}) features, got {}".format(self.feat_dim, tuple(host.shape)))
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64))
        if off.ndim != 1 or off.size < 2 or off[-1] > host.shape[0]:
            raise ValueError("offsets must be (N+1,) row indices into feats")
        n = off.size - 1
        emb = np.empty((n, self.embed_dim), dtype=np.float32)
        check(lib.xvb_extractor_extract_ragged_shard_host(self._h, C.c_void_p(host.data_ptr()), off.ctypes.data_as(C.c_void_p), n,
                                                          int(batch), int(max_frames), emb.ctypes.data_as(C.c_void_p), _stream()),
              "xvb_extractor_extract_ragged_shard_host")
        return emb

    def staging_buffer(self, rows):
        """(rows, F) float32 pinned host tensor, a view of a grow-only buffer this extractor keeps: pinning is expensive,
        so repeated ragged calls reuse it.  Valid until the next call that stages through it."""
        buf = getattr(self, "_pinned", None)
        if buf is None or buf.shape[0] < rows:
            buf = torch.empty(max(int(rows), 1), self.feat_dim, dtype=torch.float32, pin_memory=True)
            self._pinned = buf
        return buf[:rows]

    def extract_host_into(self, feats_ptr, b, t, emb_ptr):
        check(lib.xvb_extractor_extract_host(self._h, C.c_void_p(feats_ptr), b, t, C.c_void_p(emb_ptr), _stream()),
              "xvb_extractor_extract_host")

    def set_fused_pooling(self, enable):
        """Default on: tdnn5's epilogue pools over time itself; off: fp32 tensor + standalone pooling kernel."""
        check(lib.xvb_extractor_set_fused_pooling(self._h, 1 if enable else 0), "xvb_extractor_set_fused_pooling")

    def set_profiling(self, enable):
        check(lib.xvb_extractor_set_profiling(self._h, 1 if enable else 0), "xvb_extractor_set_profiling")

    def kernel_times_ms(self, max_n=64):
        """Durations (ms) between consecutive profiling events of the last extract call, launch order (needs
        set_profiling).  After extract_shard(): every batch contributes its kernels plus the gap to the next batch."""
        buf = (C.c_float * max_n)()
        n = lib.xvb_extractor_kernel_times(self._h, buf, max_n)
        if n < 0:
            check(n, "xvb_extractor_kernel_times")
        return [float(buf[i]) for i in range(n)]

    @property
    def last_launches(self):
        return lib.xvb_extractor_last_launches(self._h)

    def debug_f32(self, which, shape):
        """View of an internal fp32 buffer of the last call (which=-1: pooled stats, 0: last frame layer)."""
        ptr = lib.xvb_extractor_debug_f32(self._h, which)
        if not ptr:
            raise _lib.XvbError("no debug buffer")

        class _DevPtr:  # zero-copy view through the CUDA array interface
            __cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False),
                                        "version": 2}

        torch.cuda.synchronize()
        return torch.as_tensor(_DevPtr(), device="cuda").clone()

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib.xvb_extractor_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
