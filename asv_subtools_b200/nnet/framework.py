"""`TopVirtualNnet` plugin base + whole-utterance wrapper, mirroring
pytorch/libs/nnet/framework.py (for_extract_embedding :12-55, TopVirtualNnet :61-186).

Contract kept (SURVEY section 8b): `Cls(inputs_dim, num_targets, **params)` with `init()`,
`load_state_dict(strict=False)` on the reference's keys, `.cuda()/.cpu()/.eval()`,
`extract_embedding(feats[T,F] float32 ndarray) -> 1-D CPU float32 tensor`, the `maxChunk`
splitting rule.  What is new: `extract_embedding_batch()` for equal-length utterances and
`extract_embedding_ragged()` for a list of utterances of any lengths."""
import numpy as np
import torch


def for_extract_embedding(maxChunk=10000, isMatrix=True):
    """Decorator with the reference's semantics (framework.py:18-52).  The wrapped function
    receives a channel-contiguous CUDA tensor (1, frames, feat_dim) and returns (1, D)."""

    def wrapper(function):
        def _wrapper(self, input):
            train_status = self.training
            self.eval()
            with torch.no_grad():
                x = torch.as_tensor(np.asarray(input) if not isinstance(input, torch.Tensor) else input)
                if not isMatrix:
                    # reference layout (1, F, T) -> (T, F)
                    x = x[0].transpose(0, 1)
                if x.dtype != torch.float32:
                    # the reference fails on float64 features (SURVEY Appendix B.1)
                    raise TypeError("extract_embedding expects float32 features, got {}".format(x.dtype))
                x = x.to(self.device_for_extraction(), non_blocking=True).contiguous()
                num_frames = x.shape[0]
                num_split = (num_frames + maxChunk - 1) // maxChunk
                split_size = num_frames // num_split
                offset = 0
                acc = None
                for _ in range(num_split - 1):
                    e = function(self, x[offset:offset + split_size].unsqueeze(0))
                    acc = split_size * e if acc is None else acc + split_size * e
                    offset += split_size
                last = function(self, x[offset:].unsqueeze(0))
                emb = (num_frames - offset) * last if acc is None else acc + (num_frames - offset) * last
                emb = emb / num_frames
                if train_status:
                    self.train()
                return torch.squeeze(emb).cpu()

        return _wrapper

    return wrapper


class TopVirtualNnet(torch.nn.Module):
    """Top-level plugin base.  Subclasses implement `init(...)` (build the parameter containers)
    and `build_extractor()` (hand the current parameters to the native library)."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        name = type(self).__name__
        args_str = ",".join(repr(a) for a in args)
        kwargs_str = ",".join("{}={!r}".format(k, v) for k, v in kwargs.items())
        self.model_creation = "{}({})".format(name, ",".join(s for s in (args_str, kwargs_str) if s))
        self.loss = None
        self.use_step = False
        self.transform_keys = []
        self.rename_transform_keys = {}
        self._extractor = None
        self.init(*args, **kwargs)

    def init(self, *args, **kwargs):
        raise NotImplementedError

    def get_model_creation(self):
        return self.model_creation

    # ---- native extractor lifecycle ------------------------------------------------------
    def build_extractor(self):
        raise NotImplementedError

    def invalidate(self):
        if self._extractor is not None:
            self._extractor.close()
        self._extractor = None
        self._extractor_device = None

    def extractor(self):
        if self._extractor is None:
            self._extractor = self.build_extractor()
        return self._extractor

    def load_state_dict(self, state_dict, strict=True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self.invalidate()
        return out

    def _apply(self, fn, *a, **kw):  # .cuda()/.cpu()/.to(): packed weights live on one device
        out = super()._apply(fn, *a, **kw)
        self.invalidate()
        return out

    def device_for_extraction(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("asv_subtools_b200 has no CPU path: move the model to a B200 with .cuda() "
                               "(extract_embeddings.py --use-gpu true)")
        return dev

    def _extraction_device(self):
        """The CUDA device the packed weights live on (cached with the extractor), or None on the CPU."""
        if self._extractor is not None and getattr(self, "_extractor_device", None) is not None:
            return self._extractor_device
        dev = next(self.parameters()).device
        self._extractor_device = dev if dev.type == "cuda" else None
        return self._extractor_device

    def load_transform_state_dict(self, state_dict):
        keep = {self.rename_transform_keys.get(k, k): v for k, v in state_dict.items()
                if k.split(".")[0] in self.transform_keys or k in self.transform_keys}
        self.load_state_dict(keep, strict=False)
        return self

    # ---- extraction surface ----------------------------------------------------------------
    @for_extract_embedding(maxChunk=10000, isMatrix=True)
    def _extract_embedding_chunked(self, inputs):
        """inputs (1, frames, feat_dim) CUDA float32 -> (1, D)."""
        return self.extractor().extract(inputs)

    def extract_embedding(self, feats):
        """feats (T, F) float32 ndarray / CPU tensor -> 1-D CPU float32 tensor: the reference's plugin call
        (framework.py:12-55, :146-153).  An utterance that fits one chunk -- every utterance up to maxChunk = 10000
        frames -- goes through the C host-buffer call (H2D, the stack, D2H and one synchronisation inside the
        library, no torch kernels), which roughly halves the per-call latency; the reference's arithmetic for that
        case, `(T * emb) / T` in fp32, is applied on the host.  Longer utterances take the chunk rule."""
        x = feats.numpy() if isinstance(feats, torch.Tensor) and not feats.is_cuda else feats
        if isinstance(x, np.ndarray) and x.ndim == 2 and 0 < x.shape[0] <= 10000:
            if x.dtype != np.float32:
                raise TypeError("extract_embedding expects float32 features, got {}".format(x.dtype))
            dev = self._extraction_device()
            ex = self.extractor() if dev is not None else None
            if ex is not None and hasattr(ex, "extract_host"):
                train_status = self.training
                if train_status:
                    self.eval()
                n = np.float32(x.shape[0])
                if torch.cuda.current_device() == dev.index:
                    emb = (n * ex.extract_host(x[None])[0]) / n
                else:
                    with torch.cuda.device(dev):
                        emb = (n * ex.extract_host(x[None])[0]) / n
                if train_status:
                    self.train()
                return torch.from_numpy(emb)
        return self._extract_embedding_chunked(feats)

    def extract_embedding_batch(self, feats):
        """Equal-length utterances in one call: feats (B, T, F) float32 (CUDA tensor, CPU tensor or
        ndarray; T <= maxChunk) -> (B, D) CUDA tensor.  Same arithmetic as B calls of
        extract_embedding()."""
        with torch.no_grad():
            x = torch.as_tensor(feats)
            if x.dtype != torch.float32:
                raise TypeError("extract_embedding_batch expects float32 features")
            if x.shape[1] > 10000:
                raise ValueError("T > maxChunk: use extract_embedding() per utterance")
            x = x.to(self.device_for_extraction(), non_blocking=True).contiguous()
            return self.extractor().extract(x)

    def extract_embedding_ragged(self, feats_list):
        """Utterances of different lengths in one call: a list of (T_i, F) float32 arrays or tensors, 1 <= T_i <= maxChunk
        -> (N, D) float32 CPU tensor in input order, each row what extract_embedding() gives for that utterance alone.
        TDNN x-vector extractors run length-sorted ragged batches (xvb_extractor_extract_ragged_shard_host); extractors
        without a ragged path group the utterances by exact length and call extract_embedding_batch() per group."""
        arrays = []
        for i, f in enumerate(feats_list):
            a = f.detach().cpu().numpy() if isinstance(f, torch.Tensor) else np.asarray(f)
            if a.dtype != np.float32:
                raise TypeError("extract_embedding_ragged expects float32 features, utterance {} is {}".format(i, a.dtype))
            if a.ndim != 2 or a.shape[0] < 1:
                raise ValueError("utterance {}: expected a (T, F) matrix with T >= 1, got shape {}".format(i, a.shape))
            if a.shape[0] > 10000:
                raise ValueError("utterance {} has {} frames > maxChunk (10000): use extract_embedding() for it".format(i, a.shape[0]))
            arrays.append(a)
        if not arrays:
            raise ValueError("extract_embedding_ragged: empty list")
        dev = self.device_for_extraction()
        ex = self.extractor()
        if not hasattr(ex, "extract_ragged_shard_host"):
            groups = {}
            for i, a in enumerate(arrays):
                groups.setdefault(a.shape[0], []).append(i)
            out = None
            for idx in groups.values():
                emb = self.extract_embedding_batch(np.stack([arrays[i] for i in idx])).cpu()
                if out is None:
                    out = torch.empty(len(arrays), emb.shape[1], dtype=torch.float32)
                out[torch.as_tensor(idx)] = emb
            return out
        offsets = np.zeros(len(arrays) + 1, dtype=np.int64)
        np.cumsum([a.shape[0] for a in arrays], out=offsets[1:])
        if any(a.shape[1] != ex.feat_dim for a in arrays):
            raise ValueError("expected {}-dim features".format(ex.feat_dim))
        host = ex.staging_buffer(int(offsets[-1]))
        hv = host.numpy()
        for a, o0, o1 in zip(arrays, offsets[:-1], offsets[1:]):
            hv[o0:o1] = a
        train_status = self.training
        self.eval()
        try:
            with torch.cuda.device(dev):
                emb = ex.extract_ragged_shard_host(host, offsets)
        finally:
            if train_status:
                self.train()
        return torch.from_numpy(emb)


def build_tdnn_extractor(model, inputs_dim, frame_layers, stats, tdnn6, tdnn7, extracted_embedding):
    """Hand a TDNN x-vector family model (frame-level ReluBatchNormTdnnLayers -> StatisticsPooling ->
    tdnn6 [-> tdnn7]) to the native extractor: weights exactly as stored in the state_dict, eval
    BatchNorm folded to (scale, shift).  "far" = tdnn6.affine, "near" / "near_affine" = tdnn6 (full) ->
    tdnn7.affine (pytorch/model/xvector.py:92-96, extended_xvector.py:112-116), "near_full" = tdnn6 -> tdnn7 with
    its ReLU and BatchNorm (what snowdar_xvector.py calls "near", :291-294)."""
    from .. import ops
    if extracted_embedding not in ("far", "near", "near_affine", "near_full"):
        raise TypeError("Expected far or near position, but got {}".format(extracted_embedding))
    model.device_for_extraction()
    ex = ops.Extractor(inputs_dim)

    def arrays(layer):
        w, b, scale, shift, _ = layer.export()         # "bn-relu" layers come back with the BatchNorm folded in
        return w.cpu().numpy(), (b.cpu().numpy() if b is not None else None), scale, shift

    for layer in frame_layers:
        w, b, scale, shift = arrays(layer)
        ex.add_frame_layer(w, b, layer.affine.context, scale, shift, relu=layer.relu)
    w, b, scale, shift = arrays(tdnn6)
    if extracted_embedding == "far":               # tdnn6.affine alone: the stored weight, whatever the layer's BN order
        ex.add_segment_layer(tdnn6.affine.dense_weight().cpu().numpy(),
                             tdnn6.affine.bias.detach().float().cpu().numpy() if tdnn6.affine.bias is not None else None)
    else:
        ex.add_segment_layer(w, b, scale, shift, relu=tdnn6.relu)
        w7, b7, s7, t7 = arrays(tdnn7)
        if extracted_embedding == "near_full":     # the whole last layer (snowdar_xvector.py:291-294)
            ex.add_segment_layer(w7, b7, s7, t7, relu=tdnn7.relu)
        else:                                      # tdnn7.affine alone
            ex.add_segment_layer(tdnn7.affine.dense_weight().cpu().numpy(),
                                 tdnn7.affine.bias.detach().float().cpu().numpy() if tdnn7.affine.bias is not None else None)
    ex.finalize(pooling_eps=stats.eps)
    return ex


class _PackedAffine:
    """One TdnnAffine (+ optional ReLU / folded eval-BatchNorm) packed for the tcgen05 layer kernel on `device`:
    block-diagonal expansion for groups > 1, output rows zero-padded to a multiple of `pad_to`, `row_scale` folded into
    weight and bias (per-head temperature of the attention logits)."""

    @classmethod
    def from_layer(cls, layer, device):
        """A whole ReluBatchNormTdnnLayer (its `export()` folds the BatchNorm in for the "bn-relu" order)."""
        w, b, scale, shift, relu = layer.export()
        return cls(layer.affine, device, relu=relu, arrays=(w, b, scale, shift))

    def __init__(self, affine, device, bn=None, relu=False, pad_to=8, row_scale=None, arrays=None):
        from .. import ops
        from .components import fold_batchnorm
        w = (arrays[0] if arrays is not None else affine.dense_weight()).to(device)
        b = arrays[1] if arrays is not None else (affine.bias.detach().float() if affine.bias is not None else None)
        b = b.to(device) if b is not None else None
        if row_scale is not None:
            w = w * row_scale.to(device).view(-1, 1, 1)
            b = b * row_scale.to(device) if b is not None else None
        self.cout_real = w.shape[0]
        pad = (-w.shape[0]) % pad_to
        if pad:
            w = torch.cat([w, torch.zeros(pad, w.shape[1], w.shape[2], device=device)], 0)
            b = torch.cat([b, torch.zeros(pad, device=device)], 0) if b is not None else None
        self.context, self.cout = list(affine.context), w.shape[0]
        self.w = ops.pack_tdnn_weight(w.contiguous(), self.context)
        self.bias = b.contiguous() if b is not None else None
        scale, shift = (arrays[2], arrays[3]) if arrays is not None else fold_batchnorm(bn)
        if scale is not None and pad:                            # padded output channels come out as exact zeros
            scale, shift = np.concatenate([scale, np.zeros(pad, np.float32)]), np.concatenate([shift, np.zeros(pad, np.float32)])
        self.scale = torch.from_numpy(scale).to(device) if scale is not None else None
        self.shift = torch.from_numpy(shift).to(device) if shift is not None else None
        self.relu = relu

    def run(self, x, **kw):
        from .. import ops
        ops.tdnn_affine_ex(x, self.w, self.cout, self.context, bias=self.bias, bn_scale=self.scale, bn_shift=self.shift,
                           relu=self.relu, **kw)

    def planes(self, b, t, device):
        """(buffer to write, view of the real channels for the next layer)."""
        from .. import ops
        y = ops.SplitPlanes.empty((b, t, self.cout), device)
        return y, (y if self.cout == self.cout_real else y.slice(0, self.cout_real))


class AttentionPoolingExtractor:
    """Launch sequence of a TDNN x-vector whose pooling is one of the attention poolings or LDE (nnet/pooling.py): frame
    layers on the tcgen05 layer kernel (the last one also writes fp32, the pooling kernel's x), then either the attention
    affines as GEMMs (grouped weights expanded block-diagonally, temperature folded into the last affine, logits fp32) +
    softmax over time + weighted mean / std in one pass (`xvb_attn_head_stats_pool`), or the dictionary encoding
    (`xvb_lde_pool`); then the segment layers on T = 1."""

    def __init__(self, model, inputs_dim, frame_layers, stats, tdnn6, tdnn7, position):
        dev = model.device_for_extraction()
        self.feat_dim = inputs_dim
        self.frames = [_PackedAffine.from_layer(l, dev) for l in frame_layers]
        self.lde = self.xi = None
        if hasattr(stats, "prior_logprec"):                      # xi-vector: precision network + prior element
            self.first = _PackedAffine.from_layer(stats.lin1_relu_bn, dev)
            self.last = _PackedAffine(stats.lin2, dev)
            self.xi = (stats.prior_logprec.detach().float().reshape(-1).to(dev).contiguous(),
                       stats.prior_mean.detach().float().reshape(-1).to(dev).contiguous(), bool(stats.stddev))
            self.channels, self.pooled, self.gdiv = stats.input_dim, stats.input_dim, 1
            self.eps, self.unweighted = 1.0e-10, False           # clamp(sigma2 - phi^2, min=1e-10), pooling.py:205
            self._segments(dev, tdnn6, tdnn7, position)
            return
        if hasattr(stats, "mu"):                                 # LDEPooling: no attention network
            self.lde = (stats.mu.detach().float().to(dev).contiguous(), stats.neg_beta().to(dev).contiguous())
            self.first = self.last = None
            self._segments(dev, tdnn6, tdnn7, position)
            return
        att = stats.attention
        self.first = _PackedAffine(att.first_affine, dev, relu=True) if att.relu_affine else None
        temps = att.head_temperatures()
        row_scale = None
        if temps is not None:                                    # logits of head h are divided by t_h (pooling.py:314-316)
            row_scale = (1.0 / temps).repeat_interleave(att.final_dim)
        self.last = _PackedAffine(att.last_affine, dev, row_scale=row_scale)
        self.channels, self.pooled, self.gdiv = stats.input_dim, stats.pooled_channels(), stats.logit_divisor()
        self.eps, self.unweighted = stats.eps, not stats.stddev_attention
        self._segments(dev, tdnn6, tdnn7, position)

    def _segments(self, dev, tdnn6, tdnn7, position):
        if position == "far":
            self.segment = [_PackedAffine(tdnn6.affine, dev)]
        else:
            self.segment = [_PackedAffine.from_layer(tdnn6, dev)]
            if position == "near_full":
                self.segment.append(_PackedAffine.from_layer(tdnn7, dev))
            else:
                self.segment.append(_PackedAffine(tdnn7.affine, dev))
        self.embed_dim = self.segment[-1].cout_real
        self.last_launches = 0

    def extract(self, feats):
        from .. import ops
        if feats.shape[2] != self.feat_dim:
            raise ValueError("expected feature dim {}, got {}".format(self.feat_dim, feats.shape[2]))
        B, T, _ = feats.shape
        dev, P = feats.device, ops.SplitPlanes
        x = ops.split_f32(feats, ld=(self.feat_dim + 7) // 8 * 8)
        for layer in self.frames[:-1]:
            y, view = layer.planes(B, T, dev)
            layer.run(x, y=y)
            x = view
        top = self.frames[-1]
        y, xp = top.planes(B, T, dev)
        xf = torch.empty(B, T, top.cout, dtype=torch.float32, device=dev)
        if self.lde is not None:
            top.run(x, y_f32=xf)
            _, x = ops.lde_pool(xf[..., :top.cout_real], self.lde[0], self.lde[1], planes=True)
        else:
            top.run(x, y=y, y_f32=xf)
            h = xp
            if self.first is not None:
                y, h = self.first.planes(B, T, dev)
                self.first.run(xp, y=y)
            logits = torch.empty(B, T, self.last.cout, dtype=torch.float32, device=dev)
            self.last.run(h, y_f32=logits)
            if self.xi is not None:
                _, x = ops.attn_head_stats_pool(logits[..., :self.last.cout_real], xf[..., :top.cout_real], self.pooled, 1, floor=self.eps,
                                                planes=True, prior_logit=self.xi[0], prior_x=self.xi[1], softplus2log=True)
                if not self.xi[2]:                               # post-mean variant: phi alone
                    x = x.slice(0, self.pooled)
            else:
                _, x = ops.attn_head_stats_pool(logits[..., :self.last.cout_real], xf[..., :top.cout_real], self.pooled, self.gdiv,
                                                floor=self.eps, unweighted_var=self.unweighted, planes=True)
        for i, layer in enumerate(self.segment):
            if i + 1 == len(self.segment):
                emb = torch.empty(B, 1, layer.cout, dtype=torch.float32, device=dev)
                layer.run(x, y_f32=emb)
            else:
                y, view = layer.planes(B, 1, dev)
                layer.run(x, y=y)
                x = view
        self.last_launches = len(self.frames) + (2 if self.lde is not None else (2 if self.first is not None else 1) + 1) + 1 + \
            len(self.segment)
        return emb.view(B, -1)[:, :self.embed_dim]

    def close(self):
        pass
