"""Drop-in for the reference's ``CRN_ELU`` module: ``TemporalCRN`` with the reference's constructor kwargs, parameter
names / shapes (so reference checkpoints load, including the ``net.0`` alias keys) and methods, with every piece of
arithmetic running in the hand-written sm_100a kernels behind the C-ABI of ``include/se_b200.h``.

Reference: CRN_ELU.py:314-535 (class), :194-312 (blocks whose parameters are mirrored here), config.yaml:205-217.
PyTorch is used for parameter storage, device memory and streams only -- there is no PyTorch / CPU compute fallback:
if ``libse_b200.so`` is missing or no B200 is visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn as nn

from . import _host_pipeline, _native, stream_state
from ._native import SeCrnConfig, check, lib
from .stream_state import StreamState  # noqa: F401  (the type export_state returns)

EPS = 1e-8  # CRN_ELU.py:11


# ----------------------------------------------------------------------------------------------------------------
# Parameter containers with the reference's attribute names (no compute happens in these modules)
# ----------------------------------------------------------------------------------------------------------------
class GlobalLayerNorm(nn.Module):
    """Parameters of CRN_ELU.py:13-56 (weight/bias [1,C,1,1], or [1,1,1,C] with last=True)."""

    def __init__(self, dim, last=False, time=True):
        super().__init__()
        self.time = time
        shape = (1, 1, 1, dim) if last else (1, dim, 1, 1)
        self.weight = nn.Parameter(torch.ones(*shape))
        self.bias = nn.Parameter(torch.zeros(*shape))


class TemporalConv2d(nn.Module):
    """Parameters of CRN_ELU.py:194-252; `net` re-registers `conv` and yields the reference's `net.0.*` alias keys."""

    def __init__(self, n_inputs, n_outputs, kernel_size, stride, dilation, padding, dropout=0.0, activation="ELU"):
        super().__init__()
        if activation != "ELU":
            raise NotImplementedError(f"Not implemented activation function {activation}")
        self.padding = padding[1]
        self.conv = nn.Conv2d(n_inputs, n_outputs, kernel_size, stride=stride, padding=(padding[0], 0),
                              dilation=dilation)
        self.conv_trans = nn.Conv2d(n_outputs, n_outputs, 1, stride=1, padding=0)
        self.conv_gated = nn.Conv2d(n_outputs, n_outputs, 1, stride=1, padding=0)
        self.dropout = nn.Dropout(dropout)
        self.net = nn.Sequential(self.conv, self.dropout)
        self.norm = GlobalLayerNorm(n_outputs, time=False)


class TemporalConvTranspose2d(nn.Module):
    """Parameters of CRN_ELU.py:254-312."""

    def __init__(self, n_inputs, n_outputs, kernel_size, stride, dilation, padding, dropout=0.0, activation="ELU"):
        super().__init__()
        if activation != "ELU":
            raise NotImplementedError(f"Not implemented activation function {activation}")
        self.padding = padding[1]
        self.conv = nn.ConvTranspose2d(n_inputs, n_outputs, kernel_size, stride=stride, padding=(padding[0], 0),
                                       dilation=dilation)
        self.dropout = nn.Dropout(dropout)
        self.net = nn.Sequential(self.conv, self.dropout)
        self.residualmask = nn.Conv2d(n_outputs, n_outputs, (1, 1))
        self.residualnorm = GlobalLayerNorm(n_outputs, time=False)
        self.residual = nn.Conv2d(n_outputs, n_outputs, (1, 1))
        self.norm = GlobalLayerNorm(n_outputs, time=False)


class SequenceModel(nn.Module):
    """Parameters of CRN_ELU.py:98-192 for the configuration TemporalCRN builds (GRU + Linear + ELU + GLN(last))."""

    def __init__(self, input_size, output_size, hidden_size, num_layers, bidirectional=False, linear=True,
                 sequence_model="GRU", output_activate_function="ELU"):
        super().__init__()
        if sequence_model != "GRU" or bidirectional or not linear:
            raise NotImplementedError(f"Not implemented {sequence_model}")
        if output_activate_function != "ELU":
            raise NotImplementedError(f"Not implemented activation function {output_activate_function}")
        self.sequence_model = nn.GRU(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers,
                                     batch_first=True, bidirectional=False)
        self.fc_output_layer = nn.Linear(hidden_size, output_size)
        self.norm = GlobalLayerNorm(output_size, last=True, time=False)


# ----------------------------------------------------------------------------------------------------------------
# autograd plumbing of the training micro-step (train.py:195-198).  No arithmetic happens in PyTorch: the two graph
# nodes below only hand device pointers to se_crn_train_forward / se_crn_train_backward and se_loss_terms_grad.
# ----------------------------------------------------------------------------------------------------------------
def _save_mixture(ctx, model, mixture):
    """Keep the device copy of the mixture the forward reads when its gradient is wanted (the backward recomputes the
    mixture's 3-mic spectrum from it); returns that copy."""
    xd = model._to_device(mixture, model._pick_device(mixture))
    ctx.mixture_meta = (mixture.device, mixture.dtype) if ctx.needs_input_grad[1] else None
    ctx.save_for_backward(xd if ctx.needs_input_grad[1] else None)
    return xd


def _grads_out(ctx, flat, offsets, dmix):
    """(None, d mixture, None, *parameter gradients) for the autograd.Function inputs (model, mixture, flag, *params)."""
    grads = [None] * len(ctx.shapes) if flat is None else \
        [flat[o:o + s.numel()].view(s) for o, s in zip(offsets, ctx.shapes)]
    if dmix is not None:
        device, dtype = ctx.mixture_meta
        dmix = dmix.to(device=device, dtype=dtype)
    return (None, dmix, None, *grads)


class _RealtimeTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, mixture, flag, *params):
        ctx.model = model
        ctx.shapes = [p.shape for p in params]
        pred = model._train_forward(_save_mixture(ctx, model, mixture), flag)
        ctx.fwd_gen = model._fwd_gen  # the training context keeps the activations of its LAST forward only
        return pred

    @staticmethod
    def backward(ctx, dpred):
        if ctx.fwd_gen != ctx.model._fwd_gen:
            raise RuntimeError("backward() of a realtime_process result whose activations are gone: another forward ran "
                               "on the model's training context in between (call backward before the next "
                               "realtime_process, as train.py:195-198 does)")
        mixture, = ctx.saved_tensors
        flat, offsets, dmix = ctx.model._train_backward(dpred, mixture=mixture,
                                                        params=any(ctx.needs_input_grad[3:]))
        return _grads_out(ctx, flat, offsets, dmix)


class _LossTermsFn(torch.autograd.Function):
    """(stoi_loss, cal_si_snr) of utility.py:821-916,207-223 with their hand-written backward."""

    @staticmethod
    def forward(ctx, source, pred, length):
        dev = pred.device
        B, L = pred.shape
        src = source.detach().to(device=dev, dtype=torch.float32).contiguous()
        prd = pred.detach().to(torch.float32).contiguous()
        lens = torch.as_tensor(length).to(device=dev, dtype=torch.int32).contiguous()
        out2 = torch.empty(2, dtype=torch.float32, device=dev)
        d_stoi = torch.empty((B, L), dtype=torch.float32, device=dev)
        d_sisnr = torch.empty((B, L), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().se_loss_terms_grad(src.data_ptr(), prd.data_ptr(), lens.data_ptr(), B, L, out2.data_ptr(),
                                           d_stoi.data_ptr(), d_sisnr.data_ptr(),
                                           C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "se_loss_terms_grad")
        ctx.save_for_backward(d_stoi, d_sisnr)
        return out2[0].clone(), out2[1:2].clone()

    @staticmethod
    def backward(ctx, g_stoi, g_sisnr):
        d_stoi, d_sisnr = ctx.saved_tensors
        dev = d_stoi.device
        a = g_stoi.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        b = g_sisnr.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        out = torch.empty_like(d_stoi)
        with torch.cuda.device(dev):
            check(lib().se_axpby_dev(a.data_ptr(), d_stoi.data_ptr(), b.data_ptr(), d_sisnr.data_ptr(), out.data_ptr(),
                                     out.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "se_axpby_dev")
        return None, out, None


class TemporalCRN(nn.Module):
    """B200-native ``CRN_ELU.TemporalCRN`` (reference CRN_ELU.py:314-535).

    Extra keyword arguments (not in the reference, all optional): ``precision`` ("fp32" exact CUDA-core arithmetic,
    "3xtf32" tcgen05 tensor cores on split fp32 operands (tf32 head + tail, three products) with exact-mode epilogues,
    accurate to fp32, "tf32" tcgen05 tensor cores on fp32 storage, "fp16" tcgen05 tensor cores with fp16 operand
    storage and fp32 accumulation), ``max_streams`` (capacity of the per-stream state arena; grows on demand),
    ``device`` (CUDA device index used when tensors arrive on the CPU, as in predict.py:48).
    """

    _variant = _native.SE_VARIANT_CRN_ELU

    def __init__(self, num_channels, num_freqs, hidden, segment_length, num_layers=1, num_inputs=3, kernel_size=3,
                 dropout=0.0, sample_rate=16000, win_length=25, hop_length=10, n_fft=400, precision=None,
                 max_streams=None, device=None):
        super().__init__()
        self.segment_length = segment_length
        self.num_freqs = num_freqs
        self.num_channels = list(num_channels)
        self.hidden = hidden
        self.num_layers = num_layers
        self.num_inputs = num_inputs
        self.kernel_size = kernel_size
        self.n_fft = n_fft
        self.win_samples = int(round(sample_rate / 1000.0 * win_length))  # speechbrain STFT: ms -> samples
        self.hop_samples = int(round(sample_rate / 1000.0 * hop_length))
        activation = "ELU"
        cin0 = 2 * num_inputs - 1

        preconvs = []
        frequency_dilations = [1, 2, 4, 8]
        for i in range(3):
            preconvs += [TemporalConv2d(cin0, cin0, (5, 5), stride=(1, 1), dilation=(frequency_dilations[i], 1),
                                        padding=(2 * frequency_dilations[i], 4), dropout=dropout,
                                        activation=activation)]
        self.preconvlist = nn.ModuleList(preconvs)

        convs, deconvs = [], []
        num_levels = len(num_channels)
        for i in range(num_levels):
            d = 2 ** i
            cin = cin0 if i == 0 else num_channels[i - 1]
            cout = num_channels[i]
            convs += [TemporalConv2d(cin, cout, (5, kernel_size), stride=(2, 1), dilation=(1, d),
                                     padding=(2, (kernel_size - 1) * d), dropout=dropout, activation=activation)]
            d = 2 ** (num_levels - i - 1)
            dec = TemporalConvTranspose2d(cout, 2 if i == 0 else cin, (5, kernel_size), stride=(2, 1),
                                          dilation=(1, d), padding=(2, (kernel_size - 1) * d), dropout=dropout,
                                          activation=activation)
            deconvs = [dec] + deconvs
        self.convlist = nn.ModuleList(convs)
        self.deconvlist = nn.ModuleList(deconvs)
        feat = (num_freqs // 2 ** num_levels + 1) * num_channels[-1]
        self.gru = SequenceModel(feat, feat, hidden, num_layers, False, linear=True, sequence_model="GRU",
                                 output_activate_function=activation)

        # ---- native side -----------------------------------------------------------------------------------
        if precision is None:
            precision = os.environ.get("SE_B200_PRECISION", "fp32")
        if precision not in ("fp32", "3xtf32", "tf32", "fp16"):
            raise ValueError(f"precision must be 'fp32', '3xtf32', 'tf32' or 'fp16', got {precision!r}")
        self.precision = precision
        self._max_streams = int(max_streams) if max_streams else 0
        self._device_index = device
        self._ctx = None
        self._tctx_gen = 0  # bumped whenever the native training context is (re-)created
        self._fwd_gen = 0   # bumped by every forward on the training context
        self._ctx_device = None
        self._ctx_capacity = 0
        self._bound_versions = None
        self._fresh = True  # no chunk processed since the last reset
        # training context (chunk-major batch; created on the first realtime_process under autograd)
        # offline inference of a few long signals goes through the chunk-major batched forward (see realtime_process)
        self.chunk_batch = os.environ.get("SE_B200_CHUNK_BATCH", "1") != "0"
        self.chunk_batch_max_streams = 8
        self._state_owner = "stream"
        self._tctx = None
        self._tctx_device = None
        self._tctx_capacity = 0
        self._tbound_versions = None
        self._t_offsets = None

    # ------------------------------------------------------------------------------------------------------------
    # native context management
    # ------------------------------------------------------------------------------------------------------------
    def _config(self, capacity, training=False):
        cfg = SeCrnConfig()
        cfg.training = 1 if training else 0
        cfg.num_inputs = self.num_inputs
        cfg.num_freqs = self.num_freqs
        cfg.num_levels = len(self.num_channels)
        for i, ch in enumerate(self.num_channels):
            cfg.num_channels[i] = ch
        cfg.hidden = self.hidden
        cfg.num_layers = self.num_layers
        cfg.kernel_size = self.kernel_size
        cfg.segment_length = self.segment_length
        cfg.n_fft = self.n_fft
        cfg.win_length = self.win_samples
        cfg.hop_length = self.hop_samples
        cfg.variant = self._variant
        cfg.precision = {"fp32": _native.SE_PRECISION_FP32, "3xtf32": _native.SE_PRECISION_3XTF32,
                         "tf32": _native.SE_PRECISION_TF32, "fp16": _native.SE_PRECISION_FP16}[self.precision]
        if training and self.precision == "fp16":
            cfg.precision = _native.SE_PRECISION_TF32  # training keeps fp32 activations (tensor cores on fp32 storage)
        cfg.max_streams = capacity
        return cfg

    def _pick_device(self, tensor):
        if tensor is not None and tensor.is_cuda:
            return tensor.device.index if tensor.device.index is not None else torch.cuda.current_device()
        p = next(self.parameters())
        if p.is_cuda:
            return p.device.index
        if self._device_index is not None:
            return int(self._device_index)
        return int(os.environ.get("LOCAL_RANK", "0"))

    def _destroy_ctx(self):
        if self._ctx is not None:
            lib().se_ctx_destroy(self._ctx)
            self._ctx = None
            self._bound_versions = None
        if getattr(self, "_tctx", None) is not None:
            lib().se_ctx_destroy(self._tctx)
            self._tctx = None
            self._tbound_versions = None

    def __del__(self):
        try:
            self._destroy_ctx()
        except Exception:
            pass

    def _ensure_ctx(self, B, device, keep_state):
        need = max(B, self._max_streams, 1)
        if self._ctx is not None and (device != self._ctx_device or need > self._ctx_capacity):
            if keep_state and not self._fresh:
                raise RuntimeError(
                    "stream state would be lost: the context must be re-created (device or stream count changed) "
                    "while flag=True continues a previous call; construct TemporalCRN(max_streams=...) large enough")
            self._destroy_ctx()
        if self._ctx is None:
            ctx = C.c_void_p()
            cfg = self._config(need)
            check(lib().se_ctx_create(C.byref(ctx), device, C.byref(cfg)), "se_ctx_create")
            self._ctx, self._ctx_device, self._ctx_capacity = ctx, device, need
            self._fresh = True
        self._bind_weights()
        return self._ctx

    def _named_param_map(self):
        return dict(self.named_parameters())  # named_parameters() de-duplicates the net.0 aliases

    def _bind_weights(self):
        params = self._named_param_map()
        n = lib().se_crn_num_params(self._ctx)
        names = [lib().se_crn_param_name(self._ctx, i).decode() for i in range(n)]
        tensors = []
        for i, name in enumerate(names):
            p = params[name]
            if p.numel() != lib().se_crn_param_numel(self._ctx, i):
                raise RuntimeError(f"parameter {name}: expected {lib().se_crn_param_numel(self._ctx, i)} elements")
            tensors.append(p)
        versions = tuple((t.data_ptr(), t._version) for t in tensors)
        if versions == self._bound_versions:
            return
        keep = [t.detach().to(torch.float32).contiguous() for t in tensors]
        arr = (C.c_void_p * n)(*[t.data_ptr() for t in keep])
        check(lib().se_crn_bind_weights(self._ctx, arr, n, None), "se_crn_bind_weights")
        self._bound_versions = versions

    @staticmethod
    def _stream_ptr(device):
        return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    # ------------------------------------------------------------------------------------------------------------
    # reference API
    # ------------------------------------------------------------------------------------------------------------
    def reset(self):
        """CRN_ELU.py:408-415: forget the causal-conv buffers and the GRU state of every stream."""
        if self._ctx is not None:
            with torch.cuda.device(self._ctx_device):
                check(lib().se_crn_state_reset(self._ctx, 0, self._ctx_capacity, self._stream_ptr(self._ctx_device)),
                      "se_crn_state_reset")
        self._fresh = True

    def _to_device(self, x, device):
        return x.detach().to(device=f"cuda:{device}", dtype=torch.float32).contiguous()

    def forward(self, x):
        """x [B, M, F, T, 2] (STFT of one chunk) -> enhanced spectrum [B, F, T, 2]; advances the stream state."""
        B, M, Fq, T, _ = x.shape
        if M != self.num_inputs or Fq != self.num_freqs or T != 1 + self.segment_length // self.hop_samples:
            raise ValueError(f"forward expects [B,{self.num_inputs},{self.num_freqs},"
                             f"{1 + self.segment_length // self.hop_samples},2], got {tuple(x.shape)}")
        dev = self._pick_device(x)
        ctx = self._ensure_ctx(B, dev, keep_state=True)
        with torch.cuda.device(dev):
            xd = self._to_device(x, dev)
            out = torch.empty((B, Fq, T, 2), dtype=torch.float32, device=xd.device)
            check(lib().se_crn_forward_chunk(ctx, xd.data_ptr(), out.data_ptr(), B, self._stream_ptr(dev)),
                  "se_crn_forward_chunk")
        self._fresh = False
        return out.to(x.device)

    def stft_trans(self, x):
        """[R, M, K] -> [R, M, F, T, 2] (CRN_ELU.py:417-424)."""
        R, M, K = x.shape
        if M != self.num_inputs or K != self.segment_length:
            raise ValueError("stft_trans expects [R, num_inputs, segment_length]")
        dev = self._pick_device(x)
        ctx = self._ensure_ctx(1, dev, keep_state=True)
        T = 1 + K // self.hop_samples
        with torch.cuda.device(dev):
            xd = self._to_device(x, dev)
            out = torch.empty((R, M, self.num_freqs, T, 2), dtype=torch.float32, device=xd.device)
            check(lib().se_stft_trans(ctx, xd.data_ptr(), R, out.data_ptr(), self._stream_ptr(dev)), "se_stft_trans")
        return out.to(x.device)

    def istft_trans(self, x):
        """[R, F, T, 2] -> [R, K] (CRN_ELU.py:426-432)."""
        R, Fq, T, _ = x.shape
        dev = self._pick_device(x)
        ctx = self._ensure_ctx(1, dev, keep_state=True)
        with torch.cuda.device(dev):
            xd = self._to_device(x, dev)
            out = torch.empty((R, self.segment_length), dtype=torch.float32, device=xd.device)
            check(lib().se_istft_trans(ctx, xd.data_ptr(), R, out.data_ptr(), self._stream_ptr(dev)),
                  "se_istft_trans")
        return out.to(x.device)

    def segmentation(self, x):
        from .utility import segmentation
        return segmentation(x, self.segment_length)

    def overadd(self, x, gap):
        from .utility import over_add
        return over_add(x, gap)

    def preprocessing(self, mixture):
        """[B, M, L] -> ([N, B, M, F, T, 2], gap) (CRN_ELU.py:444-456)."""
        batch_size = len(mixture)
        seg_x, gap = self.segmentation(mixture)
        x = self.stft_trans(seg_x)
        x = x.reshape([batch_size, -1] + [*x.shape[1:]]).transpose(0, 1)
        return x, gap

    def postprocessing(self, sp, gap):
        """[N, B, F, T, 2] -> [B, L] (CRN_ELU.py:458-469)."""
        N, B, Fq, T, _ = sp.shape
        sp = self.istft_trans(sp.reshape(N * B, Fq, T, 2))
        sp = sp.reshape(N, B, -1).permute(1, 0, 2)
        return self.overadd(sp, gap)

    # ------------------------------------------------------------------------------------------------------------
    # training micro-step (train.py:195-198): realtime_process under autograd
    # ------------------------------------------------------------------------------------------------------------
    def _train_params(self):
        params = self._named_param_map()
        n = lib().se_crn_num_params(self._tctx)
        return [params[lib().se_crn_param_name(self._tctx, i).decode()] for i in range(n)]

    def _ensure_train_ctx(self, n_streams, device, keep_state):
        need = max(n_streams, self._max_streams, 1)
        if self._tctx is not None and (device != self._tctx_device or need > self._tctx_capacity):
            if keep_state:
                raise RuntimeError("flag=True continues a previous piece, but the training context must be re-created "
                                   "(more chunk-streams than before); construct TemporalCRN(max_streams=...) larger")
            lib().se_ctx_destroy(self._tctx)
            self._tctx = None
            self._tbound_versions = None
        if self._tctx is None:
            ctx = C.c_void_p()
            cfg = self._config(need, training=True)
            check(lib().se_ctx_create(C.byref(ctx), device, C.byref(cfg)), "se_ctx_create(training)")
            self._tctx, self._tctx_device, self._tctx_capacity = ctx, device, need
            self._tctx_gen += 1  # a new native object (the old handle, possibly the same address, is dead)
            n = lib().se_crn_num_params(ctx)
            self._t_offsets = [lib().se_crn_param_offset(ctx, i) for i in range(n)]
        tensors = self._train_params()
        versions = tuple((t.data_ptr(), t._version) for t in tensors)
        if versions != self._tbound_versions:  # parameters changed (optimizer step / load_state_dict): re-lay out
            with torch.cuda.device(device):
                theta = torch.cat([t.detach().to(device=f"cuda:{device}", dtype=torch.float32).reshape(-1)
                                   for t in tensors])
                check(lib().se_crn_bind_weights_flat(self._tctx, theta.data_ptr(), self._stream_ptr(device)),
                      "se_crn_bind_weights_flat")
            self._tbound_versions = versions
        return self._tctx

    @staticmethod
    def _train_capacity(B, n_chunks):
        """Chunk-streams to allocate: at least the 44 chunks of the longest piece the reference's data pipeline emits
        (config.yaml:11 max_length 60000), so that flag=True pieces of any such length find the carried state."""
        return B * max(n_chunks, 44)

    def _train_forward(self, mixture, flag):
        B, _, L = mixture.shape
        dev = self._pick_device(mixture)
        _, n_chunks = _native.chunk_grid(L + (0 if flag else self.segment_length // 2), self.segment_length)
        ctx = self._ensure_train_ctx(self._train_capacity(B, n_chunks), dev, keep_state=bool(flag))
        with torch.cuda.device(dev):
            xd = self._to_device(mixture, dev)
            pred = torch.empty((B, L), dtype=torch.float32, device=xd.device)
            check(lib().se_crn_train_forward(ctx, xd.data_ptr(), B, L, int(bool(flag)), pred.data_ptr(),
                                             self._stream_ptr(dev)), "se_crn_train_forward")
        self._fwd_gen += 1
        self._last_chunk_streams = B * n_chunks
        return pred

    def _train_backward(self, dpred, dtaps=None, mixture=None, params=True):
        """-> (flat parameter gradient or None when ``params`` is False, offsets, d mixture or None).  ``mixture``: the
        device copy of the signal the last _train_forward read; given, d loss / d mixture is computed as well."""
        dev = self._tctx_device
        with torch.cuda.device(dev):
            dp = dpred.detach().to(device=f"cuda:{dev}", dtype=torch.float32).contiguous()
            flat = torch.empty(lib().se_crn_num_theta(self._tctx), dtype=torch.float32, device=dp.device) \
                if params else None
            keep = arr = None
            if dtaps is not None:  # gradients of the distillation loss injected at the feature taps (distillation_crn.py:560-565)
                keep = [None if g is None else g.detach().to(device=dp.device, dtype=torch.float32).contiguous()
                        for g in dtaps]
                arr = (C.c_void_p * len(keep))(*[None if g is None else g.data_ptr() for g in keep])
            if mixture is not None:
                dmix = torch.empty_like(mixture)
                check(lib().se_crn_train_backward_input(self._tctx, mixture.data_ptr(), dp.data_ptr(), arr,
                                                        len(keep) if keep else 0,
                                                        None if flat is None else flat.data_ptr(), dmix.data_ptr(),
                                                        self._stream_ptr(dev)), "se_crn_train_backward_input")
                return flat, self._t_offsets, dmix
            if dtaps is None:
                check(lib().se_crn_train_backward(self._tctx, dp.data_ptr(), flat.data_ptr(), self._stream_ptr(dev)),
                      "se_crn_train_backward")
            else:
                check(lib().se_crn_train_backward_taps(self._tctx, dp.data_ptr(), arr, len(keep), flat.data_ptr(),
                                                       self._stream_ptr(dev)), "se_crn_train_backward_taps")
        return flat, self._t_offsets, None

    def _train_taps(self):
        """The pre-activation feature taps of the last _train_forward, each [chunks*B, C, F, T]
        (distillation_crn.py:343-377,466)."""
        dev = self._tctx_device
        taps = []
        with torch.cuda.device(dev):
            for k in range(lib().se_crn_train_num_taps(self._tctx)):
                c, f, t = C.c_int(), C.c_int(), C.c_int()
                check(lib().se_crn_train_tap_shape(self._tctx, k, C.byref(c), C.byref(f), C.byref(t)),
                      "se_crn_train_tap_shape")
                out = torch.empty((self._last_chunk_streams, c.value, f.value, t.value), dtype=torch.float32,
                                  device=f"cuda:{dev}")
                check(lib().se_crn_train_tap(self._tctx, k, out.data_ptr(), self._stream_ptr(dev)), "se_crn_train_tap")
                taps.append(out)
        return taps

    def realtime_process(self, mixture, flag=False):
        """[B, M, L] -> [B, L] (CRN_ELU.py:472-509).  One fused native call: padding, chunk grid, per-chunk STFT,
        network, mask, iSTFT and both overlap-adds happen on the device; with CPU tensors (predict.py:48,59-62) the
        host<->device copies are inside the native call as well.

        Under autograd in train mode (train.py:195), or in either mode when the mixture requires grad, the result carries
        a graph node whose backward is the native backward pass (parameters and / or d loss / d mixture, with the
        carried state detached as in the reference); the forward then runs batched over all chunks
        (se_crn_train_forward)."""
        B, Cm, L = mixture.shape
        if Cm != self.num_inputs:
            raise ValueError(f"mixture must be [B, {self.num_inputs}, L]")
        if torch.is_grad_enabled() and (mixture.requires_grad or (
                self.training and any(p.requires_grad for p in self.parameters()))):
            dev = self._pick_device(mixture)
            _, n_chunks = _native.chunk_grid(L + (0 if flag else self.segment_length // 2), self.segment_length)
            self._ensure_train_ctx(self._train_capacity(B, n_chunks), dev, keep_state=bool(flag))
            pred = _RealtimeTrainFn.apply(self, mixture, bool(flag), *self._train_params())
            if not self.training:  # eval mode: a flag=True continuation finds the state in the training context
                self._state_owner = "chunk-batch"
                self._fresh = False
            return pred
        dev = self._pick_device(mixture)
        # Few streams, many chunks (a file, predict.py:92): the carried state of a chunk is just the tail of the previous
        # chunk's layer inputs (CRN_ELU.py:243), so every layer can run ONCE over all chunks of all streams and only the
        # GRU recurrence stays serial -- the chunk-major forward of the training context, without a backward.
        _, n_chunks = _native.chunk_grid(L + (0 if flag else self.segment_length // 2), self.segment_length)
        batched = self._state_owner == "chunk-batch" if flag else (
            self.chunk_batch and self.precision != "fp16" and B <= self.chunk_batch_max_streams
            and 4 <= n_chunks <= 1024)  # fp16 operand mode exists only on the streaming path
        if batched:
            with torch.no_grad():
                pred = self._train_forward(mixture, flag)
            self._state_owner = "chunk-batch"
            self._fresh = False
            return pred if mixture.is_cuda else pred.cpu()
        self._state_owner = "stream"
        ctx = self._ensure_ctx(B, dev, keep_state=bool(flag))
        with torch.cuda.device(dev):
            if mixture.is_cuda:
                xd = self._to_device(mixture, dev)
                out = torch.empty((B, L), dtype=torch.float32, device=xd.device)
                check(lib().se_crn_realtime_process(ctx, xd.data_ptr(), B, L, int(bool(flag)), out.data_ptr(),
                                                    self._stream_ptr(dev)), "se_crn_realtime_process")
            else:
                xh = mixture.detach().to(torch.float32).contiguous()
                out = torch.empty((B, L), dtype=torch.float32, pin_memory=False)
                check(lib().se_crn_realtime_process_host(ctx, xh.data_ptr(), B, L, int(bool(flag)), out.data_ptr()),
                      "se_crn_realtime_process_host")
        self._fresh = False
        return out

    def process_chunk(self, chunk, out=None):
        """True-streaming step (not in the reference; SURVEY.md section 3.1 probe): chunk [B, M, K] on the device ->
        K/2 enhanced samples per stream (overlap-added with the carried half of the previous chunk)."""
        B, M, K = chunk.shape
        dev = self._pick_device(chunk)
        ctx = self._ensure_ctx(B, dev, keep_state=True)
        if not chunk.is_cuda:
            raise ValueError("process_chunk expects a CUDA tensor")
        with torch.cuda.device(dev):
            if out is None:
                out = torch.empty((B, K // 2), dtype=torch.float32, device=chunk.device)
            check(lib().se_crn_process_chunk(ctx, chunk.data_ptr(), chunk.stride(0), chunk.stride(1), out.data_ptr(),
                                             out.stride(0), B, self._stream_ptr(dev)), "se_crn_process_chunk")
        self._fresh = False
        return out

    def process_chunk_host(self, host_chunk, host_out):
        """Streaming step with pinned HOST buffers (throughput-oriented serving loop; not in the reference):
        host_chunk [B, M, K] -> host_out [B, K/2].  The host->device copy, the chunk step and the device->host copy run
        on three CUDA streams over double-buffered device staging, so that with back-to-back calls the copies of
        neighbouring steps overlap the compute.  Returns a CUDA event that completes when ``host_out`` holds this
        chunk's result (call ``.synchronize()`` before reading it).  State semantics are those of process_chunk."""
        return _host_pipeline.process_chunk_host(self, host_chunk, host_out)

    def export_state(self, rows):
        """Carried state of streams ``rows`` (ints or an int tensor; repeats allowed) -> ``StreamState`` on the
        context's device, one record per row (not in the reference).  Runs on the current torch stream of that device
        and leaves the streams untouched.  With ``import_state`` this moves live streams: compaction of the row prefix
        the step runs on, migration to a context with more rows or to another GPU, checkpoints (``.cpu()``)."""
        if self._state_owner == "chunk-batch":
            raise RuntimeError("export_state: the state was last advanced by the chunk-batched realtime_process, which "
                               "keeps it in the training context; stream with process_chunk to export it")
        if self._ctx is None:
            raise RuntimeError("export_state: no streaming context yet (nothing has been processed)")
        dev = self._ctx_device
        with torch.cuda.device(dev):
            return stream_state.export_records(
                self._ctx, dev, rows, lib().se_crn_state_bytes_per_stream(self._ctx), lib().se_crn_state_layout(self._ctx),
                lib().se_crn_state_export, self._stream_ptr(dev), "se_crn_state_export")

    def import_state(self, state, rows):
        """Write the records of ``state`` (from ``export_state`` of a model with the same configuration and precision)
        into streams ``rows`` (distinct), on the current torch stream of the context's device.  Creates the streaming
        context if there is none, with room for max(max_streams, max(rows) + 1) streams, on the device the records are
        on (CPU records: the model's device).  Captured step graphs stay valid: the state is written in place."""
        rows = stream_state.row_list(rows)
        dev = self._pick_device(state.data) if self._ctx is None else self._ctx_device
        ctx = self._ensure_ctx(max(rows, default=-1) + 1, dev, keep_state=True)
        with torch.cuda.device(dev):
            stream_state.import_records(
                ctx, dev, state, rows, lib().se_crn_state_bytes_per_stream(ctx), lib().se_crn_state_layout(ctx),
                lib().se_crn_state_import, self._stream_ptr(dev), "se_crn_state_import")
        self._state_owner = "stream"
        self._fresh = False

    def compute_loss(self, source, pred_source, length):
        """CRN_ELU.py:513-535: loss = 0.7 * stoi_loss + 0.3 * (-SI-SNR); NaN => zero-filled; prints sisnr."""
        from .utility import cal_si_snr, stoi_loss
        if pred_source.requires_grad:  # training: both terms and their backward in one native call
            mae, sisnr_db = _LossTermsFn.apply(source, pred_source, length)
            sisnr = -sisnr_db
        else:
            mae = stoi_loss(source, pred_source, length)
            sisnr = -cal_si_snr(pred_source, source, length)
        loss = 0.7 * mae + 0.3 * sisnr
        print(sisnr)
        if torch.isnan(loss):
            mae = mae.fill_(0.0)
            sisnr = sisnr.fill_(0.0)
            loss = loss.fill_(0.0)
        return loss, mae, sisnr
