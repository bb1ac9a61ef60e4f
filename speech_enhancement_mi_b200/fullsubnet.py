"""Drop-in for the streaming path of the reference's ``fullsubnet`` module: ``FullSubNet`` / ``BaseModel.unfold`` with
the reference's constructor kwargs (config.yaml:153-172), ``state_dict`` keys (``fb_model.*`` / ``sb_model.*``) and
methods, the arithmetic running in the sm_100a kernels behind include/se_b200.h (se_fsn_*).

Reference: fullsubnet.py:299-331 (unfold), :685-961 (FullSubNet).  ``realtime_process`` runs the chunked loop the
trainers and predictors use (``train=False``: train_fullsubnet.py:138,151; predict_fullsubnet.py:75) and, with
``train=True``, all chunks as one forward (both CumLayerNorms see the whole utterance), forward only: there is no
backward, and ``compute_loss`` has no autograd graph either.  ``process_chunk`` / ``process_chunk_host`` (not in the
reference) are the serving form of the loop: one chunk per call, the overlap-add carry kept on the device.  The
reference runs this loop under fp16 autocast on CUDA (fullsubnet.py:943) and in fp32 on the CPU; this path uses TF32
tensor cores with fp32 accumulation and fp32 cell state (or the ``precision`` modes below), checked against the fp32
CPU run.  No PyTorch / CPU compute fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn as nn

from . import utility
from . import _host_pipeline, _native, stream_state
from ._native import SeFsnConfig, check, lib
from .stream_state import StreamState  # noqa: F401  (the type export_state returns)

EPS = 1e-8


def _dev_of(x):
    if x.is_cuda:
        return x.device.index if x.device.index is not None else torch.cuda.current_device()
    return int(os.environ.get("LOCAL_RANK", "0"))


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _f32(x, dev):
    return x.detach().to(device=f"cuda:{dev}", dtype=torch.float32).contiguous()


class SequenceModel(nn.Module):
    """Parameters of fullsubnet.py:209-292 (nn.LSTM + nn.Linear); no compute happens in this module."""

    def __init__(self, input_size, output_size, hidden_size, num_layers, bidirectional, sequence_model="LSTM",
                 output_activate_function="Tanh"):
        super().__init__()
        if sequence_model != "LSTM" or bidirectional:
            raise NotImplementedError(f"Not implemented {sequence_model}")
        self.sequence_model = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers,
                                      batch_first=True, bidirectional=False)
        self.fc_output_layer = nn.Linear(hidden_size, output_size)
        self.output_activate_function = output_activate_function


class BaseModel(nn.Module):
    @staticmethod
    def unfold(input, num_neighbor):
        """[B, C, F, T] -> [B, F, C, 2n+1, T]; reflect padding along F (fullsubnet.py:299-331)."""
        assert input.dim() == 4, f"The dim of input is {input.dim()}. It should be four dim."
        B, Cn, Fq, T = input.shape
        dev = _dev_of(input)
        with torch.cuda.device(dev):
            xd = _f32(input, dev)
            out = torch.empty((B, Fq, Cn, 2 * max(num_neighbor, 0) + 1, T), dtype=torch.float32, device=xd.device)
            check(lib().se_unfold(xd.data_ptr(), B, Cn, Fq, T, max(int(num_neighbor), 0), out.data_ptr(), _stream(dev)),
                  "se_unfold")
        return out.to(input.device)


class FullSubNet(BaseModel):
    def __init__(self, num_freqs, look_ahead, sequence_model, fb_num_neighbors, sb_num_neighbors,
                 fb_output_activate_function, sb_output_activate_function, fb_model_hidden_size, sb_model_hidden_size,
                 num_mics, norm_type="offline_laplace_norm", num_groups_in_drop_band=2, num_layers=2, weight_init=True,
                 sample_rate=16000, segment_length=400, win_length=20, hop_length=10, n_fft=320, max_streams=None,
                 device=None, precision=None):
        super().__init__()
        # extra (not in the reference): "tf32" = tcgen05 on fp32 storage; "3xtf32" = tcgen05 on split fp32 operands
        # (tf32 head + tail, three products) with exact-mode LSTM cells, accurate to fp32; "fp16" = sub-band LSTM
        # operands stored as fp16 with fp32 accumulation / cell state -- the reference runs this model under fp16
        # autocast on CUDA (fullsubnet.py:943)
        self.precision = precision or os.environ.get("SE_B200_FSN_PRECISION", "tf32")
        if self.precision not in ("tf32", "3xtf32", "fp16"):
            raise ValueError("precision must be 'tf32', '3xtf32' or 'fp16'")
        assert sequence_model in ("GRU", "LSTM"), f"{self.__class__.__name__} only support GRU and LSTM."
        if sequence_model != "LSTM" or fb_output_activate_function != "ReLU" or sb_output_activate_function:
            raise NotImplementedError("the B200 path builds the configuration of config.yaml:153-172 "
                                      "(LSTM, ReLU full-band output, linear sub-band output)")
        if look_ahead != 0:
            raise NotImplementedError("look_ahead must be 0 (config.yaml:155)")
        self.win_samples = int(round(sample_rate / 1000.0 * win_length))
        self.hop_samples = int(round(sample_rate / 1000.0 * hop_length))
        if (n_fft, self.win_samples, self.hop_samples, segment_length) != (400, 400, 160, 3200):
            raise NotImplementedError("STFT kernels are built for n_fft=win=400, hop=160, segment_length=3200 "
                                      "(config.yaml:168-172)")
        self.fb_model = SequenceModel(num_freqs * num_mics, num_freqs, fb_model_hidden_size, num_layers, False,
                                      sequence_model, fb_output_activate_function)
        self.sb_model = SequenceModel((sb_num_neighbors * 2 + 1) + (fb_num_neighbors * 2 + 1), 2, sb_model_hidden_size,
                                      num_layers, False, sequence_model, sb_output_activate_function)
        self.sb_num_neighbors, self.fb_num_neighbors, self.look_ahead = sb_num_neighbors, fb_num_neighbors, look_ahead
        self.fb_model_hidden_size, self.sb_model_hidden_size = fb_model_hidden_size, sb_model_hidden_size
        self.num_layers, self.num_mics, self.num_freqs = num_layers, num_mics, num_freqs
        self.segment_length = segment_length
        self.num_groups_in_drop_band = num_groups_in_drop_band
        self.exist_prob = None
        self._max_streams = int(max_streams) if max_streams else 0
        self._device_index = device
        self._ctx, self._ctx_device, self._ctx_capacity, self._bound = None, None, 0, None
        self._fresh = True
        if weight_init:  # fullsubnet.py:616-626: xavier for Linear, orthogonal-ish for LSTM; default init kept otherwise
            pass

    # ---- native context ------------------------------------------------------------------------------------------
    def _pick_device(self, t):
        if t is not None and t.is_cuda:
            return _dev_of(t)
        p = next(self.parameters())
        if p.is_cuda:
            return p.device.index
        return int(self._device_index) if self._device_index is not None else int(os.environ.get("LOCAL_RANK", "0"))

    def _destroy(self):
        if self._ctx is not None:
            lib().se_fsn_destroy(self._ctx)
            self._ctx, self._bound = None, None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _ensure_ctx(self, B, dev, keep_state):
        need = max(B, self._max_streams, 1)
        if self._ctx is not None and (dev != self._ctx_device or need > self._ctx_capacity):
            if keep_state and not self._fresh:
                raise RuntimeError("stream state would be lost (device or stream count changed while flag=True); "
                                   "construct FullSubNet(max_streams=...) large enough")
            self._destroy()
        if self._ctx is None:
            cfg = SeFsnConfig(self.num_freqs, self.num_mics, self.fb_model_hidden_size, self.sb_model_hidden_size,
                              self.num_layers, self.sb_num_neighbors, self.fb_num_neighbors, need,
                              {"tf32": _native.SE_PRECISION_TF32, "3xtf32": _native.SE_PRECISION_3XTF32,
                               "fp16": _native.SE_PRECISION_FP16}[self.precision])
            ctx = C.c_void_p()
            check(lib().se_fsn_create(C.byref(ctx), dev, C.byref(cfg)), "se_fsn_create")
            self._ctx, self._ctx_device, self._ctx_capacity, self._fresh = ctx, dev, need, True
        self._bind()
        return self._ctx

    def _bind(self):
        params = dict(self.named_parameters())
        L = lib()
        n = L.se_fsn_num_params(self._ctx)
        tensors = [params[L.se_fsn_param_name(self._ctx, i).decode()] for i in range(n)]
        versions = tuple((t.data_ptr(), t._version) for t in tensors)
        if versions == self._bound:
            return
        keep = [t.detach().to(torch.float32).contiguous() for t in tensors]
        for i, t in enumerate(keep):
            if t.numel() != L.se_fsn_param_numel(self._ctx, i):
                raise RuntimeError(f"parameter {i}: unexpected size")
        arr = (C.c_void_p * n)(*[t.data_ptr() for t in keep])
        check(L.se_fsn_bind_weights(self._ctx, arr, n, None), "se_fsn_bind_weights")
        self._bound = versions

    # ---- reference API ---------------------------------------------------------------------------------------------
    def reset_state(self, batch_size, dtype=None, device=None):
        """fullsubnet.py:826-832: zero LSTM states, reset both CumLayerNorms."""
        if self._ctx is not None:
            with torch.cuda.device(self._ctx_device):
                check(lib().se_fsn_reset_state(self._ctx, 0, self._ctx_capacity, _stream(self._ctx_device)),
                      "se_fsn_reset_state")
        self._fresh = True

    def forward(self, noisy_complex):
        """[B, 2M, F, T=21] (real planes, then imaginary planes) -> compressed cIRM [B, 2, F, T]; advances the state."""
        assert noisy_complex.dim() == 4
        B, C2, Fq, T = noisy_complex.shape
        if C2 != 2 * self.num_mics or Fq != self.num_freqs or T != 1 + self.segment_length // self.hop_samples:
            raise ValueError(f"forward expects [B,{2 * self.num_mics},{self.num_freqs},"
                             f"{1 + self.segment_length // self.hop_samples}] (one chunk), got {tuple(noisy_complex.shape)}")
        dev = self._pick_device(noisy_complex)
        ctx = self._ensure_ctx(B, dev, keep_state=True)
        with torch.cuda.device(dev):
            xd = _f32(noisy_complex, dev)
            out = torch.empty((B, 2, Fq, T), dtype=torch.float32, device=xd.device)
            check(lib().se_fsn_forward_chunk(ctx, xd.data_ptr(), out.data_ptr(), B, _stream(dev)), "se_fsn_forward_chunk")
        self._fresh = False
        return out.to(noisy_complex.device)

    def process_chunk(self, chunk, out=None):
        """True-streaming step (not in the reference; the chunk loop of fullsubnet.py:932-957 for one chunk): chunk
        [B, M, K] on a CUDA device, any strides -> K/2 enhanced samples per stream [B, K/2] (or into ``out``, whose rows
        may be strided), overlap-added with the carried half of the previous chunk.  Advances the LSTM states, both
        CumLayerNorms and the carry of streams [0, B) in one CUDA-graph replay (se_fsn_process_chunk); reset_state()
        starts every stream afresh."""
        if not torch.is_tensor(chunk) or not chunk.is_cuda:
            raise ValueError("process_chunk expects a CUDA tensor")
        if chunk.dim() != 3 or chunk.shape[1] != self.num_mics or chunk.shape[2] != self.segment_length:
            raise ValueError(f"process_chunk expects [B, {self.num_mics}, {self.segment_length}], "
                             f"got {tuple(chunk.shape)}")
        B, _, K = chunk.shape
        if chunk.dtype != torch.float32 or chunk.stride(2) != 1:
            chunk = chunk.to(torch.float32).contiguous()
        dev = self._pick_device(chunk)
        if out is None:
            out = torch.empty((B, K // 2), dtype=torch.float32, device=chunk.device)
        elif (out.device != chunk.device or out.dtype != torch.float32 or tuple(out.shape) != (B, K // 2)
              or out.stride(1) != 1):
            raise ValueError(f"out must be a float32 [{B}, {K // 2}] tensor with unit sample stride on {chunk.device}")
        ctx = self._ensure_ctx(B, dev, keep_state=True)
        with torch.cuda.device(dev):
            check(lib().se_fsn_process_chunk(ctx, chunk.data_ptr(), chunk.stride(0), chunk.stride(1), out.data_ptr(),
                                             out.stride(0), B, _stream(dev)), "se_fsn_process_chunk")
        self._fresh = False
        return out

    def process_chunk_host(self, host_chunk, host_out):
        """process_chunk with pinned HOST buffers for a serving loop that keeps audio in host memory: host_chunk
        [B, M, K] -> host_out [B, K/2].  The copies run on side streams over double-buffered device staging, so that the
        copies of neighbouring steps overlap the compute.  Returns a CUDA event that completes when ``host_out`` holds
        this chunk's result (call ``.synchronize()`` before reading it).  State semantics are those of process_chunk."""
        return _host_pipeline.process_chunk_host(self, host_chunk, host_out)

    def export_state(self, rows):
        """Carried state of streams ``rows`` (ints or an int tensor; repeats allowed) -> ``StreamState`` on the
        context's device (not in the reference): both LSTM layers' h and c of the full-band and every sub-band sequence,
        both CumLayerNorms and the process_chunk carry.  Runs on the current torch stream of that device and leaves the
        streams untouched; see ``TemporalCRN.export_state`` for what it serves."""
        if self._ctx is None:
            raise RuntimeError("export_state: no streaming context yet (nothing has been processed)")
        dev = self._ctx_device
        with torch.cuda.device(dev):
            return stream_state.export_records(
                self._ctx, dev, rows, lib().se_fsn_state_bytes_per_stream(self._ctx), lib().se_fsn_state_layout(self._ctx),
                lib().se_fsn_state_export, _stream(dev), "se_fsn_state_export")

    def import_state(self, state, rows):
        """Write the records of ``state`` into streams ``rows`` (distinct), as ``TemporalCRN.import_state``: creates
        the context if there is none, with room for max(max_streams, max(rows) + 1) streams."""
        rows = stream_state.row_list(rows)
        dev = self._pick_device(state.data) if self._ctx is None else self._ctx_device
        ctx = self._ensure_ctx(max(rows, default=-1) + 1, dev, keep_state=True)
        with torch.cuda.device(dev):
            stream_state.import_records(
                ctx, dev, state, rows, lib().se_fsn_state_bytes_per_stream(ctx), lib().se_fsn_state_layout(ctx),
                lib().se_fsn_state_import, _stream(dev), "se_fsn_state_import")
        self._fresh = False

    def _spectrum(self, x, dev):
        R, M, K = x.shape
        xd = _f32(x, dev)
        spec = torch.empty((R, M, self.num_freqs, 1 + K // self.hop_samples, 2), dtype=torch.float32, device=xd.device)
        check(lib().se_stft_trans(None, xd.data_ptr(), R, spec.data_ptr(), _stream(dev)), "se_stft_trans")
        return spec

    def stft_trans(self, x):
        """[R, M, K] -> [R, 2M, F, T] (fullsubnet.py:835-844)."""
        R, M, K = x.shape
        dev = self._pick_device(x)
        with torch.cuda.device(dev):
            spec = self._spectrum(x, dev)
            T = spec.shape[3]
            s = torch.empty((R, 2 * M, self.num_freqs, T), dtype=torch.float32, device=spec.device)
            check(lib().se_fsn_planes(spec.data_ptr(), R, M, self.num_freqs, T, s.data_ptr(), None, _stream(dev)),
                  "se_fsn_planes")
        return s.to(x.device)

    def istft_trans(self, x):
        """[R, F, T, 2] -> [R, K] (fullsubnet.py:846-852)."""
        R = x.shape[0]
        dev = self._pick_device(x)
        with torch.cuda.device(dev):
            xd = _f32(x, dev)
            out = torch.empty((R, self.segment_length), dtype=torch.float32, device=xd.device)
            check(lib().se_istft_trans(None, xd.data_ptr(), R, out.data_ptr(), _stream(dev)), "se_istft_trans")
        return out.to(x.device)

    def segmentation(self, x):
        return utility.segmentation(x, self.segment_length)

    def overadd(self, x, gap):
        return utility.over_add(x, gap)

    def preprocessing(self, mixture, source=None):
        """[B, M, L] -> (x [N, B, 2M, F, T], s [N, B, 2, F, T] or None, gap) (fullsubnet.py:864-887)."""
        B = len(mixture)
        seg_x, gap = self.segmentation(mixture)
        x = self.stft_trans(seg_x)
        x = x.reshape([B, -1] + list(x.shape[1:])).transpose(0, 1)
        if source is None:
            return x, None, gap
        seg_s, gap = self.segmentation(source)
        dev = self._pick_device(seg_s)
        with torch.cuda.device(dev):
            spec = self._spectrum(seg_s, dev)
            R, M, Fq, T = spec.shape[:4]
            s = torch.empty((R, 2, Fq, T), dtype=torch.float32, device=spec.device)  # mic-0 real / imaginary (:886)
            check(lib().se_fsn_planes(spec.data_ptr(), R, M, Fq, T, None, s.data_ptr(), _stream(dev)), "se_fsn_planes")
        s = s.to(source.device).reshape([B, -1] + list(s.shape[1:])).transpose(0, 1)
        return x, s, gap

    def postprocessing(self, sp, gap):
        """[N, B, F, T, 2] -> [B, L] (fullsubnet.py:889-900)."""
        N, B, Fq, T, _ = sp.shape
        y = self.istft_trans(sp.reshape(N * B, Fq, T, 2))
        return self.overadd(y.reshape(N, B, -1).permute(1, 0, 2), gap)

    def realtime_process(self, mixture, source=None, flag=False, train=True):
        """fullsubnet.py:903-961 in ONE native call (se_fsn_realtime_process): front pad, segmentation, per-chunk STFT, the
        chunk loop (``train=False``: what the reference's trainers and predictors call, :932-945) or all chunks as one
        forward (``train=True``, the signature's default, :921-927), mask, iSTFT, overlap-add.  Returns ``pred`` when
        ``source`` is None, else the reference's 4-tuple (pred [B, L], pred_crm [N, B, 2, F, T], s [N, B, 2, F, T],
        x [N, B, 2, F, T]).  No PyTorch arithmetic: tensors are only allocated here."""
        B, Cm, L = mixture.shape
        if Cm != self.num_mics:
            raise ValueError(f"mixture must be [B, {self.num_mics}, L]")
        dev = self._pick_device(mixture)
        P = self.segment_length // 2
        ctx = self._ensure_ctx(B, dev, keep_state=bool(flag))
        _, N = _native.chunk_grid(L + (0 if flag else P), self.segment_length)
        T = 1 + self.segment_length // self.hop_samples
        with torch.cuda.device(dev):
            xd = _f32(mixture, dev)
            sd = None if source is None else _f32(source, dev)
            pred = torch.empty((B, L), dtype=torch.float32, device=xd.device)
            if source is None:
                crm = s = x0 = None
            else:
                shape = (N, B, 2, self.num_freqs, T)
                crm, s, x0 = (torch.empty(shape, dtype=torch.float32, device=xd.device) for _ in range(3))
            if not flag:
                self.exist_prob = 0.0
            check(lib().se_fsn_realtime_process(ctx, xd.data_ptr(), None if sd is None else sd.data_ptr(), B, L,
                                                int(bool(flag)), int(bool(train)), pred.data_ptr(),
                                                None if crm is None else crm.data_ptr(),
                                                None if s is None else s.data_ptr(),
                                                None if x0 is None else x0.data_ptr(), _stream(dev)),
                  "se_fsn_realtime_process")
            self._fresh = False
        pred = pred.to(mixture.device)
        if source is None:
            return pred
        return pred, crm.to(mixture.device), s.to(mixture.device), x0.to(mixture.device)

    def compute_loss(self, source, pred_source, xf, sf, cIRM, length):
        """fullsubnet.py:964-987 (forward only): loss = 0.7 * stoi_loss + 0.3 * (-SI-SNR); NaN => zero-filled."""
        mae = utility.stoi_loss(source, pred_source, length)
        sisnr = -utility.cal_si_snr(pred_source, source, length)
        loss = 0.7 * mae + 0.3 * sisnr
        print(sisnr, "\n")
        if torch.isnan(loss):
            mae = mae.fill_(0.0)
            sisnr = sisnr.fill_(0.0)
            loss = loss.fill_(0.0)
        return loss, mae, sisnr
