"""Drop-in for the reference's ``distillation_crn`` module: the student / teacher ``TemporalCRN`` with its feature taps
(distillation_crn.py:283-501) and the ``DistillationCRN`` training wrapper (distillation_crn.py:504-566).

``TemporalCRN`` is the same graph as CRN_ELU.TemporalCRN with two numerics differences the kernels switch on
(SE_VARIANT_DISTILLED): GlobalLayerNorm divides by ``sqrt(var) + 1e-8`` (distillation_crn.py:51) and the phase is
``arctan(im / (re + 1e-8) + 1e-8)`` (distillation_crn.py:340).  ``realtime_process`` returns ``(pred, features)`` as in
the reference.  ``features`` are the five PRE-activation tensors of distillation_crn.py:343-377 (last encoder conv, GRU
Linear, the three gated-skip transposed convs), each ``[chunks*B, C, F, T]`` in the chunk-major order of
distillation_crn.py:466.  They are produced by the native training context (``se_crn_train_tap``) whenever the module is
in train mode or ``return_features`` is set; under autograd they carry a graph node whose backward hands the injected
gradients to ``se_crn_train_backward_taps``.  In eval mode without ``return_features`` (the serving path,
predict_distillation.py:84 discards them) the list is empty and the streaming kernels run.

``DistillationCRN`` keeps the reference's constructor, parameter aliasing, connectors and loss.  The two networks and
their backward passes are native; the connector (1x1 conv + BatchNorm2d on five small tensors) and the margin loss are
ordinary torch modules, exactly as in the reference -- they are training-only glue outside the chunk step.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _native
from .CRN_ELU import TemporalCRN as _TemporalCRN
from .CRN_ELU import _grads_out, _save_mixture

EPS = 1e-8  # distillation_crn.py:13


class _RealtimeTapsFn(torch.autograd.Function):
    """realtime_process + feature taps under autograd: outputs (pred, tap_0 .. tap_4); no arithmetic in PyTorch."""

    @staticmethod
    def forward(ctx, model, mixture, flag, *params):
        ctx.model = model
        ctx.shapes = [p.shape for p in params]
        pred = model._train_forward(_save_mixture(ctx, model, mixture), flag)
        taps = model._train_taps()
        ctx.fwd_gen = model._fwd_gen
        return (pred, *taps)

    @staticmethod
    def backward(ctx, dpred, *dtaps):
        if ctx.fwd_gen != ctx.model._fwd_gen:
            raise RuntimeError("backward() of a realtime_process result whose activations are gone: another forward ran "
                               "on the model's training context in between")
        mixture, = ctx.saved_tensors
        flat, offsets, dmix = ctx.model._train_backward(dpred, dtaps, mixture=mixture,
                                                        params=any(ctx.needs_input_grad[3:]))
        return _grads_out(ctx, flat, offsets, dmix)


class TemporalCRN(_TemporalCRN):
    _variant = _native.SE_VARIANT_DISTILLED
    return_features = False  # eval mode: also return the feature taps (the frozen teacher of DistillationCRN)

    def forward(self, x):
        return super().forward(x), []

    def realtime_process(self, mixture, flag=False):
        if not (self.training or self.return_features):
            return super().realtime_process(mixture, flag), []
        B, Cm, L = mixture.shape
        if Cm != self.num_inputs:
            raise ValueError(f"mixture must be [B, {self.num_inputs}, L]")
        dev = self._pick_device(mixture)
        _, n_chunks = _native.chunk_grid(L + (0 if flag else self.segment_length // 2), self.segment_length)
        self._ensure_train_ctx(self._train_capacity(B, n_chunks), dev, keep_state=bool(flag))
        if torch.is_grad_enabled() and (mixture.requires_grad or any(p.requires_grad for p in self.parameters())):
            pred, *taps = _RealtimeTapsFn.apply(self, mixture, bool(flag), *self._train_params())
            return pred, list(taps)
        with torch.no_grad():
            pred = self._train_forward(mixture, flag)
            return pred, self._train_taps()

    def get_channel_num(self):  # distillation_crn.py:384-385
        c = self.num_channels
        return [c[-1], c[-1], c[2], c[1], c[0]]


class DistillationCRN(nn.Module):
    """distillation_crn.py:504-566: teacher + student + feature connectors; forward returns (loss, stoi, sisnr)."""

    def __init__(self, *args, **kargs):
        super().__init__()
        model_path = kargs.pop("path", None)
        self.teacher = TemporalCRN(*args, **kargs)
        if model_path is not None:
            self.teacher.load_state_dict(torch.load(model_path))
            self.teacher.eval()
            for param in self.teacher.parameters():
                param.requires_grad = False
        self.teacher.return_features = True
        kargs["num_channels"] = [16, 32, 64, 64]
        kargs["hidden"] = 128
        self.student = TemporalCRN(*args, **kargs)
        # distillation_crn.py:527-529: same-shaped student parameters start from (and SHARE STORAGE with) the teacher's
        self._aliased = False
        for pt, ps in zip(self.teacher.parameters(), self.student.parameters()):
            if ps.shape == pt.shape:
                ps.data = pt.data
                self._aliased = True
        t_channels = self.teacher.get_channel_num()
        s_channels = self.student.get_channel_num()
        self.connectors = nn.ModuleList([self.build_feature_connector(t, s) for t, s in zip(t_channels, s_channels)])

    def build_feature_connector(self, t_channel, s_channel):
        C = [nn.Conv2d(s_channel, t_channel, kernel_size=1, stride=1, padding=0, bias=False), nn.BatchNorm2d(t_channel)]
        for m in C:
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        return nn.Sequential(*C)

    def get_margin(self, ft):  # distillation_crn.py:548-552: per-channel mean of the negative responses
        mask = (ft < 0.0).float()
        return (ft * mask).sum(dim=(0, 2, 3), keepdim=True) / (mask.sum(dim=(0, 2, 3), keepdim=True) + EPS)

    def distillation_loss(self, ft, fs):  # distillation_crn.py:554-564
        loss = 0.0
        for i in range(len(ft)):
            t, s = ft[i], fs[i]
            t = torch.max(t, self.get_margin(t))
            s = self.connectors[i](s)
            mask = 1.0 - ((s <= t) & (t <= 0.0)).float()
            loss = loss + torch.mean((s - t) ** 2 * mask)
        return loss / len(ft)

    def forward(self, noisy, clean, length, flag):
        if self._aliased:  # an optimizer step on a student parameter also moved the teacher tensor that shares its storage
            self.teacher._tbound_versions = None
        _, ft = self.teacher.realtime_process(noisy, flag)
        pred, fs = self.student.realtime_process(noisy, flag)
        loss, stoi, sisnr = self.student.compute_loss(clean, pred, length)
        loss = loss + self.distillation_loss(ft, fs)
        return loss, stoi, sisnr
