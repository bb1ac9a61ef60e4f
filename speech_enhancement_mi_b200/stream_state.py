"""Per-stream state records of the streaming contexts (se_crn_state_export / se_fsn_state_export and their imports).

A record holds everything the next step of one stream reads; its bytes depend on the model, configuration and precision
only, so records move between rows, between contexts of any ``max_streams`` and between GPUs.  ``TemporalCRN`` and
``FullSubNet`` expose ``export_state(rows)`` / ``import_state(state, rows)`` on top of the helpers here.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple

import torch

from ._native import check


class StreamState(NamedTuple):
    """Records of n streams: ``data`` is a uint8 tensor [n, record_bytes], ``layout`` the hash that a context importing
    them must match (model kind, configuration, precision and the buffers that hold state)."""
    layout: int
    data: torch.Tensor


def row_list(rows):
    """A sequence of ints or an integer tensor -> list of Python ints."""
    if torch.is_tensor(rows):
        if rows.is_floating_point() or rows.is_complex() or rows.dim() > 1:
            raise ValueError("rows must be a 1-D integer tensor or a sequence of ints")
        return [int(r) for r in rows.tolist()]
    return [int(r) for r in rows]


def export_records(ctx, dev, rows, record_bytes, layout, export_fn, stream, what):
    """record i <- row rows[i] of the native context, on `stream` of device `dev`; returns a StreamState on that device."""
    rows = row_list(rows)
    data = torch.empty((len(rows), record_bytes), dtype=torch.uint8, device=f"cuda:{dev}")
    arr = (C.c_int32 * max(len(rows), 1))(*rows)
    check(export_fn(ctx, arr, len(rows), C.c_void_p(data.data_ptr()), stream), what)
    return StreamState(int(layout), data)


def import_records(ctx, dev, state, rows, record_bytes, layout, import_fn, stream, what):
    """row rows[i] of the native context <- record i of `state` (moved to device `dev` first if it lives elsewhere)."""
    rows = row_list(rows)
    if int(state.layout) != int(layout):
        raise ValueError(f"{what}: record layout {int(state.layout):#x} does not match this context's {int(layout):#x} "
                         "(another model, configuration or precision)")
    data = state.data
    if data.dtype != torch.uint8 or data.dim() != 2:
        raise ValueError(f"{what}: state.data must be a uint8 [n, record_bytes] tensor")
    if data.shape[1] != record_bytes:
        raise ValueError(f"{what}: record size mismatch ({data.shape[1]} bytes per stream, this context needs "
                         f"{record_bytes})")
    if data.shape[0] != len(rows):
        raise ValueError(f"{what}: {data.shape[0]} records for {len(rows)} rows")
    data = data.to(f"cuda:{dev}", non_blocking=True).contiguous()
    arr = (C.c_int32 * max(len(rows), 1))(*rows)
    # a copy made here belongs to the current stream of `dev`, the stream the import runs on: freeing it is safe
    check(import_fn(ctx, arr, len(rows), C.c_void_p(data.data_ptr()), C.c_uint64(int(layout)), stream), what)
