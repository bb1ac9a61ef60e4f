"""The serving loop's host-buffer form of a streaming step, shared by TemporalCRN and FullSubNet.process_chunk_host."""
from __future__ import annotations

import torch


def process_chunk_host(model, host_chunk, host_out):
    """host_chunk [B, M, K] -> host_out [B, K/2] through ``model.process_chunk``, with pinned HOST buffers.  The
    host->device copy, the chunk step and the device->host copy run on three CUDA streams over double-buffered device
    staging (kept in ``model._pipe``), so that with back-to-back calls the copies of neighbouring steps overlap the
    compute.  Returns a CUDA event that completes when ``host_out`` holds this chunk's result."""
    if host_chunk.is_cuda or host_out.is_cuda or not host_chunk.is_pinned() or not host_out.is_pinned():
        raise ValueError("process_chunk_host expects pinned host tensors")
    B, M, K = host_chunk.shape
    dev = model._pick_device(None)
    with torch.cuda.device(dev):
        pl = getattr(model, "_pipe", None)
        if pl is None or pl["shape"] != (B, M, K) or pl["dev"] != dev:
            d = torch.device("cuda", dev)
            pl = model._pipe = dict(
                shape=(B, M, K), dev=dev, slot=0, s_in=torch.cuda.Stream(d), s_out=torch.cuda.Stream(d),
                din=[torch.empty((B, M, K), dtype=torch.float32, device=d) for _ in range(2)],
                dout=[torch.empty((B, K // 2), dtype=torch.float32, device=d) for _ in range(2)],
                ev_in=[torch.cuda.Event() for _ in range(2)], ev_comp=[torch.cuda.Event() for _ in range(2)],
                ev_out=[torch.cuda.Event() for _ in range(2)], used=[False, False])
        k = pl["slot"]
        pl["slot"] = k ^ 1
        main = torch.cuda.current_stream(dev)
        with torch.cuda.stream(pl["s_in"]):
            if pl["used"][k]:
                pl["s_in"].wait_event(pl["ev_comp"][k])  # the step that read this staging buffer is done
            else:
                pl["s_in"].wait_stream(main)
            pl["din"][k].copy_(host_chunk, non_blocking=True)
            pl["ev_in"][k].record(pl["s_in"])
        main.wait_event(pl["ev_in"][k])
        if pl["used"][k]:
            main.wait_event(pl["ev_out"][k])  # the previous result in this output buffer has left the device
        model.process_chunk(pl["din"][k], pl["dout"][k])
        pl["ev_comp"][k].record(main)
        with torch.cuda.stream(pl["s_out"]):
            pl["s_out"].wait_event(pl["ev_comp"][k])
            host_out.copy_(pl["dout"][k], non_blocking=True)
            pl["ev_out"][k].record(pl["s_out"])
        pl["used"][k] = True
    return pl["ev_out"][k]
