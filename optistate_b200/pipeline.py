"""Double-buffered host -> device -> host pipeline around kf_batch for callers whose inputs and results live in host
memory: the upload of batch k+1 and the download of batch k-1 run on their own CUDA streams underneath the filter kernel
of batch k, so sustained end-to-end throughput is max(compute, copies) instead of their sum.

    pipe = KfHostPipeline(n_traj, n_steps, n_streams, dtype=torch.float64, labels=("truth", "nominal"))
    for batch in batches:                       # dicts of pinned host tensors: imu p dp contact f [truth nominal] Q R
        ticket = pipe.submit(batch)
        ...
        summary = pipe.result(ticket)           # pinned host tensor [52, n_traj], valid until the slot is reused

Several GPUs filtering different members of the SAME base streams (the Monte-Carlo sweep: one process per GPU, contiguous shards
of the members): with `shared_streams_group` every rank uploads only its 1/world slice of the stream arrays over PCIe and the
ranks exchange the slices over NVLink (one in-place NCCL all-gather per batch, queued LAST on the upload stream), so every byte of
the streams crosses the host interface once per batch instead of once per GPU.  Per-member noise and summaries stay per rank.
Measured on one 8-GPU B200 box: 59.9 against 65.1 ms per batch at 4 GPUs, 67.1 against 79.9 ms at 8 (profiles/r2_e2e_upload_modes.txt).
"""
from __future__ import annotations

from typing import Dict, Sequence

import torch

from . import _native as nv
from .batch import kf_batch

_STREAM_CH = {"imu": 6, "p": 12, "dp": 12, "contact": 4, "f": 12, "truth": 12, "nominal": 12}


def stream_share_plan(sizes: Dict[str, int], world: int, rank: int):
    """Shared upload: the stream arrays of a slot live back to back in one flat allocation, padded to a multiple of `world`; rank r
    owns elements [r, r + 1) * flat_len / world of it.  Returns (flat_len, {name: (begin, end)} of every array in the flat
    allocation, [(name, begin_in_array, begin_in_flat, count)] = the pieces rank `rank` uploads).  Pure arithmetic (CPU-testable):
    over all ranks the pieces tile every array exactly once."""
    ranges, off = {}, 0
    for k, n in sizes.items():
        ranges[k] = (off, off + int(n))
        off += int(n)
    flat_len = (off + world - 1) // world * world
    share = flat_len // world
    c0, c1 = rank * share, (rank + 1) * share
    pieces = []
    for k, (a, b) in ranges.items():
        lo, hi = max(a, c0), min(b, c1)
        if lo < hi:
            pieces.append((k, lo - a, lo, hi - lo))
    return flat_len, ranges, pieces


class KfHostPipeline:
    def __init__(self, n_traj: int, n_steps: int, n_streams: int, *, dtype: torch.dtype = torch.float64,
                 labels: Sequence[str] = ("truth", "nominal"), stream_offset: int = 0, n_slots: int = 2, device=None,
                 structure: str = "auto", shared_streams_group=None, trace: bool = False):
        nv.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_traj, self.n_steps, self.n_streams, self.dtype = n_traj, n_steps, n_streams, dtype
        self.labels, self.stream_offset, self.n_slots = tuple(labels), int(stream_offset), n_slots
        self.structure = structure
        names = ["imu", "p", "dp", "contact", "f", *self.labels]
        self.group, self.world, self.rank = shared_streams_group, 1, 0
        if shared_streams_group is not None:
            import torch.distributed as dist

            self.world, self.rank = dist.get_world_size(shared_streams_group), dist.get_rank(shared_streams_group)
        # the stream arrays of a slot live back to back in one allocation (padded to a multiple of the world size), so that a rank's
        # share is one contiguous range of it
        self._flat_len, self._ranges, self._pieces = stream_share_plan({k: n_steps * _STREAM_CH[k] * n_streams for k in names}, self.world, self.rank)
        self.h2d_bytes_per_batch = 0  # what this rank copies from the host per submit (set below)
        self.slots = []
        for _ in range(n_slots):
            flat = torch.empty(self._flat_len, dtype=dtype, device=self.device)
            dev = {k: flat[a:b].view(n_steps, _STREAM_CH[k], n_streams) for k, (a, b) in self._ranges.items()}
            dev["Q"] = torch.empty((12, n_traj), dtype=dtype, device=self.device)
            dev["R"] = torch.empty((10, n_traj), dtype=dtype, device=self.device)
            out = {"summary": torch.empty((nv.SUMMARY_ROWS, n_traj), dtype=dtype, device=self.device),
                   "status": torch.zeros(n_traj, dtype=torch.int32, device=self.device)}
            # "workspace" is added by the slot's first kf_batch call, at the size the library asks for
            host = torch.empty((nv.SUMMARY_ROWS, n_traj), dtype=dtype).pin_memory()
            self.slots.append({"dev": dev, "flat": flat, "out": out, "host": host, "ev_in": torch.cuda.Event(), "ev_k": torch.cuda.Event(),
                               "ev_out": torch.cuda.Event(), "busy": False})
        self.s_in, self.s_k, self.s_out = (torch.cuda.Stream(device=self.device) for _ in range(3))
        self._next = 0
        # trace: timed events per submitted batch (upload start / uploads done / inputs complete / kernel start / kernel done / result on
        # the host), read back with timeline() - a development aid for the multi-GPU pipeline, off by default
        self._trace = [] if trace else None

    def submit(self, host: Dict[str, torch.Tensor]) -> int:
        """Queues one batch (pinned host tensors) and returns its ticket; blocks only if all slots are still in flight."""
        i = self._next
        self._next = (self._next + 1) % self.n_slots
        slot = self.slots[i]
        if slot["busy"]:
            slot["ev_out"].synchronize()  # the previous result of this slot must have left the device
        dev = slot["dev"]
        tr = None
        if self._trace is not None:
            tr = {k: torch.cuda.Event(enable_timing=True) for k in ("in0", "in1", "in2", "k0", "k1", "o1")}
            self._trace.append(tr)
        with torch.cuda.stream(self.s_in):
            if slot["busy"]:
                self.s_in.wait_event(slot["ev_k"])  # do not overwrite inputs a kernel may still be reading
            if tr:
                tr["in0"].record(self.s_in)
            copied = 0
            if self.world == 1:
                for k, d in dev.items():
                    d.copy_(host[k], non_blocking=True)
                    copied += d.numel()
            else:
                # this rank's share of the stream arrays over PCIe, the other shares over NVLink; noise is per rank
                import torch.distributed as dist

                flat, share = slot["flat"], self._flat_len // self.world
                c0, c1 = self.rank * share, (self.rank + 1) * share
                for k, src0, dst0, cnt in self._pieces:
                    flat[dst0:dst0 + cnt].copy_(host[k].reshape(-1)[src0:src0 + cnt], non_blocking=True)
                    copied += cnt
                for k in ("Q", "R"):
                    dev[k].copy_(host[k], non_blocking=True)
                    copied += dev[k].numel()
                if tr:
                    tr["in1"].record(self.s_in)
                # LAST on this stream: the exchange is a kernel with large blocks and only gets onto the SMs when the filter kernel of
                # the previous batch drains, so nothing that could run underneath that kernel may queue behind it (with the noise upload
                # after it, that upload - 185 MB per rank at the contended host rate - sat between two filter kernels: +12 - 18 ms per
                # step at 4 - 8 GPUs, profiles/r2_e2e_upload_modes.txt)
                dist.all_gather_into_tensor(flat, flat[c0:c1], group=self.group)
            self.h2d_bytes_per_batch = copied * (8 if self.dtype == torch.float64 else 4)
            slot["ev_in"].record(self.s_in)
            if tr:
                tr["in2"].record(self.s_in)
        with torch.cuda.stream(self.s_k):
            self.s_k.wait_event(slot["ev_in"])
            if tr:
                tr["k0"].record(self.s_k)
            kf_batch(dev["imu"], dev["p"], dev["dp"], dev["contact"], dev["f"], Q=dev["Q"], R=dev["R"], n_traj=self.n_traj,
                     dtype=self.dtype, stream_offset=self.stream_offset, truth=dev.get("truth"), nominal=dev.get("nominal"),
                     outputs=("summary",), out=slot["out"], q_kind=nv.MAT_DIAG_PER, r_kind=nv.MAT_DIAG_PER, device=self.device,
                     structure=self.structure)
            slot["ev_k"].record(self.s_k)
            if tr:
                tr["k1"].record(self.s_k)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(slot["ev_k"])
            slot["host"].copy_(slot["out"]["summary"], non_blocking=True)
            slot["ev_out"].record(self.s_out)
            if tr:
                tr["o1"].record(self.s_out)
        slot["busy"] = True
        return i

    def result(self, ticket: int) -> torch.Tensor:
        """Pinned host summary [52, n_traj] of a submitted batch (waits for its download)."""
        slot = self.slots[ticket]
        slot["ev_out"].synchronize()
        return slot["host"]

    def drain(self):
        for slot in self.slots:
            if slot["busy"]:
                slot["ev_out"].synchronize()

    def timeline(self):
        """With trace=True: per submitted batch, milliseconds from the first batch's upload start to its events (drain() first)."""
        if not self._trace:
            return []
        self.drain()
        torch.cuda.synchronize(self.device)
        base = self._trace[0]["in0"]
        out = []
        for tr in self._trace:
            row = {}
            for k, ev in tr.items():
                try:
                    row[k] = round(base.elapsed_time(ev), 2)
                except Exception:  # an event that was never recorded (in1 outside the shared upload mode)
                    row[k] = None
            out.append(row)
        return out

