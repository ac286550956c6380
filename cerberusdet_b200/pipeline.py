"""Streaming engine of the post-head path on one GPU: static buffers, CUDA graphs, and a two-stage software pipeline
in which the decode of batch k overlaps the NMS of batch k-1.

Why overlap.  The decode kernel is memory-bound (all SMs streaming 330 MB per config-3 batch); the NMS kernel is a
latency-bound chain of short phases that keeps the SMs ~30 % busy and touches little memory.  Run back to back they
take 64 + 52 us; run concurrently -- NMS of the previous batch on a second stream while the next batch is decoded --
a step takes ~98 us (profiles/r02_nms.md, "The overlapped step").  Both kernels are the same launches as in the serial path; only their
placement in time changes, so results are bit-identical to ``ops.decode_heads`` + ``ops.nms_batched``.

Step k (one CUDA-graph replay):      stream A:  decode(inputs)      -> Y[k & 1]
                                     stream B:  NMS(Y[(k-1) & 1])   -> OUT[(k-1) & 1]
``flush()`` runs the NMS of the last decoded batch.  Inputs are static device tensors (a serving loop copies -- or
lets the conv towers write -- each batch into them before ``step()``); outputs are static ``(dets, counts)`` buffers,
which may be caller-provided (e.g. ``shard.DetectionGatherer`` buffers, or rank 0's peer-mapped memory).
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import torch

from . import ops


# tools/ A/B only: "piggyback" (default) = the delivery rides on the NMS launches; "branch3" = stand-alone delivery kernels
# on a third branch of the step graph; "after" = small graphs replayed after the step graph; "off" = never (nothing is
# delivered: timing experiments only)
_SIDE = os.environ.get("CERB_SIDE", "piggyback")
# how the two kernels of an overlapped step are made concurrent: "pdl" = ONE stream, NMS(k-1) then decode(k) launched with
# the programmatic-serialization attribute (its CTAs are dispatched as soon as every NMS CTA is running, never before: the
# NMS CTAs, 109 KB of shared memory each, must be placed first or they wait for decode CTAs to drain); "streams" = two
# graph branches (the launch order of two root nodes is a race: 0.098 or 0.106 ms per step, profiles/r02_multi_gpu.md)
_SCHEDULE = os.environ.get("CERB_SCHEDULE", "pdl")
_STANDALONE = ("branch3", "last3", "pre_nms", "post_nms", "post_decode")  # where the stand-alone delivery kernel sits in the step graph


class PostHeadPipeline:
    def __init__(self, heads: Sequence[Sequence[torch.Tensor]], strides: Sequence[float], nms_kw: dict,
                 outs: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor]]] = None, timed_parities: Sequence[int] = (),
                 overlap: bool = True, delivery=None, timed_steps: Sequence[int] = ()):
        """``heads[t][l]``: static raw head tensors ``[B, 64+nc_t, H_l, W_l]`` on one CUDA device.  ``outs``: two
        ``(dets[T,B,max_det,6] float32, counts[T,B] int32)`` buffer pairs (allocated here when omitted).
        ``timed_parities`` additionally captures one instrumented step graph per entry (the NMS kernel, then the decode
        kernel alone, each between timing events recorded by the graph itself) for ``step(timed=i)``; entry i is the
        parity (step index & 1) of the step slot i will be used at.  ``overlap=False`` captures the serial
        order (decode -> NMS of the same batch, one stream) behind the same interface.
        ``delivery`` (N > 1): a ``shard.PeerDelivery`` (``in_graph``): its push / collect kernels are captured on a side
        branch of the step graphs (see ``_capture``), so a step stays ONE graph replay on every rank."""
        first = heads[0][0]
        if not first.is_cuda:
            raise TypeError("PostHeadPipeline needs CUDA tensors (cerberusdet_b200 has no CPU path)")
        self.device = first.device
        self.heads, self.strides, self.kw = [list(lv) for lv in heads], [float(s) for s in strides], dict(nms_kw)
        self.overlap = bool(overlap)
        self.delivery = delivery if (delivery is not None and getattr(delivery, "in_graph", False)) else None
        if self.delivery is not None:
            if outs is None:
                outs = self.delivery.outs
            if not self.overlap:
                raise ValueError("in-graph delivery is wired for the overlapped schedule")
        T, B = len(heads), int(first.shape[0])
        max_det = int(self.kw.get("max_det", 300))
        if outs is None:
            outs = [(torch.empty((T, B, max_det, 6), dtype=torch.float32, device=self.device),
                     torch.empty((T, B), dtype=torch.int32, device=self.device)) for _ in range(2)]
        if len(outs) != 2:
            raise ValueError("outs must hold exactly two (dets, counts) buffer pairs")
        self.outs = list(outs)
        self.k = 0            # steps issued in this run (a run = k = 0 .. n-1, then flush(); set k = 0, pending = None to start one)
        self.pending = None   # parity of the decoded batch whose NMS has not been issued yet
        with torch.cuda.device(self.device):
            self.ybuf = [ops.decode_buffers(self.heads) for _ in range(2)]
            self.sa, self.sb, self.sc = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
            # eager warm-up of both kernels (module load, function attributes) before anything is captured
            ys = ops.decode_heads(self.heads, self.strides, out=self.ybuf[0])
            ops.nms_batched(ys, out=self.outs[0], **self.kw)
            torch.cuda.synchronize(self.device)
            self._g_first = [self._capture(p, nms_of=None) for p in (0, 1)]              # decode only (first step)
            self._g_step = [self._capture(p, nms_of=p if not self.overlap else 1 - p) for p in (0, 1)]
            self._g_flush = [self._capture(None, nms_of=p) for p in (0, 1)]              # NMS only (drain)
            if self.delivery is not None:
                # steady state (step k >= 3): the step graph also carries, on a third branch, this rank's side of the
                # delivery -- writers push batch k-2, rank dst collects batch k-3; the first steps of a run, instrumented
                # steps and the flush use the plain graphs above plus these two small ones
                self._g_full = [self._capture(p, nms_of=1 - p, side=True) for p in (0, 1)]
                self._g_flush_full = [self._capture(None, nms_of=p, side=True) for p in (0, 1)]
                self._g_push = [self._capture_side(p, "push") for p in (0, 1)]
                self._g_collect = [self._capture_side(p, "collect") for p in (0, 1)]
            self.timed: List[Tuple[torch.cuda.CUDAGraph, list]] = []
            # ``timed_steps`` (optional, same length): the step index each instrumented slot is used at; with a delivery,
            # slots used at steps >= 3 carry the side branch like the steady-state graph does
            self.timed_parity = [int(p) & 1 for p in timed_parities]
            self.timed_has_side = [self.delivery is not None and _SIDE == "piggyback" and i < len(timed_steps) and int(timed_steps[i]) >= 3
                                   for i in range(len(self.timed_parity))]
            for p, side in zip(self.timed_parity, self.timed_has_side):
                self.timed.append(self._capture_timed(p, side))
            torch.cuda.synchronize(self.device)

    # ------------------------------------------------------------------ graph construction
    def _decode(self, p, pdl: bool = False):
        if not pdl:
            return ops.decode_heads(self.heads, self.strides, out=self.ybuf[p])
        from . import _lib

        _lib.debug_set("decode_pdl", 1)  # thread-local launch option of the C ABI (include/cerb_post.h)
        try:
            return ops.decode_heads(self.heads, self.strides, out=self.ybuf[p])
        finally:
            _lib.debug_set("decode_pdl", 0)

    def _nms(self, p, piggyback: bool = False):
        T = len(self.heads)
        ys = self.ybuf[p][:T]
        ops._publish_summaries(ys, self.ybuf[p][T:])  # the summary of a static buffer describes whatever decode wrote last
        deliver = self.delivery.nms_deliver_args(p, piggyback) if self.delivery is not None else None
        return ops.nms_batched(ys, out=self.outs[p], deliver=deliver, **self.kw)

    def _capture_side(self, slot: int, what: str):
        """A graph holding only this rank's delivery kernel for ``slot`` (None where that side does not exist here)."""
        dv = self.delivery
        on_dst = dv.rank == dv.dst
        if (what == "collect") != on_dst or (what == "push" and dv.direct):
            return None
        g = torch.cuda.CUDAGraph()
        self.sa.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.sa):
            with torch.cuda.graph(g, stream=self.sa):
                dv.collect(slot) if on_dst else dv.push(slot)
        torch.cuda.current_stream(self.device).wait_stream(self.sa)
        return g

    def _capture(self, dec: Optional[int], nms_of: Optional[int], side: bool = False):
        """``side`` (in-graph delivery, steady state): the NMS launch also carries this rank's side of the delivery of an
        earlier batch (``PeerDelivery.nms_deliver_args(slot, piggyback=True)``): a writer's launch for batch j pushes
        batch j-1, rank dst's launch for batch j takes batch j-2.  CERB_SIDE=branch (tools/ A/B) puts the stand-alone
        kernels on a third branch instead."""
        dv = self.delivery
        standalone = side and _SIDE in _STANDALONE and (dv.rank == dv.dst or not dv.direct)
        piggy = side and not standalone

        def side_kernel():
            if dv.rank == dv.dst:
                dv.collect(1 - dec)
            else:
                dv.push(dec)

        g = torch.cuda.CUDAGraph()
        self.sa.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.sa):
            with torch.cuda.graph(g, stream=self.sa):
                if self.overlap and nms_of is not None and dec is not None and _SCHEDULE == "pdl" and not standalone:
                    self._nms(nms_of, piggy)         # NMS of the previous batch: releases its dependents at entry
                    self._decode(dec, pdl=True)      # runs beside it; reads nothing it writes, so it never waits for it
                elif self.overlap or dec is None or nms_of is None:
                    if nms_of is not None and dec is not None:
                        self.sb.wait_stream(self.sa)
                        if standalone and _SIDE == "branch3":      # third branch, created first
                            self.sc.wait_stream(self.sa)
                            with torch.cuda.stream(self.sc):
                                side_kernel()
                        if standalone and _SIDE == "last3":        # third branch, created after the two big kernels
                            self.sc.wait_stream(self.sa)
                        with torch.cuda.stream(self.sb):
                            if standalone and _SIDE == "pre_nms":
                                side_kernel()
                            self._nms(nms_of, piggy)
                            if standalone and _SIDE == "post_nms":
                                side_kernel()
                        self._decode(dec)
                        if standalone and _SIDE == "post_decode":
                            side_kernel()
                        if standalone and _SIDE == "last3":
                            with torch.cuda.stream(self.sc):
                                side_kernel()
                        self.sa.wait_stream(self.sb)
                        if standalone and _SIDE in ("branch3", "last3"):
                            self.sa.wait_stream(self.sc)
                    elif dec is not None:
                        self._decode(dec)
                    else:
                        self._nms(nms_of, piggy)
                else:  # serial: decode -> NMS of the SAME batch (the NMS kernel starts under programmatic dependent launch)
                    self._decode(dec)
                    self._nms(nms_of)
        torch.cuda.current_stream(self.device).wait_stream(self.sa)
        return g

    def _capture_timed(self, p: int, side: bool = False):
        """Instrumented step: the same two launches as a normal step (decode of this batch, NMS of the previous one) in
        SERIAL order with timing events recorded by graph nodes:  E0 ; decode ; {E1 on a side branch} ; NMS ; E2.
        E1 hangs off the decode kernel on a second stream (which waits for the launching stream first), so the NMS kernel
        keeps its programmatic (early-launch) edge to the decode kernel; E0..E1 is the decode kernel alone on the GPU,
        E1..E2 the NMS kernel.  (With E1 on the launching stream itself the decode reads 1 us shorter and the NMS 5.5 us
        longer -- it loses the early launch -- which costs the driver's 20-step run 3 % of its value: gpurun_out/call_v3.)"""
        ev = [torch.cuda.Event(enable_timing=True, external=True) for _ in range(3)]
        g = torch.cuda.CUDAGraph()
        self.sa.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self.sa):
            with torch.cuda.graph(g, stream=self.sa):
                ev[0].record(self.sa)
                self._decode(p)
                self.sb.wait_stream(self.sa)
                ev[1].record(self.sb)
                self._nms(1 - p, side)  # (side: the launch carries this rank's delivery work, as in the steady-state graph)
                ev[2].record(self.sa)
                self.sa.wait_stream(self.sb)
        torch.cuda.current_stream(self.device).wait_stream(self.sa)
        return g, ev

    # ------------------------------------------------------------------ running
    def _deliver_side(self, k: int) -> None:
        """This rank's delivery work that belongs to step ``k`` -- push batch k-2 (writers), collect batch k-3 (dst) -- as
        stand-alone kernels (the first steps of a run, instrumented steps without the piggyback, CERB_SIDE=after)."""
        dv = self.delivery
        if _SIDE == "off":
            return
        if dv.rank == dv.dst:
            if k >= 3:
                self._g_collect[(k - 3) & 1].replay()
                self._collected = k - 2
        elif k >= 2:
            if self._g_push[0] is not None:
                self._g_push[(k - 2) & 1].replay()
            self._pushed = k - 1

    def step(self, timed: Optional[int] = None) -> Optional[int]:
        """Issue one pipeline step on the current stream.  Returns the index of the ``outs`` buffer that this step's
        NMS fills (the detections of the PREVIOUS batch; of this batch when ``overlap=False``), or None on the first
        step of an overlapped pipeline."""
        k = self.k
        p = k & 1
        self.k += 1
        if not self.overlap:
            self._g_step[p].replay()
            return p
        if self.pending is None:
            self._g_first[p].replay()
            self.pending = p
            self._pushed = self._collected = 0  # batches of this run already pushed (writer) / collected (dst)
            return None
        in_launch = self.delivery is not None and k >= 3 and (_SIDE == "piggyback" or _SIDE in _STANDALONE)
        if timed is not None:
            g, _ = self.timed[timed]
            if self.timed_parity[timed] != p:
                raise ValueError("timed slot parity does not match the step parity")
            g.replay()
            in_launch = in_launch and self.timed_has_side[timed]
        elif in_launch:
            self._g_full[p].replay()
        else:
            self._g_step[p].replay()
        if self.delivery is not None:
            if in_launch:  # the step's launches did it: push k-2 / collect k-3
                self._pushed, self._collected = k - 1, k - 2
            else:
                self._deliver_side(k)
        done, self.pending = self.pending, p
        return done

    def flush(self) -> Optional[int]:
        """NMS of the last decoded batch (end of a stream of batches), and -- with a delivery -- everything of this run that
        is still on its way to rank dst.  Returns the ``outs`` index of the last batch."""
        if not self.overlap or self.pending is None:
            return None
        p, self.pending = self.pending, None
        n = self.k  # steps of this run = batches 0 .. n-1
        dv = self.delivery
        if dv is not None and n >= 3 and _SIDE == "piggyback":
            self._g_flush_full[p].replay()  # the last NMS launch carries push n-2 / collect n-3 like every other one
            self._pushed, self._collected = n - 1, n - 2
        else:
            self._g_flush[p].replay()
        if dv is not None and _SIDE != "off":
            if dv.rank == dv.dst:
                for j in range(self._collected, n):
                    self._g_collect[j & 1].replay()
                self._collected = n
            else:
                for j in range(self._pushed, n):
                    if self._g_push[0] is not None:
                        self._g_push[j & 1].replay()
                self._pushed = n
        return p

    def timed_ms(self, i: int) -> Tuple[float, float]:
        """(NMS ms, decode ms) of the last replay of instrumented slot ``i`` (synchronise first)."""
        _, ev = self.timed[i]
        return ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[1])
