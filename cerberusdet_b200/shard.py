"""Image sharding across the GPUs of one box and the single exchange of the path.

Every (image, task) segment is independent in decode and NMS (reference
utils/general.py:424 loops over images; tasks are separate calls at
cerberusdet_inference.py:125-135), so a batch shards by image with no data-path
collective.  The only exchange is that the padded detections
``[T, B_loc, max_det, 6]`` + counts ``[T, B_loc]`` of every rank reach rank 0: through
peer-mapped memory over NVLink with a flag / acknowledge hand-shake the kernels run
themselves (``PeerDelivery``), or one ``dist.gather`` per batch (``GatherDelivery``:
NCCL fallback, gloo in the CPU tests).
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(n_images: int, rank: int, world: int) -> range:
    """Contiguous block of images owned by ``rank``; remainder images go to the low ranks."""
    base, rem = divmod(n_images, world)
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))


def shard_sizes(n_images: int, world: int) -> List[int]:
    return [len(shard_range(n_images, r, world)) for r in range(world)]


def gather_detections(
    dets: torch.Tensor, counts: torch.Tensor, dst: int = 0, n_images: Optional[int] = None, group=None
) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Gather per-rank ``dets[T, B_loc, max_det, 6]`` / ``counts[T, B_loc]`` to ``dst``.

    Returns ``(dets[T, B, max_det, 6], counts[T, B])`` on ``dst`` (image order = rank
    order = global image order) and ``(None, None)`` elsewhere.  With ``n_images`` given,
    ranks may hold unequal shards (``shard_range``): shards are padded to the largest one
    for the collective and the padding is dropped on ``dst``.
    """
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return dets, counts
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    T, b_loc = counts.shape
    sizes = shard_sizes(n_images, world) if n_images is not None else [b_loc] * world
    b_max = max(sizes)
    if b_loc != sizes[rank]:
        raise ValueError(f"rank {rank} holds {b_loc} images, shard_range says {sizes[rank]}")
    if b_loc < b_max:  # pad the tail shard; masked by counts == 0
        pad_d = dets.new_zeros((T, b_max - b_loc) + tuple(dets.shape[2:]))
        pad_c = counts.new_zeros((T, b_max - b_loc))
        dets, counts = torch.cat((dets, pad_d), 1), torch.cat((counts, pad_c), 1)
    dets, counts = dets.contiguous(), counts.contiguous()
    if rank == dst:
        d_list = [torch.empty_like(dets) for _ in range(world)]
        c_list = [torch.empty_like(counts) for _ in range(world)]
    else:
        d_list = c_list = None
    dist.gather(dets, d_list, dst=dst, group=group)
    dist.gather(counts, c_list, dst=dst, group=group)
    if rank != dst:
        return None, None
    return (torch.cat([d[:, :n] for d, n in zip(d_list, sizes)], 1),
            torch.cat([c[:, :n] for c, n in zip(c_list, sizes)], 1))


class DetectionGatherer:
    """Persistent buffers for the per-batch gather: the NMS kernel writes ``dets`` and ``counts`` straight
    into one packed buffer per rank, so a batch needs ONE collective (``dist.gather`` of
    ``T*B*(max_det*6+1)`` 32-bit words) and no per-step allocation.  ``launch()`` is asynchronous; the
    gathered tensors on ``dst`` are valid after ``wait()``.  Equal shards only (pad the batch otherwise,
    or use ``gather_detections``)."""

    def __init__(self, T: int, b_loc: int, max_det: int, device, dst: int = 0, group=None):
        self.T, self.b_loc, self.max_det, self.dst, self.group = T, b_loc, max_det, dst, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        n_d, n_c = T * b_loc * max_det * 6, T * b_loc
        self.local = torch.empty(n_d + n_c, dtype=torch.float32, device=device)
        self.dets = self.local[:n_d].view(T, b_loc, max_det, 6)
        self.counts = self.local[n_d:].view(torch.int32).view(T, b_loc)
        self.all = None
        if self.rank == dst and self.world > 1:
            self.all = torch.empty((self.world, n_d + n_c), dtype=torch.float32, device=device)
            self._views = [self.all[r] for r in range(self.world)]
        self._n_d = n_d
        self._work = None

    @property
    def out(self):
        return self.dets, self.counts

    def launch(self):
        if self.world > 1:
            self._work = dist.gather(self.local, self._views if self.rank == self.dst else None, dst=self.dst,
                                     group=self.group, async_op=True)
        return self._work

    def wait(self):
        if self._work is not None:
            self._work.wait()
            self._work = None

    def result(self) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """``(dets[T, world*B_loc, max_det, 6], counts[T, world*B_loc])`` on ``dst`` in global image order."""
        self.wait()
        if self.world == 1:
            return self.dets, self.counts
        if self.rank != self.dst:
            return None, None
        d = self.all[:, : self._n_d].view(self.world, self.T, self.b_loc, self.max_det, 6)
        c = self.all[:, self._n_d :].view(torch.int32).view(self.world, self.T, self.b_loc)
        return (d.permute(1, 0, 2, 3, 4).reshape(self.T, self.world * self.b_loc, self.max_det, 6),
                c.permute(1, 0, 2).reshape(self.T, self.world * self.b_loc))


# ------------------------------------------------------------------------------------------------ per-batch delivery to rank 0
class GatherDelivery:
    """Per-batch delivery of the padded detections to ``dst`` by one asynchronous ``dist.gather`` per batch
    (``DetectionGatherer``), two alternating buffers.  Works on every backend (NCCL on GPUs, gloo in the CPU tests)."""

    kind = "one asynchronous gather per batch (torch.distributed)"
    in_graph = False

    def __init__(self, T: int, b_loc: int, max_det: int, device, dst: int = 0, group=None):
        self.g = [DetectionGatherer(T, b_loc, max_det, device, dst=dst, group=group) for _ in range(2)]
        self.outs = [g.out for g in self.g]

    def before_write(self, slot: int) -> None:
        """Call before a kernel overwrites ``outs[slot]``: the previous batch in that slot must have left."""
        self.g[slot].wait()

    def after_write(self, slot: int) -> None:
        """Call after the kernel that filled ``outs[slot]`` was enqueued: starts the delivery of that batch."""
        self.g[slot].launch()

    def drain(self) -> None:
        for g in self.g:
            g.wait()

    def result(self, slot: int):
        return self.g[slot].result()

    def nms_deliver_args(self, slot: int):
        return None

    def collect(self, slot: int) -> None:
        pass

    def push(self, slot: int) -> None:
        pass


class PeerDelivery:
    """Per-batch delivery WITHOUT a collective: every rank pushes the padded detections of its batch straight into rank
    ``dst``'s memory over NVLink (``torch.distributed._symmetric_memory``: peer-mapped device memory, region (slot, r) of
    dst's buffer) and the hand-shake is a pair of 32-bit words per slot, moved by the kernels themselves:

      * writer r: ``push(slot)`` = ``cerb_deliver_push`` -- a small kernel that waits until dst has acknowledged the batch
        that was in the slot, copies the packed rows with 128-bit stores, orders them (GPU-scope release per CTA, one
        system-scope release by the last CTA) and publishes the slot's batch count in dst's ``flags[slot][r]``;
      * dst: ``collect(slot)`` = ``cerb_deliver_collect`` -- one 32-thread kernel: thread r waits for rank r's flag and
        stores the acknowledgement into rank r's ``ack[slot]``.

    The NMS kernel writes LOCAL memory exactly as on one GPU.  In steady state neither side is a kernel of its own: the
    NEXT NMS launch carries them (``nms_deliver_args(slot, piggyback=True)`` -> ``cerb_nms_deliver``) in a few extra CTAs
    beside its segment CTAs: a writer's push the previous batch and publish the flag, one on dst does the collect.  The step graph keeps the shape it has on one GPU (a third graph
    branch, however small its kernel, costs the decode / NMS overlap: +13 us per step, profiles/r02_multi_gpu.md), the
    NVLink round trips of the fences are on nobody's critical path, and a step stays one graph replay on every rank.
    ``push`` / ``collect`` as stand-alone kernels serve the first and last batches of a run.  No NCCL kernel takes SMs
    from the decode, no stream waits for a gather, nothing on the host scales with the number of ranks.

    ``direct=True`` is the variant without the staging copy: ``outs[slot]`` ARE dst's memory and the NMS kernel runs the
    writer's side of the hand-shake itself (``cerb_nms_deliver``); its fences then sit at the end of the NMS kernel
    (+7 us per step at N=2, profiles/r02_multi_gpu.md), so it is not the default.

    Control words (uint32, after the data regions of the symmetric buffer; every rank allocates the same layout):
    ``flags[slot][r]`` at ``ctrl + 16*slot + r`` (used on dst), ``ack[slot]`` at ``ctrl + 32 + slot`` (used on writers).
    """

    in_graph = True
    MAX_WORLD = 16

    def __init__(self, T: int, b_loc: int, max_det: int, device, dst: int = 0, group=None, direct: bool = False):
        import torch.distributed._symmetric_memory as symm_mem

        group = group if group is not None else dist.group.WORLD
        self.world, self.rank, self.dst = dist.get_world_size(group), dist.get_rank(group), dst
        if self.world > self.MAX_WORLD:
            raise ValueError(f"PeerDelivery supports at most {self.MAX_WORLD} ranks")
        self.direct = bool(direct)
        self.kind = ("rows pushed into rank 0's peer-mapped symmetric memory over NVLink by " +
                     ("the NMS kernel as it produces them (cerb_nms_deliver, direct form)" if self.direct else
                      "the NEXT NMS launch at its start (cerb_nms_deliver, piggyback form: staged locally, 128-bit stores)") +
                     "; flag / acknowledge words instead of a collective, published / taken by the same launches; "
                     "no extra node in the step graphs")
        self.T, self.b_loc, self.max_det = T, b_loc, max_det
        self.n_d, self.n_c = T * b_loc * max_det * 6, T * b_loc
        self.n = (self.n_d + self.n_c + 63) // 64 * 64  # words per (slot, rank) region, 256-byte aligned
        self.ctrl = 2 * self.world * self.n             # first control word
        try:
            symm_mem.enable_symm_mem_for_group(group.group_name)
        except Exception:
            pass  # newer builds enable it inside rendezvous()
        self.local = symm_mem.empty(self.ctrl + 64, dtype=torch.float32, device=device)
        self.local[self.ctrl :].zero_()
        self.hdl = symm_mem.rendezvous(self.local, group)
        on_dst = self.rank == dst
        # local protocol state: seq[2], done[2] (writers), collected[2] (dst)
        self.state = torch.zeros(8, dtype=torch.int32, device=device)
        base = self.local.data_ptr() + 4 * self.ctrl
        self.outs, self._remote, self._stage = [], [None, None], [None, None]
        self._words = [None, None]    # writers: (flag_remote, ack_local, seq_local, done_local) per slot
        self._collect = [None, None]  # dst: (flags_local, [ack_remote per rank], collected_local) per slot
        self._peers = []              # keep the mapped views alive
        for slot in range(2):
            off = (slot * self.world + self.rank) * self.n
            if on_dst:
                region = self.local[off : off + self.n]
            else:
                self._remote[slot] = self.hdl.get_buffer(dst, (self.n,), torch.float32, off)  # rank dst's memory, mapped here
                if self.direct:
                    region = self._remote[slot]
                else:
                    region = self._stage[slot] = torch.zeros(self.n, dtype=torch.float32, device=device)
            self.outs.append((region[: self.n_d].view(T, b_loc, max_det, 6),
                              region[self.n_d : self.n_d + self.n_c].view(torch.int32).view(T, b_loc)))
            if not on_dst:
                flag = self.hdl.get_buffer(dst, (1,), torch.float32, self.ctrl + 16 * slot + self.rank)
                self._peers.append(flag)
                self._words[slot] = (flag.data_ptr(), base + 4 * (32 + slot), self.state.data_ptr() + 4 * slot,
                                     self.state.data_ptr() + 4 * (2 + slot))
            else:
                acks = []
                for r in range(self.world):
                    if r == dst:
                        acks.append(None)
                    else:
                        a = self.hdl.get_buffer(r, (1,), torch.float32, self.ctrl + 32 + slot)
                        self._peers.append(a)
                        acks.append(a.data_ptr())
                self._collect[slot] = (base + 4 * 16 * slot, acks, self.state.data_ptr() + 4 * (4 + slot))
        torch.cuda.synchronize(device)
        self.hdl.barrier(channel=7)

    def nms_deliver_args(self, slot: int, piggyback: bool = False):
        """``deliver=`` argument (a ``_lib.Delivery`` or None) of ``ops.nms_batched`` for the NMS launch that fills
        ``outs[slot]``.  ``piggyback``: the launch also does this rank's side of the delivery of an EARLIER batch -- a
        writer pushes the batch it left in the other slot's staging by its previous launch, rank dst takes the batch the
        writers pushed into this slot's parity during the previous step (see ``PostHeadPipeline``).  ``direct`` mode: a
        writer's launch stores into dst's memory and signals for its own batch."""
        from . import _lib

        on_dst = self.rank == self.dst
        if self.direct:
            if on_dst:
                return self._collect_struct(slot) if piggyback else None
            d = _lib.Delivery()
            d.flag_remote, d.ack_local, d.seq_local, d.done_local = self._words[slot]
            return d
        if not piggyback:
            return None
        if on_dst:
            return self._collect_struct(slot)
        prev = 1 - slot
        d = _lib.Delivery()
        d.push_src, d.push_dst, d.push_words = self._stage[prev].data_ptr(), self._remote[prev].data_ptr(), self.n
        d.flag_remote, d.ack_local, d.seq_local, d.done_local = self._words[prev]
        return d

    def _collect_struct(self, slot: int):
        from . import _lib

        flags, acks, collected = self._collect[slot]
        d = _lib.Delivery()
        d.collect_flags, d.collect_count, d.world, d.dst = flags, collected, self.world, self.dst
        for r, a in enumerate(acks):
            d.collect_ack[r] = a
        return d

    def push(self, slot: int) -> None:
        """Writer: enqueue (current stream) the kernel that moves the batch in ``outs[slot]`` into dst's slot and signals
        it.  A no-op on dst and in ``direct`` mode."""
        if self.rank == self.dst or self.direct:
            return
        from . import _lib, ops

        ops._launch(_lib.load().cerb_deliver_push, self.local.device, self._stage[slot].data_ptr(), self._remote[slot].data_ptr(),
                    self.n, *self._words[slot])

    def collect(self, slot: int) -> None:
        """dst: enqueue (current stream) the kernel that waits for every rank's batch in ``slot`` and acknowledges it.
        A no-op on the other ranks."""
        if self.rank != self.dst:
            return
        from . import _lib, ops

        flags, acks, collected = self._collect[slot]
        ops._launch(_lib.load().cerb_deliver_collect, self.local.device, flags, _lib.ptr_array(acks), collected, self.world, self.dst)

    # the hand-shake lives in kernels the pipeline enqueues: nothing to do around a write
    def before_write(self, slot: int) -> None:
        pass

    def after_write(self, slot: int) -> None:
        pass

    def drain(self) -> None:
        pass

    def result(self, slot: int):
        """``(dets[T, world*B_loc, max_det, 6], counts[T, world*B_loc])`` on ``dst`` (after the slot's ``collect`` has run
        and the device was synchronised), ``(None, None)`` elsewhere."""
        if self.rank != self.dst:
            return None, None
        reg = self.local[slot * self.world * self.n : (slot + 1) * self.world * self.n].view(self.world, self.n)
        d = reg[:, : self.n_d].reshape(self.world, self.T, self.b_loc, self.max_det, 6)
        c = reg[:, self.n_d : self.n_d + self.n_c].contiguous().view(torch.int32).view(self.world, self.T, self.b_loc)
        return (d.permute(1, 0, 2, 3, 4).reshape(self.T, self.world * self.b_loc, self.max_det, 6),
                c.permute(1, 0, 2).reshape(self.T, self.world * self.b_loc))


def make_delivery(T: int, b_loc: int, max_det: int, device, dst: int = 0, group=None, prefer_peer: bool = True):
    """The per-batch delivery to rank ``dst``: peer-mapped symmetric memory on CUDA when every rank can set it up
    (all ranks agree, so nobody is left in a collective alone), else the gather."""
    import os

    mode = os.environ.get("CERB_DELIVERY", "peer")
    want_peer = prefer_peer and torch.device(device).type == "cuda" and mode != "gather"
    if want_peer:
        ok, deliv = 1, None
        try:
            deliv = PeerDelivery(T, b_loc, max_det, device, dst=dst, group=group, direct=(mode == "peer_direct"))
        except Exception as exc:  # pragma: no cover - depends on the box / torch build
            import sys

            print(f"[cerberusdet_b200.shard] symmetric memory unavailable ({type(exc).__name__}: {exc}); using the gather", file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 1:
            return deliv
    return GatherDelivery(T, b_loc, max_det, device, dst=dst, group=group)
