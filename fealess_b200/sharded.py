"""Template-sharded matching across GPUs (SURVEY.md 8e): one process per GPU, ``torch.distributed`` for the plumbing.

Templates are independent units (the ``matchClass`` loop, reference linemod/linemod.cpp:1458), so they are dealt
round-robin by global template index; every rank runs the (cheap) front end on the whole frame redundantly and
``matchClass`` on its shard.  The only exchange step of the path is the candidate list: ONE all-gather per frame of a
fixed-capacity block ``[header | records]`` (20-byte ``fl_match_t`` records, count in the header), after which every rank
sorts + prunes the union redundantly (``fl_sort_unique_device``), so no broadcast is needed and the result is
shard-invariant.

The block packing / gathering / splitting helpers work on CPU tensors with the ``gloo`` backend too; that is how the
N > 1 host logic is tested without GPUs (tests/test_sharding_gloo.py).
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

from . import RECO_MAX_HYP, synth

RECORD_INTS = 5  # fl_match_t = 5 x int32-sized fields


def shard_indices(n_templates: int, rank: int, world: int) -> np.ndarray:
    """Global template indices owned by ``rank`` (round-robin balances the data-dependent candidate counts)."""
    return np.arange(rank, n_templates, world, dtype=np.int64)


def shard_template_set(tset: "synth.TemplateSet", rank: int, world: int) -> Tuple["synth.TemplateSet", np.ndarray]:
    """Returns (shard, template_ids): ``template_ids[i]`` is the GLOBAL per-class template_id of shard template i, to be
    installed with ``Handle.set_template_ids`` so gathered candidates carry shard-invariant ids."""
    idx = shard_indices(tset.n_templates, rank, world)
    first = {}
    for t in range(tset.n_templates):
        first.setdefault(int(tset.class_of[t]), t)
    gids = np.array([t - first[int(tset.class_of[t])] for t in idx], np.int32)
    return tset.subset(idx.tolist()), gids


def block_ints(capacity: int) -> int:
    return (capacity + 1) * RECORD_INTS


def pack_block(block, records, count) -> None:
    """``block``: int32 tensor [(capacity+1)*5]; writes the count into the header record.  ``records`` is a view of
    block[5:] that the producer already filled (the CUDA path writes candidates straight into it)."""
    block[0] = count


def records_view(block):
    return block[RECORD_INTS:]


def gather_blocks(block, world: int, group=None):
    """One collective per frame: all-gather of the fixed-size blocks.  Returns an int32 tensor [world, capacity+1, 5]."""
    import torch
    import torch.distributed as dist
    out = torch.empty((world,) + tuple(block.shape), dtype=block.dtype, device=block.device)
    if world == 1 or not dist.is_initialized():
        out[0].copy_(block)
    else:
        dist.all_gather_into_tensor(out.view(-1), block.contiguous(), group=group)
    return out.view(world, -1, RECORD_INTS)


def split_blocks(gathered) -> Tuple["object", "object"]:
    """(counts[world] int32 contiguous, records[world, capacity, 5]) views/copies of a gathered tensor."""
    counts = gathered[:, 0, 0].contiguous()
    return counts, gathered[:, 1:, :]


def merge_on_host(gathered_np: np.ndarray) -> np.ndarray:
    """Reference merge used by the CPU tests: concatenate live records of all blocks -> structured array (unsorted)."""
    from . import MATCH_DTYPE
    recs = []
    for b in gathered_np:
        n = int(b[0, 0])
        r = np.ascontiguousarray(b[1:1 + n]).view(MATCH_DTYPE).reshape(-1)
        recs.append(r[r["template_id"] >= 0])
    return np.concatenate(recs) if recs else np.zeros(0, MATCH_DTYPE)


class ShardedMatcher:
    """One rank of a template-sharded detector.  ``match_device`` = front end + matchClass on the local shard, exchange of
    the candidate blocks, sort + unique of the union on every rank.

    exchange = "p2p" (default on a multi-GPU job): every rank's exchange buffer is a torch symmetric-memory allocation
    mapped into all processes; the library's own sort kernel pushes the local block into every peer over NVLink, signals,
    waits for the peers and merges (``fl_exchange_sort_unique_device``) - ONE kernel, no collective-library call on the data
    path.  exchange = "nccl": one ``all_gather_into_tensor`` of fixed-size blocks followed by
    ``fl_sort_unique_blocks_device`` (the block layout ``[header | records]`` is consumed as it is)."""

    def __init__(self, handle, tset, rank: int, world: int, capacity: int = 2048, device=None, exchange: str = "auto"):
        import torch
        import torch.distributed as dist
        self.h, self.rank, self.world, self.cap = handle, rank, world, capacity
        shard, gids = shard_template_set(tset, rank, world)
        handle.upload_templates(shard)
        handle.set_template_ids(gids)
        self.n_local = shard.n_templates
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.block = torch.zeros(block_ints(capacity), dtype=torch.int32, device=dev)
        self.gathered = torch.zeros(world * block_ints(capacity), dtype=torch.int32, device=dev)
        self.stream = torch.cuda.ExternalStream(handle.stream_ptr(), device=dev)
        self._torch = torch
        self.epoch = 0
        self.exchange = "nccl"
        self.exchange_error = None
        if exchange in ("auto", "p2p") and world > 1 and dist.is_initialized() and world <= 8:
            try:
                import torch.distributed._symmetric_memory as symm_mem
                from . import lib
                nbytes = int(lib().fl_exchange_buffer_bytes(world, capacity))
                self._xbuf = symm_mem.empty(nbytes, dtype=torch.uint8, device=dev)
                self._xhdl = symm_mem.rendezvous(self._xbuf, dist.group.WORLD)
                self._xbuf.zero_()
                torch.cuda.synchronize()
                dist.barrier()
                import ctypes
                self._peers = (ctypes.c_void_p * world)(*[int(p) for p in self._xhdl.buffer_ptrs])   # built once: the per-frame calls pass it as is
                self._block_ptr = self.block.data_ptr()
                self.exchange = "p2p"
            except Exception as e:  # noqa: BLE001  (no peer mapping available: fall back to the collective)
                self.exchange_error = repr(e)
                if exchange == "p2p":
                    raise
            # all ranks must agree on the mode
            ok = torch.tensor([1 if self.exchange == "p2p" else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                self.exchange = "nccl"

    def match_device_async(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, masks=None) -> bool:
        """One frame, enqueue only: the local match and (p2p exchange) the exchange + merge kernel go onto the handle's stream.
        Returns True when ``match_wait`` is all that is left (p2p); with the NCCL exchange the collective and the merge are
        issued by ``match_wait``.  ``masks``: None, or one device pointer (0 = unmasked) per modality, valid until ``match_wait``."""
        if self.world == 1:                                      # nothing to exchange: the plain three-launch frame
            self.h.match_device_async(d_bgr, d_depth, W, H, threshold, masks=masks)
            return True
        if self.exchange == "p2p":
            # front end + matchClass, then ONE launch: refinement, push to the peers, wait, sort of the union
            self.epoch += 1
            self.h.match_shard_exchange_device_async(d_bgr, d_depth, W, H, threshold, self.rank, self.world, self._peers, self.cap,
                                                     self._block_ptr, self.epoch, masks=masks)
            return True
        recs = records_view(self.block)
        # the count lives in the header record of the block, so the candidates + count travel together
        self.h.match_shard_device(d_bgr, d_depth, W, H, threshold, recs.data_ptr(), self.cap, self.block.data_ptr(), masks=masks)
        return False

    def match_host_async(self, bgr: np.ndarray, depth: np.ndarray, threshold: float, masks=None) -> bool:
        """``match_device_async`` for a frame in host memory: with the p2p exchange ONE C call uploads the frame and enqueues the
        local match and the exchange (fl_match_shard_exchange_masked_async); with the NCCL exchange the frame is copied into the rank's
        device buffers first.  ``masks``: as in ``Handle.match`` (numpy arrays)."""
        H, W = depth.shape[:2]
        if self.world == 1:
            self._host_frame = (bgr, depth)
            self.h.match_async(bgr, depth, threshold, masks=masks)
            return True
        if self.exchange == "p2p":
            self.epoch += 1
            self._host_frame = (bgr, depth)                     # page-locked buffers are read by DMA until match_wait
            self.h.match_shard_exchange_async(bgr, depth, threshold, self.rank, self.world, self._peers, self.cap, self._block_ptr, self.epoch,
                                              masks=masks)
            return True
        torch = self._torch
        if getattr(self, "_d_in", None) is None or self._d_in[0].numel() != H * W * 3:
            self._d_in = (torch.empty(H * W * 3, dtype=torch.uint8, device=self.block.device), torch.empty(H * W, dtype=torch.int16, device=self.block.device))
        # the copies go on torch's current stream and the handle's stream waits for them: torch remembers on which stream a
        # page-locked block was used and records an event there when the block is freed - that must not be a handle's stream,
        # which may be gone by then
        cur = torch.cuda.current_stream()
        self._d_in[0].copy_(torch.from_numpy(bgr).view(-1), non_blocking=True)
        self._d_in[1].copy_(torch.from_numpy(depth.view(np.int16)).view(-1), non_blocking=True)
        d_masks = None
        if masks:
            from . import host_masks
            _, keep = host_masks(masks, self.h.M, W, H)
            self._d_masks = [None if k is None else torch.from_numpy(k).to(self.block.device, non_blocking=True) for k in keep]
            d_masks = [0 if t is None else t.data_ptr() for t in self._d_masks]
        self.stream.wait_stream(cur)
        return self.match_device_async(self._d_in[0].data_ptr(), self._d_in[1].data_ptr(), W, H, threshold, masks=d_masks)

    def match_wait(self) -> None:
        torch = self._torch
        import torch.distributed as dist
        if self.exchange == "p2p" or self.world == 1:
            self.h.match_wait()
            return
        with torch.cuda.stream(self.stream):
            if self.world == 1 or not dist.is_initialized():
                self.gathered.copy_(self.block)
            else:
                dist.all_gather_into_tensor(self.gathered, self.block)
        self.h.sort_unique_blocks_device(self.gathered.data_ptr(), self.world, self.cap)

    def match_device(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float) -> None:
        """One frame: the local match, the exchange and the merge; returns when the merged match list is ready (``fetch``)."""
        self.match_device_async(d_bgr, d_depth, W, H, threshold)
        self.match_wait()

    def fetch(self) -> np.ndarray:
        return self.h.match_fetch()

    def close(self) -> None:
        """Releases the matcher's device tensors, THEN the handle: torch's allocator notes on which streams a tensor was used and
        records an event there when the tensor is freed - the handle's stream must still exist at that point."""
        if self.h is None:
            return
        self._torch.cuda.synchronize()
        self.block = self.gathered = None
        self._d_in = self._d_masks = None
        self._host_frame = None
        self._xhdl = None
        self._xbuf = None
        self.stream = None
        self._torch.cuda.synchronize()
        self.h.close()
        self.h = None


class ShardedPipe:
    """Several frames in flight on every rank of a template-sharded detector: ``depth`` ShardedMatchers (each with its own handle,
    stream, candidate block and exchange buffer), frames dealt round-robin, lists collected in submission order.  Every rank has
    to submit and collect the same sequence of frames (frame i's exchange pairs slot i % depth of all ranks); a kernel that waits
    for a peer's block holds one CTA, so the other slots' frames keep the GPU busy meanwhile.  With one rank this is fl_pipe's
    schedule driven from Python (the bench uses it at N = 1 too, so that every N runs the same loop)."""

    def __init__(self, make_handle, tset, rank: int, world: int, depth: int = 4, capacity: int = 2048, device=None, exchange: str = "auto"):
        self.depth = int(depth)
        self.slots = [ShardedMatcher(make_handle(), tset, rank, world, capacity=capacity, device=device, exchange=exchange) for _ in range(self.depth)]
        modes = {s.exchange for s in self.slots}
        if len(modes) != 1:
            raise RuntimeError("the slots of a ShardedPipe disagree on the exchange mode: %s" % sorted(modes))
        self.exchange = self.slots[0].exchange
        self.submitted = self.collected = 0

    def in_flight(self) -> int:
        return self.submitted - self.collected

    def _next_slot(self) -> "ShardedMatcher":
        if self.in_flight() >= self.depth:
            raise RuntimeError("ShardedPipe: %d frames in flight already - collect one first" % self.depth)
        s = self.slots[self.submitted % self.depth]
        self.submitted += 1
        return s

    def submit_device(self, d_bgr: int, d_depth: int, W: int, H: int, threshold: float, masks=None) -> "ShardedMatcher":
        s = self._next_slot()
        s.match_device_async(d_bgr, d_depth, W, H, threshold, masks=masks)
        return s

    def submit_host(self, bgr: np.ndarray, depth: np.ndarray, threshold: float, masks=None) -> "ShardedMatcher":
        s = self._next_slot()
        s.match_host_async(bgr, depth, threshold, masks=masks)
        return s

    def collect(self) -> "ShardedMatcher":
        """Waits for the oldest frame in flight; returns its slot (``slot.fetch()`` = the merged match list)."""
        if self.in_flight() == 0:
            raise RuntimeError("ShardedPipe: no frame in flight")
        s = self.slots[self.collected % self.depth]
        self.collected += 1
        s.match_wait()
        return s

    def launch_count(self) -> int:
        return sum(s.h.launch_count() for s in self.slots)

    def close(self) -> None:
        for s in self.slots:
            s.close()


class NativeShardedPipe:
    """The same schedule as ``ShardedPipe`` with the per-frame host work inside the library: one ``fl_pipe`` per rank in template-sharded
    mode (``fl_pipe_set_exchange``).  torch only provides the symmetric-memory exchange buffers (one per slot, mapped into every process)
    and the rendezvous; ``match_batch`` is ONE C call for any number of frames.  Peer-memory exchange only.

    Recognition (``upload_model_depths``, ``set_recognition``, then ``submit_recognition`` / ``collect_recognition`` or ``recognize``, the
    arguments and return values of ``Pipe``'s methods): frame f is matched on every rank, refined and suppressed by rank f % world alone,
    and its results reach every rank through peer memory (fl_pipe_set_recognition_sharded); every rank collects the single detector's
    results for every frame."""

    def __init__(self, tset, rank: int, world: int, depth: int = 4, capacity: int = 2048, device=None, T=(5, 8), modality_kind=(0, 1),
                 max_width: int = 640, max_height: int = 480, max_candidates: int = 1 << 16):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        from . import Pipe, lib
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.rank, self.world, self.depth, self.cap = rank, world, int(depth), capacity
        self._tset, self._dev, self._reco_err = tset, dev, None        # the whole set: the recognition set-up selects from the merged list
        # Everything that can fail on ONE rank alone (device allocations, the template upload) happens before the first collective, and
        # the ranks agree on the outcome: a rank that failed must not leave its peers waiting inside the rendezvous that follows.
        self.pipe, self._xbufs, self._xhdls, self._blocks, err = None, [], [], [], None
        try:
            self.pipe = Pipe(self.depth, T, modality_kind, max_width, max_height, device=dev.index or 0,
                             max_candidates=max(max_candidates, world * (capacity + 1) + 16))
            shard, gids = shard_template_set(tset, rank, world)
            self.pipe.upload_templates(shard)
            if shard.n_templates:
                self.pipe.set_template_ids(gids)
            self.n_local = shard.n_templates
            nbytes = int(lib().fl_exchange_buffer_bytes(world, capacity))
            self._xbufs = [symm_mem.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(self.depth)]
            self._blocks = [torch.zeros(block_ints(capacity), dtype=torch.int32, device=dev) for _ in range(self.depth)]
        except Exception as e:  # noqa: BLE001
            err = e
        flag = torch.tensor([0 if err else 1], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if self.pipe is not None:
                self.pipe.close()
            raise RuntimeError("NativeShardedPipe: set-up failed on %s: %r" % ("this rank" if err else "another rank", err))
        peers = []
        for xb in self._xbufs:
            xh = symm_mem.rendezvous(xb, dist.group.WORLD)
            xb.zero_()
            self._xhdls.append(xh)
            peers.append([int(p) for p in xh.buffer_ptrs])
        torch.cuda.synchronize()
        dist.barrier()
        self.pipe.set_exchange(rank, world, capacity, peers, [b.data_ptr() for b in self._blocks])
        self.exchange = "p2p"

    def match_batch(self, frames, threshold: float, capacity_per_frame: int = 1 << 12, out=None, copy: bool = True):
        return self.pipe.match_batch(frames, threshold, capacity_per_frame=capacity_per_frame, out=out, copy=copy)

    def in_flight(self) -> int:
        return self.pipe.in_flight()

    def upload_model_depths(self, model_depths, rects_model) -> None:
        """``Pipe.upload_model_depths`` on this rank.  A failure here is raised by ``set_recognition`` on every rank, once the ranks
        have agreed on it: a rank that raised alone would leave its peers waiting."""
        self._reco_err = None
        try:
            self.pipe.upload_model_depths(model_depths, rects_model)
        except Exception as e:  # noqa: BLE001
            self._reco_err = e

    def set_recognition(self, crop_of_template, pose12=None, params=None) -> None:
        """``Pipe.set_recognition_sharded`` with the whole set this pipe was built from; crop index and pose of every template of that
        set.  Collective: the ranks agree on the outcome of the crop upload and of this set-up before any frame is submitted."""
        import torch
        import torch.distributed as dist
        err, self._reco_err = self._reco_err, None
        if err is None:
            try:
                self.pipe.set_recognition_sharded(self._tset, crop_of_template, pose12, params)
            except Exception as e:  # noqa: BLE001
                err = e
        flag = torch.tensor([0 if err else 1], device=self._dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            raise RuntimeError("NativeShardedPipe: recognition set-up failed on %s: %r" % ("this rank" if err else "another rank", err))

    def submit_recognition(self, bgr, depth, K, W=None, H=None) -> None:
        self.pipe.submit_recognition(bgr, depth, K, W, H)

    def collect_recognition(self, capacity: int = RECO_MAX_HYP):
        return self.pipe.collect_recognition(capacity)

    def recognize(self, bgr, depth, K, W=None, H=None, capacity: int = RECO_MAX_HYP):
        """One frame, submitted and collected (nothing else may be in flight)."""
        from . import FL_ERR_STATE, FealessError
        if self.in_flight():
            raise FealessError(FL_ERR_STATE, "NativeShardedPipe.recognize", "%d frame(s) in flight - collect them first" % self.in_flight())
        self.submit_recognition(bgr, depth, K, W, H)
        return self.collect_recognition(capacity)

    def close(self) -> None:
        import torch
        torch.cuda.synchronize()
        self.pipe.close()                                          # (the exchange buffers are only ever touched through raw pointers)
        self._blocks = self._xbufs = self._xhdls = None


# ---------------------------------------------------------------------------------------------------
# Hypothesis-sharded pose refinement (SURVEY.md 8e: "ICP hypotheses are dealt across GPUs; small all-gather of the refined
# poses before NMS").  After the candidate exchange every rank holds the SAME sorted match list, so hypothesis k of the top-K
# goes to rank k % world without any negotiation; each rank refines its share in one batched ICP launch
# (Handle.detection_batch_resident / detection_batch), one all-gather of fixed-size result blocks brings all poses to every
# rank, and every rank runs the reference's nonMaximumSuppression (ICP/NMS.cpp:6-39) redundantly on the complete list - in
# the ORIGINAL hypothesis order, which is what makes the greedy result independent of the number of GPUs.
# ---------------------------------------------------------------------------------------------------
def hypothesis_share(n_hyp: int, rank: int, world: int) -> np.ndarray:
    """Indices (into the sorted hypothesis list) refined by ``rank``: k with k % world == rank."""
    return np.arange(rank, n_hyp, world, dtype=np.int64)


def refine_sharded(n_hyp: int, refine_fn, rank: int, world: int, group=None, device=None) -> np.ndarray:
    """Refines ``n_hyp`` hypotheses across ``world`` ranks.  ``refine_fn(indices) -> ICP_RESULT_DTYPE[len(indices)]`` runs this rank's
    batched ICP for the given hypothesis indices (it is not called with an empty share).  Returns all ``n_hyp`` records in
    hypothesis order on every rank.  One collective (all-gather of ``ceil(n_hyp / world)`` records per rank)."""
    import torch
    import torch.distributed as dist
    from . import ICP_RESULT_DTYPE
    mine = hypothesis_share(n_hyp, rank, world)
    res = refine_fn(mine) if len(mine) else np.zeros(0, ICP_RESULT_DTYPE)
    res = np.ascontiguousarray(res, dtype=ICP_RESULT_DTYPE)
    if len(res) != len(mine):
        raise ValueError("refine_fn returned %d records for %d hypotheses" % (len(res), len(mine)))
    if world == 1 or not dist.is_initialized():
        return res
    per_rank = (n_hyp + world - 1) // world
    nbytes = per_rank * ICP_RESULT_DTYPE.itemsize
    if device is None:
        device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    block = torch.zeros(nbytes, dtype=torch.uint8)
    block[: res.nbytes] = torch.from_numpy(res.view(np.uint8).reshape(-1).copy())
    block = block.to(device)
    out = torch.empty(world * nbytes, dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(out, block, group=group)
    blocks = out.cpu().numpy().reshape(world, nbytes)
    merged = np.zeros(n_hyp, ICP_RESULT_DTYPE)
    for r in range(world):
        idx = hypothesis_share(n_hyp, r, world)
        merged[idx] = blocks[r, : len(idx) * ICP_RESULT_DTYPE.itemsize].copy().view(ICP_RESULT_DTYPE)
    return merged
