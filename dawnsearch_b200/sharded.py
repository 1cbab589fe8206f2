"""Multi-GPU layer: the corpus is sharded by contiguous id range, one process per GPU.

The reference already answers a query this way across WAN peers: scatter the query, every
instance returns its local top-k, the caller merges by distance
(/root/reference/src/net/udp_service.rs:314-330, src/search/search_service.rs:201-277).  On
one NVSwitch box the same shape becomes: local exact top-k on every GPU (libdawn_b200) ->
ONE all-gather of a packed block of k (label, distance) pairs per query over NCCL/NVLink ->
device-side merge (dawn_merge_results_device).  Because every shard returns bit-exact
distances and the order is defined on (distance, label), the merged result is bit-identical
to a single index holding the whole corpus (with every label stored once: a label two shards
hold at the same distance comes back once, see dawn_merge_results_device).

torch is plumbing here (device buffers, streams, torch.distributed); all compute is in
libdawn_b200.so.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from .index import EM_LEN, Index, IndexOptions, merge_results_device, new_index


def shard_range(rank: int, world: int, rows: int):
    """Contiguous id-range shard of `rank`: (first_row, n_rows).  ceil(rows/world) per rank, the
    last ranks may hold fewer (or zero) rows."""
    per = (rows + world - 1) // world
    first = min(rank * per, rows)
    return first, max(0, min(per, rows - first))


class ResultBlock:
    """One shard's answer for a batch, packed so that it crosses NVLink as ONE message:
    [batch*k u64 labels][batch*k f32 distances][batch u32 counts][batch u32 flags], padded to 16 bytes.
    flags bit0 = this shard's exactness certificate held for the query; travelling with the block lets
    every rank see, without an extra exchange, whether any shard has to re-run a query exactly."""

    def __init__(self, batch: int, k: int):
        self.batch, self.k = batch, k
        self.off_dist = batch * k * 8
        self.off_counts = self.off_dist + batch * k * 4
        self.off_flags = self.off_counts + batch * 4
        self.nbytes = (self.off_flags + batch * 4 + 15) // 16 * 16

    def views(self, buf: torch.Tensor):
        """(labels int64 [B,k], distances f32 [B,k], counts int32 [B]) aliasing a uint8 buffer."""
        b, k = self.batch, self.k
        return (buf[: self.off_dist].view(torch.int64).view(b, k),
                buf[self.off_dist: self.off_counts].view(torch.float32).view(b, k),
                buf[self.off_counts: self.off_counts + b * 4].view(torch.int32))

    def flags(self, buf: torch.Tensor):
        """int32 [B] view of the certificate flags of one block, or [world, B] of a gathered buffer."""
        b = self.batch
        if buf.dim() == 2:
            return buf[:, self.off_flags: self.off_flags + b * 4].contiguous().view(torch.int32).view(buf.shape[0], b)
        return buf[self.off_flags: self.off_flags + b * 4].view(torch.int32)


def all_gather_blocks(local: torch.Tensor, gathered: torch.Tensor, group=None):
    """The one exchange step of a sharded search: [nbytes] uint8 per rank -> [world, nbytes] on
    every rank.  NCCL on the GPUs; gloo in the CPU tests, and -- staged through the host -- when several
    ranks share one GPU (NCCL refuses that; used to test the sharded logic on a one-GPU box)."""
    if local.is_cuda and dist.get_backend(group) == "gloo":
        g = torch.empty(gathered.shape, dtype=torch.uint8)
        dist.all_gather_into_tensor(g.view(-1), local.cpu(), group=group)
        gathered.copy_(g)
        return
    dist.all_gather_into_tensor(gathered.view(-1), local, group=group)


class ShardedIndex:
    """One rank's shard plus the collective search.  All ranks must call `search*` together."""

    def __init__(self, device: int, capacity: int, group=None, quantization: int = 0):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.device = device
        self.tdev = torch.device("cuda", device)
        self.index: Index = new_index(IndexOptions(device=device, capacity=capacity, quantization=quantization))
        self._ws = {}
        self._side = None
        self._last_merged = None
        self.last_search_escalated = 0  # queries this rank re-ran exactly in the last search() call

    def close(self):
        self.index.close()

    def _workspace(self, batch: int, k: int):
        key = (batch, k)
        ws = self._ws.get(key)
        if ws is None:
            d = self.tdev
            blk = ResultBlock(batch, k)
            ws = {
                "blk": blk,
                "q": torch.empty((batch, EM_LEN), dtype=torch.float32, device=d),
                "local": torch.zeros(blk.nbytes, dtype=torch.uint8, device=d),
                "gathered": torch.zeros((self.world, blk.nbytes), dtype=torch.uint8, device=d),
                "out": torch.zeros(blk.nbytes, dtype=torch.uint8, device=d),
                "h_q": torch.empty((batch, EM_LEN), dtype=torch.float32).pin_memory(),
                "h_out": torch.empty(blk.nbytes, dtype=torch.uint8).pin_memory(),
                "h_flags": torch.empty((self.world, batch), dtype=torch.int32).pin_memory(),
            }
            self._ws[key] = ws
        return ws

    def search_device(self, d_queries: torch.Tensor, k: int, pipelined: bool = False, distance_limit=None):
        """Queries already on this rank's GPU ([B,384] f32).  Enqueues local search, the all-gather
        and the merge; returns the packed result block (uint8, device) that `ResultBlock.views`
        decodes.

        pipelined=False: everything is enqueued on the current stream.
        pipelined=True (back-to-back batches): the exchange + merge of batch i run on a side stream
        while the current stream already searches batch i+1, so the NCCL latency and the wait for the
        slowest shard are hidden behind compute; call `wait_results()` before reading the block.

        distance_limit (UdpPacket::Search, udp_packets.rs:29-39): every shard pushes it into its kernels and cuts its
        counts on the device, so only hits with distance < limit are exchanged and merged."""
        batch = d_queries.shape[0]
        ws = self._workspace(batch, k)
        blk: ResultBlock = ws["blk"]
        # torch reports the legacy default stream as 0, which the C ABI reads as "the index's own
        # stream"; cudaStreamLegacy (0x1) names the default stream explicitly.
        main = torch.cuda.current_stream(self.tdev)
        stream = main.cuda_stream or 1
        if self.world == 1:
            base = ws["local"].data_ptr()
            self.index.search_device(d_queries.data_ptr(), batch, k, base, base + blk.off_dist, base + blk.off_counts,
                                     base + blk.off_flags, stream, distance_limit)
            return ws["local"]
        if not pipelined:
            base = ws["local"].data_ptr()
            self.index.search_device(d_queries.data_ptr(), batch, k, base, base + blk.off_dist, base + blk.off_counts,
                                     base + blk.off_flags, stream, distance_limit)
            all_gather_blocks(ws["local"], ws["gathered"], self.group)
            g, o = ws["gathered"].data_ptr(), ws["out"].data_ptr()
            merge_results_device(self.device, g, g + blk.off_dist, g + blk.off_counts, self.world, batch, k,
                                 o, o + blk.off_dist, o + blk.off_counts, stream, list_stride_bytes=blk.nbytes)
            return ws["out"]
        # ---- pipelined: double-buffered blocks, exchange + merge on a side stream
        if "pipe" not in ws:
            d = self.tdev
            ws["pipe"] = {
                "local": [torch.zeros(blk.nbytes, dtype=torch.uint8, device=d) for _ in range(2)],
                "gathered": [torch.zeros((self.world, blk.nbytes), dtype=torch.uint8, device=d) for _ in range(2)],
                "out": [torch.zeros(blk.nbytes, dtype=torch.uint8, device=d) for _ in range(2)],
                "searched": [torch.cuda.Event() for _ in range(2)],
                "merged": [None, None],
                "step": 0,
            }
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.tdev)
        pp = ws["pipe"]
        p = pp["step"] & 1
        pp["step"] += 1
        if pp["merged"][p] is not None:  # the side stream must be done with these buffers (two batches ago)
            main.wait_event(pp["merged"][p])
        base = pp["local"][p].data_ptr()
        self.index.search_device(d_queries.data_ptr(), batch, k, base, base + blk.off_dist, base + blk.off_counts,
                                 base + blk.off_flags, stream, distance_limit)
        pp["searched"][p].record(main)
        side = self._side
        side.wait_event(pp["searched"][p])
        with torch.cuda.stream(side):
            all_gather_blocks(pp["local"][p], pp["gathered"][p], self.group)
            g, o = pp["gathered"][p].data_ptr(), pp["out"][p].data_ptr()
            merge_results_device(self.device, g, g + blk.off_dist, g + blk.off_counts, self.world, batch, k,
                                 o, o + blk.off_dist, o + blk.off_counts, side.cuda_stream, list_stride_bytes=blk.nbytes)
            ev = torch.cuda.Event()
            ev.record(side)
        pp["merged"][p] = ev
        self._last_merged = ev
        return pp["out"][p]

    def wait_results(self):
        """Make the current stream wait for the last pipelined batch's exchange + merge."""
        if self._last_merged is not None:
            torch.cuda.current_stream(self.tdev).wait_event(self._last_merged)

    def _exchange(self, ws, k: int):
        """all-gather of ws["local"] + merge into ws["out"] on the current stream."""
        blk: ResultBlock = ws["blk"]
        main = torch.cuda.current_stream(self.tdev)
        stream = main.cuda_stream or 1
        all_gather_blocks(ws["local"], ws["gathered"], self.group)
        g, o = ws["gathered"].data_ptr(), ws["out"].data_ptr()
        merge_results_device(self.device, g, g + blk.off_dist, g + blk.off_counts, self.world, blk.batch, k,
                             o, o + blk.off_dist, o + blk.off_counts, stream, list_stride_bytes=blk.nbytes)

    def search(self, queries: np.ndarray, k: int, distance_limit=None):
        """Host queries in, host results out (every rank gets the full merged answer).

        Exactness across shards: a shard whose certificate failed for a query (near-ties deeper than the
        candidate slack, or a candidate-log overflow on the tensor-core path) re-runs that query through
        the host API -- which escalates to the exact scan -- patches its block, and the exchange + merge
        are repeated.  The flags ride in the gathered blocks, so all ranks take that decision together
        and the common case costs no extra synchronisation."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, EM_LEN)
        batch = q.shape[0]
        ws = self._workspace(batch, k)
        blk: ResultBlock = ws["blk"]
        self.last_search_escalated = 0
        with torch.cuda.device(self.tdev):
            main = torch.cuda.current_stream(self.tdev)
            ws["h_q"].copy_(torch.from_numpy(q))
            ws["q"].copy_(ws["h_q"], non_blocking=True)
            out = self.search_device(ws["q"], k, distance_limit=distance_limit)
            ws["h_out"].copy_(out, non_blocking=True)
            if self.world > 1:
                ws["h_flags"].copy_(blk.flags(ws["gathered"]), non_blocking=True)
            else:
                ws["h_flags"].copy_(blk.flags(ws["local"]).view(1, batch), non_blocking=True)
            main.synchronize()
            flags = ws["h_flags"].numpy()
            if (flags & 1).min() == 0:  # same data on every rank -> same decision on every rank
                mine = np.nonzero((flags[self.rank] & 1) == 0)[0]
                if len(mine):
                    # exact: escalates to the f32 scan
                    rl, rd, rc = (self.index.search_batch(q[mine], k) if distance_limit is None
                                  else self.index.search_batch_limit(q[mine], k, distance_limit))
                    lab, dist_, cnt = blk.views(ws["local"])
                    sel = torch.from_numpy(mine).to(self.tdev)
                    lab[sel] = torch.from_numpy(rl.view(np.int64)).to(self.tdev)
                    dist_[sel] = torch.from_numpy(rd).to(self.tdev)
                    cnt[sel] = torch.from_numpy(rc.astype(np.int32)).to(self.tdev)
                    blk.flags(ws["local"])[sel] = 1
                    self.last_search_escalated = int(len(mine))
                if self.world > 1:
                    self._exchange(ws, k)
                    out = ws["out"]
                else:
                    out = ws["local"]
                ws["h_out"].copy_(out, non_blocking=True)
                main.synchronize()
        labels, dists, counts = blk.views(ws["h_out"])
        return (labels.numpy().astype(np.uint64), dists.numpy().copy(), counts.numpy().astype(np.int64))
