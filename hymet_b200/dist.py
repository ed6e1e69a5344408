"""Multi-GPU screen: one process per GPU, query sharded, sketch table replicated.

SURVEY.md 8e / BASELINE north_star: k-mers are independent, so each rank streams its
own shard of the contigs against a full copy of the table (sketch DBs fit 180 GB HBM
many times over).  The only cross-rank state is
  * counts[E]  -- per-hash multiplicities, summed with ONE NCCL all-reduce over NVLink
                  (uint32 sums are order independent => bit-exact), and
  * the mixture bottom-s set -- each rank's s smallest distinct hashes, all-gathered
                  (s*8 bytes per rank) and merged.
Everything after that (per-sketch reduction, -w, statistics) runs replicated.

torch.distributed is plumbing only (rendezvous + NCCL/gloo collectives).
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import screen as hs


class _DevMem:
    """Expose a raw device allocation of the library to torch (no copy)."""

    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def counts_tensor(scr: hs.Screen, device: int) -> torch.Tensor:
    """counts[E] of a flushed screen as an int32 CUDA tensor aliasing the library's buffer
    (two's-complement sums equal uint32 sums mod 2^32, which is S8's wrap rule)."""
    ptr, n = scr.counts_devptr()
    if n == 0:
        return torch.zeros(0, dtype=torch.int32, device=f"cuda:{device}")
    return torch.as_tensor(_DevMem(ptr, n, "<i4"), device=f"cuda:{device}")


def record_aligned_range(buf, rank: int, world: int) -> Tuple[int, int]:
    """Byte range of FASTA text `buf` owned by `rank`: cut at the first line starting
    with '>' at or after rank*n/world, so no record (hence no k-mer) spans two shards."""
    n = len(buf)
    if n and bytes(buf[:1]) == b"@":      # FASTQ ('@' also appears in quality lines): not splittable
        return (0, n) if rank == 0 else (n, n)

    def cut(i: int) -> int:
        if i <= 0:
            return 0
        if i >= n:
            return n
        j = buf.find(b"\n>", i - 1)
        return n if j < 0 else j + 1

    return cut(rank * n // world), cut((rank + 1) * n // world)


def merge_bottom_s(parts, s: int) -> np.ndarray:
    """Union of per-rank bottom-s sets -> the global s smallest distinct hashes (S9)."""
    allh = np.concatenate([np.asarray(p, np.uint64) for p in parts]) if len(parts) else np.zeros(0, np.uint64)
    return np.unique(allh)[:s]


def all_gather_mixture(local: np.ndarray, s: int, device: Optional[torch.device] = None, group=None):
    """Every rank's local mixture hashes (<= s each), as a list of uint64 arrays."""
    world = dist.get_world_size(group)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    buf = torch.zeros(s + 1, dtype=torch.int64, device=device)
    buf[0] = len(local)
    if len(local):
        buf[1:1 + len(local)] = torch.from_numpy(np.asarray(local, np.uint64).view(np.int64).copy()).to(device)
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf, group=group)
    parts = []
    for t in out:
        t = t.cpu().numpy()
        parts.append(t[1:1 + int(t[0])].view(np.uint64))
    return parts


def init_from_env(backend: Optional[str] = None) -> Tuple[int, int, int]:
    """(rank, world, local_rank) from torchrun's environment; initialises the process group."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local


# ---- the exchange records (layout shared with hs_screen_counts_absorb / hs_screen_mixture_merge_device) ----
#   pair record     [n_pairs | up to cap (entry id << 32 | count) pairs]         1 + cap int64 words
#   mixture record  [length  | s hashes, zero padded]                            1 + s int64 words
def mixture_record(mixture: np.ndarray, s: int) -> np.ndarray:
    """What hs_screen_mixture_record writes for a settled local mixture."""
    h = np.zeros(1 + s, np.int64)
    n = len(mixture)
    h[0] = n
    if n:
        h[1:1 + n] = np.asarray(mixture, np.uint64).view(np.int64)
    return h


def parse_mixture_rows(rows: np.ndarray):
    """rows[world, 1 + s] (int64) -> list of per-rank mixture arrays."""
    return [rows[r, 1:1 + int(rows[r, 0])].view(np.uint64) for r in range(rows.shape[0])]


def next_cap(most: int, cap: int, n_entries: int) -> int:
    """Capacity (pairs) of the next record given the largest pair count just seen: a quarter more than
    that, in steps of 65 536 pairs (the collective moves world x cap x 8 bytes whatever is in them: the
    round-1 rule, the next power of two above 1.5 x, sent 4 M-pair records for 1.5 M pairs at C3), never
    more than one pair per entry; unchanged unless this record overflowed or the next one could be a
    third smaller.  Every rank computes it from the same numbers."""
    step = 1 << 16
    want = max(4096, -(-(most + most // 4) // step) * step)
    want = min(want, max(4096, int(n_entries)))
    return want if (most > cap or want * 3 <= cap * 2) else cap


def pack_pairs(ids: np.ndarray, counts: np.ndarray) -> np.ndarray:
    """What the compaction kernel writes: (entry id << 32) | count, as int64 words."""
    return ((np.asarray(ids, np.uint64) << np.uint64(32)) | np.asarray(counts, np.uint64)).view(np.int64)


def unpack_pairs(pairs: np.ndarray):
    p = np.asarray(pairs).view(np.uint64)
    return (p >> np.uint64(32)).astype(np.int64), (p & np.uint64(0xFFFFFFFF)).astype(np.uint32)


class DistributedScreen:
    """hs.Screen whose finish() first exchanges counts and mixture with the other ranks.

    Default ("auto").  Once the last feed is enqueued counts[] is final in stream order, so each rank
    turns its record of touched entries into (entry id, count) pairs -- O(present hashes), no scan of
    the table-sized vector -- inside a fixed-size record [pair count | up to `cap` pairs] and starts an
    ASYNCHRONOUS all-gather of the records; the mixture finaliser (hs_screen_flush) runs underneath
    it.  Each rank then writes its <= s mixture hashes into a second, small record on the device,
    all-gathers those, and enqueues two library calls that consume the gathered buffers where they
    lie: hs_screen_mixture_merge_device (sort + unique + set size on the device) and
    hs_screen_counts_absorb (ONE launch over all ranks' pairs).  The host never looks at the gathered
    data, and since round 2 it does not wait for the mixture finaliser either (hs_screen_flush_async: the
    selection's verdict travels inside the mixture record): between the last feed and the results there
    is ONE synchronisation, the final one of hs_screen_finish, so the host enqueues all of this while the
    stream kernel is still running.

    `cap` follows the previous screen (next_cap).  If any rank's record is too small the absorb
    kernel adds nothing and says so in the stats that come back with the results; every rank sees the
    same records, takes the same decision, and redoes the count exchange as the north star's single
    dense NCCL all-reduce of counts[E] (`exchange="dense"` forces that path).  Both are exact
    integer sums.
    """

    def __init__(self, db: hs.Database, device: int, exchange: str = "auto", **kw):
        self.db, self.device = db, device
        # the library's kernels and torch's collectives must be ordered on ONE stream
        if kw.get("stream_ptr"):
            self._tstream = torch.cuda.ExternalStream(kw["stream_ptr"], device=torch.device("cuda", device))
        else:
            self._tstream = torch.cuda.Stream(device=torch.device("cuda", device))
            kw["stream_ptr"] = self._tstream.cuda_stream
        self.scr = hs.Screen(db, **kw)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.exchange_mode = os.environ.get("HYMET_SCREEN_EXCHANGE", exchange)
        self.last_exchange = None
        self.cap = int(min(1 << 20, max(4096, int(db.n_entries) // 8)))
        if self.exchange_mode == "sparse":      # forced: room for every entry, never falls back
            self.cap = int(max(4096, db.n_entries))
        self._rec = self._all = self._mix = self._mix_all = None
        self.n_unsettled = 0

    def __getattr__(self, name):      # feed_*, reset, stats, set_option ...
        return getattr(self.scr, name)

    def _dense(self):
        t = counts_tensor(self.scr, self.device)
        self._tstream.synchronize()
        if t.numel():
            dist.all_reduce(t, op=dist.ReduceOp.SUM)      # the one dense NCCL all-reduce of the path
        self._tstream.synchronize()
        self.last_exchange = "dense"

    def exchange(self):
        if self.world == 1:
            return          # nothing to exchange; finish() settles the mixture underneath the per-sketch reduction
        with torch.cuda.stream(self._tstream):
            self._exchange()

    def _exchange(self):
        dev = torch.device("cuda", self.device)
        s, cap = self.db.s, self.cap
        sparse = self.exchange_mode != "dense"
        if self._mix is None:
            self._mix = torch.zeros(1 + s, dtype=torch.int64, device=dev)
            self._mix_all = torch.empty(self.world * (1 + s), dtype=torch.int64, device=dev)
        work = None
        if sparse:
            n_rec = 1 + cap                               # [pair count | pairs]
            if self._rec is None or self._rec.numel() != n_rec:
                self._rec = torch.zeros(n_rec, dtype=torch.int64, device=dev)
                self._all = torch.empty(self.world * n_rec, dtype=torch.int64, device=dev)
            self.scr.counts_compact_async(self._rec[1:].data_ptr(), cap, self._rec.data_ptr())
            work = dist.all_gather_into_tensor(self._all, self._rec, async_op=True)
        if sparse:
            # one host synchronisation per screen: the host enqueues the whole exchange and the reduction while
            # the stream kernel still runs; the bottom-s selection's verdict travels inside the record
            self.scr.flush_async()
        else:
            self.scr.flush()                              # host round trips of the mixture finaliser: the collective runs underneath
        self.scr.mixture_record(self._mix.data_ptr())
        dist.all_gather_into_tensor(self._mix_all, self._mix)             # world x (1 + s) words
        self.scr.mixture_merge_device(self._mix_all.data_ptr(), self.world)
        if not sparse:
            return self._dense()
        work.wait()                                       # stream-level wait, the host does not block
        self.scr.counts_absorb(self._all.data_ptr(), self.world, cap, self.rank)
        self._cap_used = cap
        self.last_exchange = "sparse"

    def finish(self, wta: bool = False) -> hs.ScreenResult:
        return self._finish(wta, self.scr.finish)

    def finish_hits(self, wta: bool = False) -> hs.ScreenHits:
        """Same, returning only the references with hits (O(hits) on the way back to the host)."""
        return self._finish(wta, self.scr.finish_hits)

    def _finish(self, wta, fin):
        self.exchange()
        res = fin(wta)
        if self.world > 1 and res.stats.get("mix_unsettled"):
            # some rank's device-side selection did not hold (every rank read that from the same gathered
            # records): settle the mixtures the slow way and exchange them again; the counts are already merged
            self.n_unsettled += 1
            with torch.cuda.stream(self._tstream):
                self.scr.flush()
                self.scr.mixture_record(self._mix.data_ptr())
                dist.all_gather_into_tensor(self._mix_all, self._mix)
                self.scr.mixture_merge_device(self._mix_all.data_ptr(), self.world)
            res = fin(wta)
        if self.world > 1 and self.last_exchange == "sparse":
            most = int(res.stats["exchange_max_pairs"])
            if self.exchange_mode != "sparse":
                # size the next record from what this one carried: the collective moves world x cap x 8
                # bytes whatever is in them (every rank sees the same records, so takes the same decision)
                self.cap = next_cap(most, self._cap_used, self.db.n_entries)
            if res.stats["exchange_overflow"]:
                # some rank had more distinct hits than its record holds: nothing was added; redo the
                # count exchange densely and reduce again (the mixture is already merged)
                with torch.cuda.stream(self._tstream):
                    self._dense()
                res = fin(wta)
        return res
