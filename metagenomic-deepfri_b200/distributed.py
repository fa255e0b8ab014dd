"""One process per GPU: shard a protein set by length-balanced bins, stream each bin through the path in chunks, gather the
score matrix on rank 0.  `torch.distributed` is used for the rendezvous and the single final gather only - there is no
collective on the compute path (SURVEY.md §8e; the reference's loop over proteins is embarrassingly parallel,
`pipeline.py:301-319`)."""
from __future__ import annotations

from collections import deque
from typing import Callable, Iterable, List, Optional, Sequence, Tuple, Union

import numpy as np

from .sharding import ALPHA, BETA, chunks_by_residues, lpt_bins

#: one chunk = one launch of the whole path; bounded by proteins and residues (HBM workspace ~ 6 KB per residue)
CHUNK_PROTEINS, CHUNK_RESIDUES = 16384, 5_200_000


def shard_job(lengths: Sequence[int], world: int, max_proteins: int = CHUNK_PROTEINS,
              max_residues: int = CHUNK_RESIDUES, alpha: float = ALPHA, beta: float = BETA) -> List[List[np.ndarray]]:
    """LPT bins over `world` ranks, each cut into launch-sized chunks: `result[rank]` = list of protein-index arrays.  The bins
    balance the cost alpha L^2 + beta L (`sharding.cost`): the GCN path's fit by default; the sequence-only DeepCNN branch works
    per residue tile, with no L^2 term, so it shards with `alpha=0`."""
    return [chunks_by_residues(b, lengths, max_residues, max_proteins) for b in lpt_bins(lengths, world, alpha, beta)]


def stream_chunks(submit: Callable[[object, np.ndarray], object], chunks: Iterable[Tuple[object, int]],
                  out: Union[np.ndarray, Sequence[np.ndarray]], depth: int = 2,
                  on_done: Optional[Callable[[int, np.ndarray], None]] = None) -> None:
    """Software pipeline over chunks: `submit(chunk, out_rows)` returns a job with `.wait()`; at most `depth` jobs are in flight,
    so chunk k + 1 is packed and copied while chunk k computes (`Predictor.submit_structures`, `Predictor.submit_sequences`).
    `chunks` yields `(chunk, n_proteins)`.  With one array as `out`, the scores of the chunks land in consecutive rows of it; with a
    list of `depth` arrays (each with at least as many rows as the largest chunk), chunk k's scores land in the first n rows of
    `out[k % depth]`, so only the chunks in flight hold result memory.  `on_done(k, rows)` runs after chunk k's scores are on the
    host, while the following chunks compute (e.g. `ScoreBoard.put`), and before chunk k + depth is submitted - with a ring the
    rows are overwritten after that.  If a submit, wait or `on_done` raises, the jobs still in flight are waited for (their own
    errors dropped) before the exception propagates: a job that is never waited for would keep its context's slot busy."""
    ring = isinstance(out, (list, tuple))
    if ring and len(out) != depth:
        raise ValueError(f"stream_chunks: a ring of result buffers needs exactly depth = {depth} arrays, got {len(out)}")
    jobs = deque()
    row = 0
    try:
        for k, (chunk, n) in enumerate(chunks):
            if ring:
                if n > len(out[k % depth]):
                    raise ValueError(f"stream_chunks: chunk {k} has {n} rows, its ring buffer {len(out[k % depth])}")
                rows = out[k % depth][:n]
            else:
                rows = out[row:row + n]
            jobs.append((submit(chunk, rows), k, rows))
            row += n
            if len(jobs) >= depth:
                j, kk, rr = jobs.popleft()
                j.wait()
                if on_done is not None:
                    on_done(kk, rr)
        while jobs:
            j, kk, rr = jobs.popleft()
            j.wait()
            if on_done is not None:
                on_done(kk, rr)
    except BaseException:
        for j, _, _ in jobs:
            try:
                j.wait()
            except Exception:
                pass
        raise


class ScoreBoard:
    """The job's result matrix `[n_total, C]` float32 in node-local POSIX shared memory, mapped (and page-locked for the GPU) by
    every rank of the box: a rank's scores go where they belong as soon as they are on the host - `rows(lo, hi)` is a view the
    path can copy into directly (device -> shared pinned memory, no staging copy) when a rank owns a contiguous row range,
    `put(ids, scores)` scatters rows into protein order - and the "final gather" is a barrier: `finish()` returns the matrix on
    `dst`.  No collective moves data; on the 8-GPU box the NCCL gather + the single 2.5 GB device -> host copy on rank 0 that
    this replaces cost 11 % of the end-to-end time.  One node only (`torch.distributed` ranks on several hosts: use
    `ScoreGather`)."""

    def __init__(self, n_total: int, n_terms: int, dst: int = 0, pin: bool = True):
        from multiprocessing import shared_memory
        self.n_total, self.n_terms, self.dst = int(n_total), int(n_terms), dst
        self._shm = None
        self._registered = 0
        self.rank, self.world, self.dist_on = 0, 1, False
        try:
            import torch.distributed as dist
            self.dist_on = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
            if self.dist_on:
                self.rank, self.world = dist.get_rank(), dist.get_world_size()
        except ImportError:
            dist = None
        nbytes = max(1, self.n_total * self.n_terms * 4)
        if self.dist_on:
            import socket
            hosts = [None] * self.world
            dist.all_gather_object(hosts, socket.gethostname())
            if len(set(hosts)) != 1:
                raise RuntimeError("ScoreBoard: ranks on several hosts (%s); use ScoreGather" % sorted(set(hosts)))
            # every failure is agreed on by all ranks before anybody raises (a rank that raised alone would leave the others in
            # the next collective): the caller can then fall back to ScoreGather on all ranks
            name = [None]
            if self.rank == dst:
                try:
                    self._shm = shared_memory.SharedMemory(create=True, size=nbytes)
                    name[0] = self._shm.name
                except OSError:
                    name[0] = None
            dist.broadcast_object_list(name, src=dst)
            ok = name[0] is not None
            if ok and self.rank != dst:
                try:
                    self._shm = shared_memory.SharedMemory(name=name[0])
                    try:    # Python < 3.13 registers attached segments with this process's resource tracker, which would unlink
                        from multiprocessing import resource_tracker  # (and warn about) the creator's segment at exit
                        resource_tracker.unregister(self._shm._name, "shared_memory")
                    except Exception:
                        pass
                except OSError:
                    ok = False
            oks = [None] * self.world
            dist.all_gather_object(oks, bool(ok))
            if not all(oks):
                if self._shm is not None:
                    try:
                        if self.rank == dst:
                            self._shm.unlink()
                        self._shm.close()
                    except Exception:
                        pass
                    self._shm = None
                raise RuntimeError("ScoreBoard: node-local shared memory is unavailable (/dev/shm too small?); use ScoreGather")
        else:
            self._shm = shared_memory.SharedMemory(create=True, size=nbytes)
        self.array = np.ndarray((self.n_total, self.n_terms), np.float32, buffer=self._shm.buf)
        if self.rank == dst or not self.dist_on:
            self.array[...] = 0.0                       # first touch by the owner (and defined rows for ids nobody writes)
        if self.dist_on:
            dist.barrier()
        if pin:
            try:
                import torch
                if torch.cuda.is_available():
                    rc = torch.cuda.cudart().cudaHostRegister(self.array.ctypes.data, nbytes, 0)
                    if int(rc) == 0:
                        self._registered = nbytes
            except Exception:
                self._registered = 0                    # pageable shared memory still works, the copies are just staged

    def rows(self, lo: int, hi: int) -> np.ndarray:
        return self.array[lo:hi]

    def put(self, ids: np.ndarray, scores: np.ndarray) -> None:
        self.array[np.asarray(ids, np.int64)] = scores

    def finish(self) -> Optional[np.ndarray]:
        """Every rank calls it after its last `put` / direct write; returns the full matrix on `dst` (valid until `close`)."""
        if self.dist_on:
            import torch.distributed as dist
            dist.barrier()
        return self.array if (self.rank == self.dst or not self.dist_on) else None

    def close(self) -> None:
        if self._shm is None:
            return
        if self._registered:
            try:
                import torch
                torch.cuda.cudart().cudaHostUnregister(self.array.ctypes.data)
            except Exception:
                pass
            self._registered = 0
        if self.dist_on:
            import torch.distributed as dist
            dist.barrier()                               # nobody unlinks while another rank still reads or writes
        self.array = None
        owner = self.rank == self.dst or not self.dist_on
        if owner:
            try:
                self._shm.unlink()
            except FileNotFoundError:
                pass
        try:
            self._shm.close()
        except BufferError:                              # a caller still holds a view: the mapping goes away with the last view
            pass
        self._shm = None

    def __del__(self):
        try:
            if self._shm is not None and not self.dist_on:
                self.close()
        except Exception:
            pass


class ScoreGather:
    """The job's one collective, with every buffer allocated up front (page-locking 2 GB of host memory or growing the CUDA
    caching allocator inside the gather costs more than the gather itself).  Tensors, not pickles: one `gather` of the padded
    score blocks and one of the index vectors - NCCL: over NVLink, the scatter into protein order done on the GPU and ONE
    device->host copy into pinned memory; gloo: on the host."""

    def __init__(self, n_local: int, n_total: int, n_terms: int, dst: int = 0):
        import torch
        import torch.distributed as dist
        self.n_local, self.n_total, self.n_terms, self.dst = int(n_local), int(n_total), int(n_terms), dst
        self.dist_on = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if not self.dist_on:
            return
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.cuda = dist.get_backend() == "nccl"
        dev = torch.device("cuda", torch.cuda.current_device()) if self.cuda else torch.device("cpu")
        mine = torch.tensor([self.n_local], dtype=torch.int64, device=dev)
        counts = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(counts, mine)
        self.counts = [int(c.item()) for c in counts]
        self.nmax = max(max(self.counts), 1)
        self.sc = torch.zeros((self.nmax, n_terms), dtype=torch.float32, device=dev)
        self.ix = torch.zeros(self.nmax, dtype=torch.int64, device=dev)
        self.sc_all = self.ix_all = self.final = self.host = None
        if self.rank == dst:
            self.sc_all = [torch.empty_like(self.sc) for _ in range(self.world)]
            self.ix_all = [torch.empty_like(self.ix) for _ in range(self.world)]
            self.final = torch.zeros((n_total, n_terms), dtype=torch.float32, device=dev)
            self.host = torch.empty((n_total, n_terms), dtype=torch.float32, pin_memory=self.cuda)

    def gather(self, local_idx: np.ndarray, local_scores: np.ndarray) -> Optional[np.ndarray]:
        """-> [n_total, C] float32 in original protein order on `dst` (a view of this object's host buffer), None elsewhere."""
        import torch
        import torch.distributed as dist
        if len(local_idx) != self.n_local:
            raise ValueError("ScoreGather.gather: local size differs from the one announced at construction")
        if not self.dist_on:
            if len(local_idx) == self.n_total and (len(local_idx) == 0 or (local_idx[0] == 0 and local_idx[-1] == self.n_total - 1
                                                                          and np.all(np.diff(local_idx) == 1))):
                return local_scores
            out = np.zeros((self.n_total, self.n_terms), np.float32)
            out[local_idx] = local_scores
            return out
        n = self.n_local
        if n:
            self.sc[:n].copy_(torch.from_numpy(np.ascontiguousarray(local_scores, np.float32)), non_blocking=True)
            self.ix[:n].copy_(torch.from_numpy(np.ascontiguousarray(local_idx, np.int64)), non_blocking=True)
        dist.gather(self.sc, self.sc_all, dst=self.dst)
        dist.gather(self.ix, self.ix_all, dst=self.dst)
        if self.rank != self.dst:
            return None
        for r in range(self.world):
            if self.counts[r]:
                self.final.index_copy_(0, self.ix_all[r][:self.counts[r]], self.sc_all[r][:self.counts[r]])
        self.host.copy_(self.final, non_blocking=self.cuda)
        if self.cuda:
            torch.cuda.synchronize()
        return self.host.numpy()


def gather_scores(local_idx: np.ndarray, local_scores: np.ndarray, n_total: int, n_terms: int,
                  dst: int = 0) -> Optional[np.ndarray]:
    """One-shot form of `ScoreGather` (allocates its buffers on every call)."""
    return ScoreGather(len(local_idx), n_total, n_terms, dst).gather(np.asarray(local_idx, np.int64), local_scores)


def predict_sharded(forward: Callable[[np.ndarray], np.ndarray], lengths: Sequence[int], n_terms: int,
                    rank: int, world: int, max_residues: int = CHUNK_RESIDUES,
                    max_proteins: int = CHUNK_PROTEINS) -> Optional[np.ndarray]:
    """`forward(indices) -> scores[len(indices), C]` is run on this rank's LPT bin chunk by chunk; rank 0 returns the
    [len(lengths), C] matrix in input order, the other ranks None."""
    mine = shard_job(lengths, world, max_proteins, max_residues)[rank]
    try:
        board = ScoreBoard(len(lengths), n_terms, pin=False) if world > 1 else None
    except RuntimeError:            # ranks on several hosts: one collective at the end instead
        board = None
    if board is not None:
        for ch in mine:
            board.put(ch, forward(ch))
        final = board.finish()
        out = None if final is None else np.array(final)
        final = None
        board.close()
        return out
    parts = [forward(ch) for ch in mine]
    local_idx = np.concatenate(mine) if mine else np.zeros(0, np.int64)
    local_sc = np.concatenate(parts) if parts else np.zeros((0, n_terms), np.float32)
    return gather_scores(local_idx, local_sc, len(lengths), n_terms)
