"""Drop-in for the hot-path functions of `mDeepFRI.bio_utils` (`bio_utils.py:196-227`, `:348-385`).

`calculate_contact_map` and `build_align_contact_map` keep the reference signatures.  The batched
`build_align_contact_maps` is what `pipeline.py:476-481` should call instead of
`Pool.map(build_align_contact_map, ...)`: one launch for all alignments, no process pool.
"""
from __future__ import annotations

import ctypes as C
import logging
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .batching import pack_structures, with_float32_coords
from .contact_map_utils import pairwise_sqeuclidean

logger = logging.getLogger(__name__)


def threshold_sq(threshold) -> np.float32:
    """`threshold**2` is a Python scalar in the reference, so NumPy 2 compares the fp32 distance
    matrix against float32(threshold**2) (weak-scalar promotion), `bio_utils.py:214-220`."""
    with np.errstate(over="ignore"):
        return np.float32(threshold ** 2)


def calculate_contact_map(coordinates: np.ndarray, threshold=6.0, distance="sqeuclidean",
                          mode="matrix") -> np.ndarray:
    """`bio_utils.py:196-227`.  matrix -> int32 [n,n]; sparse -> int32 [nnz,2] in argwhere order."""
    distance_functions = {"sqeuclidean": pairwise_sqeuclidean}
    if distance == "sqeuclidean":
        thr = threshold_sq(threshold)
    else:
        thr = np.float32(threshold)
    distance_functions[distance]            # KeyError for unknown metrics, like the reference
    coords = coordinates
    if not isinstance(coords, np.ndarray) or coords.dtype != np.float32 or coords.ndim != 2 \
            or not coords.flags["C_CONTIGUOUS"]:
        # pairwise_sqeuclidean's typed memoryview would reject these
        from .contact_map_utils import _require_buffer
        _require_buffer(coords, np.float32, "coordinates")
    n, m = coords.shape
    ctx = _lib.default_context()
    L = _lib.lib()
    if m != 3:
        # generic column count: distance matrix on the GPU, threshold on the returned matrix
        cmap = (pairwise_sqeuclidean(coords) < thr).astype(np.int32)
        return np.argwhere(cmap == 1).astype(np.int32) if mode == "sparse" else cmap
    if mode == "sparse":
        nnz = C.c_int64(0)
        _lib.check(L.mdf_contact_map_sparse(ctx.handle, _lib.fp(coords), n, float(thr), None, 0, C.byref(nnz)))
        pairs = np.empty((nnz.value, 2), np.int32)
        if nnz.value:
            _lib.check(L.mdf_contact_map_sparse(ctx.handle, _lib.fp(coords), n, float(thr), _lib.ip(pairs),
                                                nnz.value, C.byref(nnz)))
        return pairs
    cmap = np.empty((n, n), np.int32)
    _lib.check(L.mdf_contact_map_dense(ctx.handle, _lib.fp(coords), n, float(thr), _lib.ip(cmap)))
    return cmap


def _packed_ragged(gq: Sequence[str], gt: Sequence[str], coords: Sequence[np.ndarray], thr: float, gen: int,
                   arena: Optional[np.ndarray]):
    """Bit-packed maps of n alignments held as Python lists, through `mdf_cmap_build_transfer_ragged`: the CPython glue collects
    the per-alignment pointers, the library counts the query lengths, packs into pinned staging on host threads and runs the
    fused kernels (the Python packer below costs more than the whole GPU stage).  -> (buffer, packed_off, seq_off) or None when
    the glue module is not built.  `arena`: caller-owned uint32 buffer (ideally page-locked) that receives the maps."""
    try:
        host = _lib.pyhost()
    except Exception:
        return None
    if not hasattr(host, "cmap_ragged"):
        return None
    ctx = _lib.default_context()
    fn = _lib.fn_addr("mdf_cmap_build_transfer_ragged")
    rc, poff, soff = host.cmap_ragged(fn, ctx.handle.value, gq, None, None, thr, gen, 0, 0)        # sizes only: no GPU work
    _lib.check(rc)
    packed_off = np.frombuffer(poff, np.int64)
    seq_off = np.frombuffer(soff, np.int64)
    total = int(packed_off[-1])
    if arena is not None:
        if arena.dtype != np.uint32 or arena.ndim != 1 or not arena.flags["C_CONTIGUOUS"] or arena.size < total:
            raise ValueError(f"out must be a C-contiguous 1-D uint32 buffer of at least {total} words")
        buf = arena
    else:
        buf = np.empty(total, np.uint32)
    rc, _, _ = with_float32_coords(lambda cs: host.cmap_ragged(fn, ctx.handle.value, gq, gt, cs, thr, gen, buf.ctypes.data, buf.size),
                                   coords)
    _lib.check(rc)
    return buf, packed_off, seq_off


def build_align_contact_maps(alignments: Sequence, threshold: float = 6, generated_contacts: int = 2,
                             packed: bool = False, out: Optional[np.ndarray] = None) -> List[Optional[np.ndarray]]:
    """Batched `build_align_contact_map`: every alignment with coordinates goes through one fused
    K1+K2 launch.  Returns, per alignment, int32 [Lq,Lq] (or bit-packed uint32 rows when
    `packed`) - `None` where `alignment.coords is None` (`bio_utils.py:381-383`).  `out` (packed only): a caller-owned 1-D
    uint32 buffer the maps are written into - the returned arrays are views of it; page-locked memory that is reused across
    calls turns the device -> host copy of the maps (48 KB for a 600-residue query) into one DMA instead of a staged copy into
    freshly faulted pages."""
    live = [i for i, a in enumerate(alignments) if a.coords is not None]
    out_list: List[Optional[np.ndarray]] = [None] * len(alignments)
    for i, a in enumerate(alignments):
        if a.coords is None:
            logger.warning(f"No coordinates found for {a.target_name}.")
    if not live:
        return out_list
    if packed:
        res = _packed_ragged([alignments[i].gapped_sequence for i in live], [alignments[i].gapped_target for i in live],
                             [alignments[i].coords for i in live], float(threshold_sq(threshold)), int(generated_contacts), out)
        if res is not None:
            buf, packed_off, seq_off = res
            lens = np.diff(seq_off)
            for k, i in enumerate(live):
                Lq = int(lens[k])
                out_list[i] = buf[packed_off[k]:packed_off[k + 1]].reshape(Lq, _lib.packed_row_words(Lq))
            return out_list
    out = out_list
    ps = pack_structures([alignments[i].gapped_sequence for i in live],
                         [alignments[i].gapped_target for i in live],
                         [alignments[i].coords for i in live])
    ctx = _lib.default_context()
    L = _lib.lib()
    n = len(live)
    thr = float(threshold_sq(threshold))
    if packed:
        buf = np.empty(int(ps.packed_off[-1]), np.uint32)
        _lib.check(L.mdf_cmap_build_transfer(ctx.handle, n, _lib.fp(ps.coords), _lib.lp(ps.coord_off), ps.q_aln,
                                             ps.t_aln, _lib.lp(ps.aln_off), _lib.lp(ps.seq_off), thr,
                                             int(generated_contacts), _lib.up(buf), _lib.lp(ps.packed_off), None, None))
        for k, i in enumerate(live):
            Lq = int(ps.seq_off[k + 1] - ps.seq_off[k])
            out[i] = buf[ps.packed_off[k]:ps.packed_off[k + 1]].reshape(Lq, _lib.packed_row_words(Lq))
        return out
    lens = np.diff(ps.seq_off)
    dense_off = np.zeros(n + 1, np.int64)
    np.cumsum(lens * lens, out=dense_off[1:])
    buf = np.empty(int(dense_off[-1]), np.int32)
    _lib.check(L.mdf_cmap_build_transfer(ctx.handle, n, _lib.fp(ps.coords), _lib.lp(ps.coord_off), ps.q_aln, ps.t_aln,
                                         _lib.lp(ps.aln_off), _lib.lp(ps.seq_off), thr, int(generated_contacts),
                                         None, None, _lib.ip(buf), _lib.lp(dense_off)))
    for k, i in enumerate(live):
        Lq = int(lens[k])
        out[i] = buf[dense_off[k]:dense_off[k + 1]].reshape(Lq, Lq)
    return out


def build_align_contact_map(alignment, threshold: float = 6,
                            generated_contacts: int = 2) -> Tuple[object, Optional[np.ndarray]]:
    """`bio_utils.py:348-385`: (alignment, int32[Lq,Lq]) or (alignment, None) without coordinates."""
    return (alignment, build_align_contact_maps([alignment], threshold, generated_contacts)[0])
