"""Ragged-batch packing for the C ABI: lists of proteins -> flat arrays + CSR offsets."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from ._lib import packed_row_words


@dataclass
class PackedStructures:
    n: int
    q_aln: bytes
    t_aln: bytes
    aln_off: np.ndarray     # int64 [n+1]
    coords: np.ndarray      # float32 [sum Lt, 3]
    coord_off: np.ndarray   # int64 [n+1] (rows)
    seq_off: np.ndarray     # int64 [n+1] query residues (non-gap query columns)
    packed_off: np.ndarray  # int64 [n+1] uint32 words of the bit-packed maps


def query_lengths(gapped_queries: Sequence[bytes]) -> np.ndarray:
    return np.array([len(q) - q.count(b"-") for q in gapped_queries], dtype=np.int64)


def packed_offsets(lengths: np.ndarray) -> np.ndarray:
    off = np.zeros(len(lengths) + 1, np.int64)
    words = np.array([int(L) * packed_row_words(int(L)) for L in lengths], dtype=np.int64)
    np.cumsum(words, out=off[1:])
    return off


def pack_structures(gapped_query: Sequence[str], gapped_target: Sequence[str],
                    coords: Sequence[np.ndarray]) -> PackedStructures:
    n = len(gapped_query)
    qb = [s.encode("ascii") for s in gapped_query]
    tb = [s.encode("ascii") for s in gapped_target]
    for i in range(n):
        if len(qb[i]) != len(tb[i]):
            raise ValueError(f"alignment {i}: query and target alignments differ in length")
    aln_off = np.zeros(n + 1, np.int64)
    np.cumsum([len(q) for q in qb], out=aln_off[1:])
    cs = []
    for i, c in enumerate(coords):
        c = np.asarray(c)
        if c.ndim != 2 or c.shape[1] != 3:
            raise ValueError(f"structure {i}: coordinates must have shape (Lt, 3)")
        cs.append(np.ascontiguousarray(c, dtype=np.float32))
    coord_off = np.zeros(n + 1, np.int64)
    np.cumsum([c.shape[0] for c in cs], out=coord_off[1:])
    allc = np.concatenate(cs, axis=0) if cs else np.zeros((0, 3), np.float32)
    lens = query_lengths(qb)
    seq_off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=seq_off[1:])
    return PackedStructures(n, b"".join(qb), b"".join(tb), aln_off, np.ascontiguousarray(allc), coord_off,
                            seq_off, packed_offsets(lens))


def float32_coords(coords) -> list:
    """Structures as C-contiguous float32 [Lt, 3] arrays, converted like the reference's astype(np.float32) (contact_map.py:25)."""
    conv = []
    for i, c in enumerate(coords):
        c = np.ascontiguousarray(c, dtype=np.float32)
        if c.ndim != 2 or c.shape[1] != 3:
            raise ValueError(f"structure {i}: coordinates must have shape (Lt, 3)")
        conv.append(c)
    return conv


def with_float32_coords(call, coords):
    """`call(coords)` into the CPython glue, which takes structures only as C-contiguous float32 [Lt, 3] arrays and raises
    TypeError for any other (lists, float64 ...): then once more with every structure converted by `float32_coords`."""
    try:
        return call(coords)
    except TypeError:
        return call(float32_coords(coords))


def pack_sequences(seqs: Sequence[str]):
    sb = [s.encode("ascii") for s in seqs]
    off = np.zeros(len(sb) + 1, np.int64)
    np.cumsum([len(s) for s in sb], out=off[1:])
    return b"".join(sb), off


def unpack_bits(packed_rows: np.ndarray, L: int) -> np.ndarray:
    """uint32 [L, row_words] -> int32 [L, L] (host helper for tests / debugging)."""
    if L == 0:
        return np.zeros((0, 0), np.int32)
    bits = np.unpackbits(packed_rows.view(np.uint8).reshape(L, -1), axis=1, bitorder="little")
    return bits[:, :L].astype(np.int32)


def pack_bits(dense: np.ndarray) -> np.ndarray:
    """int [L, L] 0/1 -> uint32 [L, row_words] (host helper for tests)."""
    L = dense.shape[0]
    rw = packed_row_words(L)
    padded = np.zeros((L, rw * 32), np.uint8)
    padded[:, :L] = dense != 0
    return np.packbits(padded, axis=1, bitorder="little").view(np.uint32).reshape(L, rw)
