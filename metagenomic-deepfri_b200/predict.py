"""Drop-in for `mDeepFRI.predict` (`predict.pyx`): `seq2onehot` and `Predictor`.

`Predictor(model_path, threads)` keeps the reference constructor and public attributes
(`model_path`, `threads`, `session`, `input_names`, `predict.pyx:50-60`) and
`forward_pass(seqres, cmap)` keeps its contract (`predict.pyx:75-102`): a float32 vector with
one score per GO term (channel 0 of the [1, C, 2] softmax output).  Instead of an onnxruntime
session, the `.onnx` file is decoded and recognised by the library itself (`mdf_model_load`, `csrc/onnx_load.cu`) and
executed by the fused CUDA pipeline behind the C ABI.  Batched entry points (`forward_batch`, `forward_structures`) run the same
kernels over many proteins per launch; `forward_pass` is a batch of one.

A single-input `.onnx` file (the `DeepCNN-MERGED_*` models) is the reference's sequence-only CNN
branch: `forward_pass(seqres)` with `cmap=None` (`predict.pyx:91-95`) and the batched
`forward_sequences` (or its asynchronous form `submit_sequences`) run it through the tcgen05 convolution kernel
(`csrc/cnn_tc.cu`).  There is no CPU or library fallback on either branch.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .batching import float32_coords, pack_structures, packed_offsets, with_float32_coords

_ALPHABET = b"-DGULNTKHYWCPVSOIEFXQABZRM"          # predict.pyx:26
_LUT = np.full(256, -1, np.int16)
_LUT[np.frombuffer(_ALPHABET, np.uint8)] = np.arange(26)


def _encode(seq: str) -> bytes:
    b = seq.encode("ascii")                         # UnicodeEncodeError like predict.pyx:19
    codes = _LUT[np.frombuffer(b, np.uint8)]
    bad = np.flatnonzero(codes < 0)
    if bad.size:
        raise ValueError(f"Invalid character in sequence: {seq[int(bad[0])]}")
    return b


def _pack_checked(seqs: Sequence[str]):
    """n sequences -> (ASCII bytes of all residues, int64 CSR offsets), validated in one vectorised pass with the error
    behaviour of `_encode` (per-sequence NumPy calls cost more than the GPU work for short proteins)."""
    n = len(seqs)
    joined = "".join(seqs)
    b = joined.encode("ascii")                      # UnicodeEncodeError like predict.pyx:19
    if b:
        bad = np.flatnonzero(_LUT[np.frombuffer(b, np.uint8)] < 0)
        if bad.size:
            raise ValueError(f"Invalid character in sequence: {joined[int(bad[0])]}")
    off = np.zeros(n + 1, np.int64)
    if n:
        np.cumsum(np.fromiter(map(len, seqs), np.int64, n), out=off[1:])
    return b, off


def seq2onehot(seq: str) -> np.ndarray:
    """`predict.pyx:17-48`: float32 [L, 26] one-hot over "-DGULNTKHYWCPVSOIEFXQABZRM"."""
    b = _encode(seq)
    out = np.zeros((len(b), 26), np.float32)
    if len(b):
        out[np.arange(len(b)), _LUT[np.frombuffer(b, np.uint8)]] = 1.0
    return out


class _Session:
    """Stands where the reference keeps its `onnxruntime.InferenceSession` (`predict.pyx:67-72`)."""

    class _Arg:
        def __init__(self, name):
            self.name = name

    def __init__(self, plan, handle, ctx: _lib.Context):
        self.plan = plan
        self.handle = handle
        self.ctx = ctx

    def get_inputs(self):
        return [self._Arg(n) for n in self.plan.input_names]

    def get_providers(self):
        return ["B200ExecutionProvider"]


class ModelInfo:
    """What `mdf_onnx_inspect` reports about the loaded file: head sizes, hyper-parameters, which initialiser plays which role."""

    def __init__(self, info: dict):
        self.info = info
        self.input_names = list(info["input_names"])
        self.n_terms = int(info["n_terms"])
        self.roles = dict(info.get("roles", {}))
        for k in ("lstm_hidden", "lm_dim", "fc_dim", "gc_dims", "gc_activation", "gc_alpha", "eps", "lm_fingerprint", "n_lstm",
                  "conv_filters", "conv_width", "conv_pad_left"):
            if k in info:
                setattr(self, k, info[k])


class PathInputs:
    """Path inputs of n proteins packed once into flat host arrays (optionally pinned through
    torch so that the per-call host->device copies are truly asynchronous)."""

    def __init__(self, seqs: Sequence[str], gapped_query: Sequence[str], gapped_target: Sequence[str],
                 coords: Sequence[np.ndarray], pin: bool = False):
        ps = pack_structures(gapped_query, gapped_target, coords)
        seq_bytes, seq_off = _pack_checked(seqs)
        if not np.array_equal(seq_off, ps.seq_off):
            raise ValueError("query sequences do not match the gap-stripped query alignments")
        self.n = len(seqs)
        self._pinned = []

        def host(a: np.ndarray) -> np.ndarray:
            if not pin or a.nbytes == 0:
                return np.ascontiguousarray(a)
            import torch
            t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
            self._pinned.append(t)
            v = t.numpy().view(a.dtype).reshape(a.shape)
            v[...] = a
            return v
        self.seq = host(np.frombuffer(seq_bytes, np.uint8))
        self.q_aln = host(np.frombuffer(ps.q_aln, np.uint8))
        self.t_aln = host(np.frombuffer(ps.t_aln, np.uint8))
        self.coords = host(ps.coords)
        self.seq_off, self.coord_off, self.aln_off = seq_off, ps.coord_off, ps.aln_off
        self.packed_off = ps.packed_off
        self.pin = pin
        self.h2d_bytes = int(self.seq.nbytes + self.q_aln.nbytes + self.t_aln.nbytes + self.coords.nbytes
                             + 8 * (seq_off.size + ps.coord_off.size + ps.aln_off.size))

    def output_buffer(self, n_terms: int) -> np.ndarray:
        if not self.pin:
            return np.empty((self.n, n_terms), np.float32)
        import torch
        t = torch.empty((self.n, n_terms), dtype=torch.float32, pin_memory=True)
        self._pinned.append(t)
        return t.numpy()


class PathBatch:
    """A batch of path inputs uploaded once and kept resident in HBM (`mdf_batch_upload`)."""

    def __init__(self, ctx: _lib.Context, seqs: Sequence[str], gapped_query: Sequence[str],
                 gapped_target: Sequence[str], coords: Sequence[np.ndarray]):
        ps = pack_structures(gapped_query, gapped_target, coords)
        seq_bytes, seq_off = _pack_checked(seqs)
        if not np.array_equal(seq_off, ps.seq_off):
            raise ValueError("query sequences do not match the gap-stripped query alignments")
        self.n = len(seqs)
        self.ctx = ctx
        self._keep = (ps, seq_bytes, seq_off)
        h = C.c_void_p()
        _lib.check(_lib.lib().mdf_batch_upload(
            ctx.handle, self.n, seq_bytes, _lib.lp(seq_off), ps.coords.ctypes.data, _lib.lp(ps.coord_off),
            ps.q_aln, ps.t_aln, _lib.lp(ps.aln_off), C.byref(h)))
        self.handle = h
        self.seq_off = seq_off
        self.packed_off = ps.packed_off
        self.h2d_bytes = (len(seq_bytes) + ps.coords.nbytes + 2 * len(ps.q_aln)
                          + 8 * (seq_off.size + ps.coord_off.size + ps.aln_off.size))

    def invalidate(self) -> None:
        """Drop what `run(share=True)` keeps between heads (contact maps, LSTM-LM output): the next run recomputes them."""
        _lib.check(_lib.lib().mdf_batch_invalidate(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            _lib.lib().mdf_batch_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PairBatch(PathBatch):
    """A `PathBatch` made from (query, target, coordinates) pairs (`mdf_batch_upload_pairs`): the pairs are aligned on the device
    once, at upload, and the alignment traceback writes the query frame of the contact-map stage; `Predictor.run` / `fetch` /
    `unpack_dense` work on it as on any uploaded batch."""

    def __init__(self, ctx: _lib.Context, queries: Sequence[str], targets: Sequence[str], coords: Sequence[np.ndarray],
                 scoring_matrix="VTML80", gap_open: int = 10, gap_extend: int = 1):
        from .alignment import resolve_matrix
        if not len(queries) == len(targets) == len(coords):
            raise ValueError("queries, targets and coords must have the same length")
        alphabet, m = resolve_matrix(scoring_matrix)
        qs, ts = [q.upper() for q in queries], [t.upper() for t in targets]
        seq_bytes, seq_off = _pack_checked(qs)
        t_bytes = "".join(ts).encode("ascii")
        t_off = np.zeros(len(ts) + 1, np.int64)
        np.cumsum(np.fromiter(map(len, ts), np.int64, len(ts)), out=t_off[1:])
        cs = float32_coords(coords)
        c_off = np.zeros(len(cs) + 1, np.int64)
        np.cumsum(np.fromiter((c.shape[0] for c in cs), np.int64, len(cs)), out=c_off[1:])
        flat = np.ascontiguousarray(np.concatenate(cs) if cs else np.zeros((0, 3), np.float32))
        self.n = len(qs)
        self.ctx = ctx
        self.handle = None
        h = C.c_void_p()
        _lib.check(_lib.lib().mdf_batch_upload_pairs(
            ctx.handle, self.n, seq_bytes, _lib.lp(seq_off), t_bytes, _lib.lp(t_off), flat.ctypes.data, _lib.lp(c_off),
            m.ctypes.data, alphabet.encode("ascii"), len(alphabet), int(gap_open), int(gap_extend), C.byref(h)))
        self.handle = h
        self.seq_off = seq_off
        self.packed_off = packed_offsets(np.diff(seq_off))
        self._ops_off = np.zeros(self.n + 1, np.int64)
        self._ops_off[1:] = seq_off[1:] + t_off[1:]
        self.h2d_bytes = 2 * len(seq_bytes) + len(t_bytes) + flat.nbytes + 8 * (seq_off.size + c_off.size)   # queries: ASCII + codes

    def alignment(self, ops: bool = False):
        """Per pair: (int32 NW score, alignment length, M columns[, alignment strings over M / X / I / D])."""
        stats = np.empty((3, self.n), np.int32)
        buf = np.empty(int(self._ops_off[-1]) + 1, np.uint8) if ops else None
        ops_len = np.empty(self.n, np.int32) if ops else None
        _lib.check(_lib.lib().mdf_batch_fetch_alignment(
            self.handle, stats[0].ctypes.data, stats[1].ctypes.data, stats[2].ctypes.data, buf.ctypes.data if ops else None,
            self._ops_off.ctypes.data if ops else None, ops_len.ctypes.data if ops else None))
        out = (stats[0], stats[1], stats[2])
        return out + (_decode_ops(buf, self._ops_off, ops_len),) if ops else out


def _decode_ops(buf: np.ndarray, off: np.ndarray, lens: np.ndarray) -> List[str]:
    b = buf.tobytes()
    return [b[off[p]:off[p] + lens[p]].decode("ascii") for p in range(len(lens))]


class PairJob:
    """An in-flight `Predictor.submit_pairs` call: `wait()` returns `(scores, nw_score, aln_len, n_match)`, plus the alignment
    strings when they were asked for."""

    def __init__(self, handle: Optional[int], out: np.ndarray, stats: np.ndarray, ops, queries):
        self._handle, self._out, self._stats, self._ops, self._queries = handle, out, stats, ops, queries
        self._result = None

    def wait(self):
        if self._handle is not None:
            h, self._handle = self._handle, None
            try:
                _lib.check(_lib.lib().mdf_path_wait(C.c_void_p(h)))
            except ValueError as e:
                if "Invalid character" in str(e):      # name the residue the way the reference does (predict.pyx:45-46)
                    for s in self._queries:
                        _encode(s)
                raise
            finally:
                self._queries = None
        if self._result is None:
            self._result = (self._out, self._stats[0], self._stats[1], self._stats[2])
            if self._ops is not None:
                buf, off, lens = self._ops
                self._result += (_decode_ops(buf, off, lens),)
        return self._result


class PathJob:
    """An in-flight `Predictor.submit_structures` or `Predictor.submit_sequences` call."""

    def __init__(self, pred: "Predictor", handle: int, out: np.ndarray, inputs):
        self._pred, self._handle, self._out, self._inputs = pred, handle, out, inputs

    def wait(self) -> np.ndarray:
        if self._handle is None:
            return self._out
        h, self._handle = self._handle, None
        try:
            _lib.check(_lib.lib().mdf_path_wait(C.c_void_p(h)))
        except ValueError as e:
            # the device only flags THAT an input was bad; name it the way the reference does (predict.pyx:45-46)
            seqs, gq, _ = self._inputs
            if "Invalid character" in str(e):
                for s in seqs:
                    _encode(s)
            if "does not match" in str(e):
                raise ValueError("query sequences do not match the gap-stripped query alignments") from None
            raise
        finally:
            self._inputs = None
        return self._out


class Predictor:
    def __init__(self, model_path: str, threads: int = 1, device: Optional[int] = None,
                 context: Optional[_lib.Context] = None):
        self.model_path = model_path
        self.threads = threads          # accepted for compatibility; the GPU path ignores it
        self._ctx = context if context is not None else _lib.default_context(device)
        self.session = None
        self.input_names: List[str] = []
        self._load_model()

    # -- predict.pyx:62-73
    def _load_model(self):
        L = _lib.lib()
        path = os.fsencode(self.model_path)
        info = _lib.inspect_onnx(self.model_path)     # FileNotFoundError / RuntimeError / UnsupportedModelError on bad files
        self.is_cnn = info["kind"] == "cnn"
        h = C.c_void_p()
        if self.is_cnn:
            _lib.check(L.mdf_cnn_model_load(self._ctx.handle, path, C.byref(h)))
            self.n_pooled = int(sum(info["conv_filters"]))
        else:
            _lib.check(L.mdf_model_load(self._ctx.handle, path, C.byref(h)))
        self._handle = h
        self.n_terms = int(info["n_terms"])
        self.plan = ModelInfo(info)
        self.session = _Session(self.plan, h, self._ctx)
        self.input_names = list(info["input_names"])

    # -- predict.pyx:91-95, batched: the sequence-only branch for n sequences
    def forward_sequences(self, seqs: Sequence[str], out: Optional[np.ndarray] = None) -> np.ndarray:
        if not self.is_cnn:
            raise ValueError("forward_sequences needs a sequence-only DeepCNN model; this Predictor holds a GCN head")
        n = len(seqs)
        seq_bytes, seq_off = _pack_checked(seqs)
        if out is None:
            out = np.empty((n, self.n_terms), np.float32)
        if n == 0:
            return out
        _lib.check(_lib.lib().mdf_cnn_forward(self._handle, n, seq_bytes, _lib.lp(seq_off), out.ctypes.data))
        return out

    def submit_sequences(self, seqs: Sequence[str], out: Optional[np.ndarray] = None) -> "PathJob":
        """Asynchronous `forward_sequences`: packs the n sequences into pinned staging memory (C, worker threads, GIL released),
        enqueues H2D + every kernel + the D2H of the scores and returns a `PathJob`; `job.wait()` returns the score matrix.
        The jobs share the context's two slots with `submit_structures`, so the next chunk's packing and copies overlap this
        chunk's kernels.  An empty sequence raises here; a residue outside the alphabet raises at `wait()`."""
        if not self.is_cnn:
            raise ValueError("submit_sequences needs a sequence-only DeepCNN model; this Predictor holds a GCN head")
        n = len(seqs)
        if out is None:
            out = np.empty((n, self.n_terms), np.float32)
        if out.shape != (n, self.n_terms) or out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("out must be a C-contiguous float32 array of shape (n, n_terms)")
        rc, job = _lib.pyhost().submit_sequences(_lib.fn_addr("mdf_cnn_submit_ragged"), self._handle.value, seqs, out.ctypes.data)
        _lib.check(rc)
        return PathJob(self, job, out, (seqs, None, None))

    def upload_sequences(self, seqs: Sequence[str]) -> int:
        """Keep n sequences resident in HBM for `run_sequences` / `fetch_sequences` (bench); returns the bytes copied."""
        if not self.is_cnn:
            raise ValueError("upload_sequences needs a sequence-only DeepCNN model")
        seq_bytes, seq_off = _pack_checked(seqs)
        _lib.check(_lib.lib().mdf_cnn_upload(self._handle, len(seqs), seq_bytes, _lib.lp(seq_off)))
        self._n_resident = len(seqs)
        return len(seq_bytes) + seq_off.nbytes

    def run_sequences(self) -> None:
        _lib.check(_lib.lib().mdf_cnn_run(self._handle))

    def fetch_sequences(self, pooled: bool = False):
        out = np.empty((self._n_resident, self.n_terms), np.float32)
        pl = np.empty((self._n_resident, self.n_pooled), np.float32) if pooled else None
        _lib.check(_lib.lib().mdf_cnn_fetch(self._handle, out.ctypes.data, pl.ctypes.data if pooled else None))
        return (out, pl) if pooled else out

    def _require_gcn(self, what: str) -> None:
        # the C handle of a DeepCNN Predictor is an mdf_cnn_model*: never hand it to an entry point that takes mdf_model*
        if self.is_cnn:
            raise ValueError(f"{what} needs a GCN head (cmap, seq); this Predictor holds a sequence-only DeepCNN model")

    def set_engine(self, engine: str) -> None:
        """'simt' = exact-fp32 CUDA-core engine, 'tc' = tcgen05 tensor-core engine."""
        self._require_gcn("set_engine")
        _lib.check(_lib.lib().mdf_model_set_engine(self._handle, {"simt": 0, "tc": 1}[engine]))

    @property
    def engine(self) -> str:
        self._require_gcn("engine")
        return {0: "simt", 1: "tc"}[_lib.lib().mdf_model_get_engine(self._handle)]

    # -- predict.pyx:75-102
    def forward_pass(self, seqres: str, cmap=None) -> np.ndarray:
        seq = _encode(seqres)
        if cmap is None:
            if not self.is_cnn:
                # the reference would feed one input to a two-input graph and onnxruntime would reject it
                raise ValueError("forward_pass(seqres) without a contact map needs a sequence-only DeepCNN model; "
                                 "this Predictor holds a GCN head (inputs: %s)" % ", ".join(self.input_names))
            if len(seq) == 0:
                raise ValueError("forward_pass: empty sequence (the max-pool over residues needs at least one)")
            return self.forward_sequences([seqres])[0]
        if self.is_cnn:
            # predict.pyx:87-90 would index input_names[1] of a single-input model
            raise ValueError("forward_pass(seqres, cmap): this Predictor holds a sequence-only DeepCNN model (one input)")
        A = cmap.reshape(cmap.shape[0], cmap.shape[1])
        L = len(seq)
        if A.shape != (L, L):
            raise ValueError(f"cmap shape {A.shape} does not match sequence length {L}")
        if A.dtype != np.int32:
            Ai = A.astype(np.int32)
            if not np.array_equal(Ai, A):
                raise ValueError("forward_pass: contact map holds values other than 0/1")
            A = Ai
        A = np.ascontiguousarray(A)
        y = np.empty(self.n_terms, np.float32)
        _lib.check(_lib.lib().mdf_gcn_forward_dense(self._handle, seq, L, _lib.ip(A), _lib.fp(y)))
        return y

    def forward_batch(self, seqs: Sequence[str], packed_cmaps: Sequence[np.ndarray]) -> np.ndarray:
        """GCN forward for n proteins with bit-packed maps (uint32 [L, row_words] each)."""
        self._require_gcn("forward_batch")
        n = len(seqs)
        seq_bytes, seq_off = _pack_checked(seqs)
        poff = packed_offsets(np.diff(seq_off))
        flat = np.concatenate([np.ascontiguousarray(c, np.uint32).reshape(-1) for c in packed_cmaps]) \
            if n else np.zeros(0, np.uint32)
        if flat.size != poff[-1]:
            raise ValueError("packed contact maps do not match the sequence lengths")
        out = np.empty((n, self.n_terms), np.float32)
        _lib.check(_lib.lib().mdf_gcn_forward_packed(self._handle, n, seq_bytes, _lib.lp(seq_off), _lib.up(flat),
                                                     _lib.lp(poff), _lib.fp(out)))
        return out

    def submit_structures(self, seqs: Sequence[str], gapped_query: Sequence[str], gapped_target: Sequence[str],
                          coords: Sequence[np.ndarray], threshold: float = 6, generated_contacts: int = 2,
                          out: Optional[np.ndarray] = None) -> "PathJob":
        """Asynchronous `forward_structures`: packs the n proteins into pinned staging memory (C, worker threads, GIL released),
        enqueues H2D + every kernel + the D2H of the scores and returns a `PathJob`; `job.wait()` returns the score matrix.
        Two jobs may be in flight per context, so the next batch's packing and copies overlap this batch's kernels."""
        from .bio_utils import threshold_sq
        self._require_gcn("submit_structures")
        n = len(seqs)
        if out is None:
            out = np.empty((n, self.n_terms), np.float32)
        if out.shape != (n, self.n_terms) or out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("out must be a C-contiguous float32 array of shape (n, n_terms)")
        host = _lib.pyhost()
        args = (_lib.fn_addr("mdf_path_submit_ragged"), self._handle.value, seqs, gapped_query, gapped_target)
        tail = (float(threshold_sq(threshold)), int(generated_contacts), out.ctypes.data)
        rc, job = with_float32_coords(lambda cs: host.submit_ragged(*args, cs, *tail), coords)
        _lib.check(rc)
        return PathJob(self, job, out, (seqs, gapped_query, gapped_target))

    def forward_structures(self, seqs: Sequence[str], gapped_query: Sequence[str], gapped_target: Sequence[str],
                           coords: Sequence[np.ndarray], threshold: float = 6, generated_contacts: int = 2,
                           out: Optional[np.ndarray] = None) -> np.ndarray:
        """The whole path for n proteins (contact map build + alignment transfer + GCN), host
        buffers in, host scores out: what `pipeline.py:476-481` + `:301-319` compute together."""
        return self.submit_structures(seqs, gapped_query, gapped_target, coords, threshold, generated_contacts, out).wait()

    def submit_pairs(self, queries: Sequence[str], targets: Sequence[str], coords: Sequence[np.ndarray], scoring_matrix="VTML80",
                     gap_open: int = 10, gap_extend: int = 1, threshold: float = 6, generated_contacts: int = 2,
                     out: Optional[np.ndarray] = None, alignments: bool = False) -> PairJob:
        """Align and predict in one asynchronous job: pair p is (query, best-hit target sequence, target C-alpha coordinates).
        The pairs are aligned on the device (global alignment as `alignment.nw_align`: same matrices, gap penalties, scores
        and alignment strings; sequences upper-cased) and the traceback builds the contact-map input directly, so the result
        equals `submit_structures(queries, *insert_gaps(query, target, ops), coords)` with no alignment string passing through
        the host.  `job.wait()` returns `(scores, nw_score, aln_len, n_match)` - identity = n_match / aln_len - and the
        alignment strings as a fifth item with `alignments=True`.  Jobs share the two slots of `submit_structures`."""
        from .alignment import resolve_matrix
        from .bio_utils import threshold_sq
        self._require_gcn("submit_pairs")
        n = len(queries)
        if len(targets) != n or len(coords) != n:
            raise ValueError("queries, targets and coords must have the same length")
        if out is None:
            out = np.empty((n, self.n_terms), np.float32)
        if out.shape != (n, self.n_terms) or out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("out must be a C-contiguous float32 array of shape (n, n_terms)")
        alphabet, m = resolve_matrix(scoring_matrix)
        qs, ts = [q.upper() for q in queries], [t.upper() for t in targets]
        stats = np.empty((3, n), np.int32)
        ops = None
        if alignments:
            off = np.zeros(n + 1, np.int64)
            if n:
                np.cumsum(np.fromiter((len(q) + len(t) for q, t in zip(qs, ts)), np.int64, n), out=off[1:])
            ops = (np.empty(int(off[-1]) + 1, np.uint8), off, np.empty(n, np.int32))
        if n == 0:
            return PairJob(None, out, stats, ops, None)
        host = _lib.pyhost()
        head = (_lib.fn_addr("mdf_path_submit_pairs"), self._handle.value, qs, ts)
        tail = (m.ctypes.data, alphabet.encode("ascii"), int(gap_open), int(gap_extend), float(threshold_sq(threshold)),
                int(generated_contacts), out.ctypes.data, stats[0].ctypes.data, stats[1].ctypes.data, stats[2].ctypes.data,
                *((ops[0].ctypes.data, ops[1].ctypes.data, ops[2].ctypes.data) if alignments else (0, 0, 0)))
        rc, job = with_float32_coords(lambda cs: host.submit_pairs(*head, cs, *tail), coords)
        _lib.check(rc)
        return PairJob(job, out, stats, ops, qs)

    def forward_pairs(self, queries: Sequence[str], targets: Sequence[str], coords: Sequence[np.ndarray], scoring_matrix="VTML80",
                      gap_open: int = 10, gap_extend: int = 1, threshold: float = 6, generated_contacts: int = 2,
                      out: Optional[np.ndarray] = None, alignments: bool = False):
        """`submit_pairs(...).wait()`."""
        return self.submit_pairs(queries, targets, coords, scoring_matrix, gap_open, gap_extend, threshold, generated_contacts, out,
                                 alignments).wait()

    def forward_inputs(self, inputs: PathInputs, threshold: float = 6, generated_contacts: int = 2,
                       out: Optional[np.ndarray] = None) -> np.ndarray:
        """`forward_structures` on pre-packed (optionally pinned) host buffers: per call this does
        the host->device copies, every kernel of the path and the device->host copy of the scores."""
        from .bio_utils import threshold_sq
        self._require_gcn("forward_inputs")
        if out is None:
            out = inputs.output_buffer(self.n_terms)
        _lib.check(_lib.lib().mdf_path_forward(
            self._handle, inputs.n, inputs.seq.ctypes.data, _lib.lp(inputs.seq_off), inputs.coords.ctypes.data,
            _lib.lp(inputs.coord_off), inputs.q_aln.ctypes.data, inputs.t_aln.ctypes.data, _lib.lp(inputs.aln_off),
            float(threshold_sq(threshold)), int(generated_contacts), out.ctypes.data))
        return out

    # -- resident-batch interface (bench / multi-head reuse)
    def upload(self, seqs, gapped_query, gapped_target, coords) -> PathBatch:
        self._require_gcn("upload")
        return PathBatch(self._ctx, seqs, gapped_query, gapped_target, coords)

    def upload_pairs(self, queries, targets, coords, scoring_matrix="VTML80", gap_open: int = 10, gap_extend: int = 1) -> PairBatch:
        """Resident form of `submit_pairs`: aligns once at upload; `run(batch, ..., share=True)` then serves every head."""
        self._require_gcn("upload_pairs")
        return PairBatch(self._ctx, queries, targets, coords, scoring_matrix, gap_open, gap_extend)

    def run(self, batch: PathBatch, threshold: float = 6, generated_contacts: int = 2, upto: int = 4,
            share: bool = False) -> None:
        """Run the path on an uploaded batch.  `share=True` keeps what an earlier run of ANOTHER head on this batch
        already computed and this head shares (contact maps, LSTM-LM output); the default recomputes everything."""
        from .bio_utils import threshold_sq
        self._require_gcn("run")
        if share:
            if upto != 4:
                raise ValueError("run(share=True) runs the whole path")
            _lib.check(_lib.lib().mdf_path_run_shared(self._handle, batch.handle, float(threshold_sq(threshold)),
                                                      int(generated_contacts)))
            return
        _lib.check(_lib.lib().mdf_path_run_stages(self._handle, batch.handle, float(threshold_sq(threshold)),
                                                  int(generated_contacts), upto))

    def fetch_scores(self, batch: PathBatch, out: Optional[np.ndarray] = None) -> np.ndarray:
        self._require_gcn("fetch_scores")
        if out is None:
            out = np.empty((batch.n, self.n_terms), np.float32)
        _lib.check(_lib.lib().mdf_batch_fetch_scores(self._handle, batch.handle, out.ctypes.data))
        return out

    def unpack_dense(self, batch: PathBatch) -> int:
        """Writes the contact maps of the last run in the reference's dense int32 [Lq, Lq] layout to workspace scratch
        (the HBM-bound variant of the contact-map stage, timed by bench.py / tools/cmap_bench.py); returns the cell count."""
        cells = C.c_int64(0)
        _lib.check(_lib.lib().mdf_batch_unpack_dense(batch.handle, None, C.byref(cells)))
        return int(cells.value)

    _TAPS = {"packed": 0, "deg": 1, "lstm1": 2, "lstm2": 3, "x0": 4, "pooled": 5, "gc_last": 6}

    def fetch(self, batch: PathBatch, what: str) -> np.ndarray:
        self._require_gcn("fetch")
        T = int(batch.seq_off[-1])
        p = self.plan
        shape, dt = {
            "packed": ((int(batch.packed_off[-1]),), np.uint32), "deg": ((T,), np.float32),
            "lstm1": ((T, p.lstm_hidden), np.float32), "lstm2": ((T, p.lstm_hidden), np.float32),
            "x0": ((T, p.lm_dim), np.float32), "pooled": ((batch.n, sum(p.gc_dims)), np.float32),
            "gc_last": ((T, p.gc_dims[-1]), np.float32)}[what]
        out = np.empty(shape, dt)
        _lib.check(_lib.lib().mdf_batch_fetch(self._handle, batch.handle, self._TAPS[what], out.ctypes.data, out.nbytes))
        return out

    def close(self):
        if getattr(self, "_handle", None):
            if getattr(self, "is_cnn", False):
                _lib.lib().mdf_cnn_model_destroy(self._handle)
            else:
                _lib.lib().mdf_model_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
