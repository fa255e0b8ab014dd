"""GPU tests of the threaded host packing behind the ragged entry points (`mdf_path_submit_ragged`, `mdf_path_submit_pairs`,
`mdf_cmap_build_transfer_ragged`).  With 2,048 items and MDF_HOST_THREADS = 1, 4 or 7 (7: ranges of uneven size) each packs on
that many threads, and every result equals a route that packs nothing on the host: the flat C ABI or a resident upload."""
import ctypes as C
import os

import numpy as np
import pytest

from metagenomic_deepfri_b200 import _lib, alignment, batching, bio_utils, predict, synth

pytestmark = pytest.mark.gpu
N = 2048
B62 = (alignment.BLOSUM62_ALPHABET, alignment.BLOSUM62)


@pytest.fixture(scope="module")
def wl():
    return synth.keyed_workload(np.arange(N), 17, lmax=400)


@pytest.fixture(scope="module", params=[1, 4, 7])
def mf(request, model_dir):
    """A predictor on a context of its own, created while MDF_HOST_THREADS is set (a context reads it at creation)."""
    old = os.environ.get("MDF_HOST_THREADS")
    os.environ["MDF_HOST_THREADS"] = str(request.param)
    try:
        ctx = _lib.Context()
    finally:
        if old is None:
            del os.environ["MDF_HOST_THREADS"]
        else:
            os.environ["MDF_HOST_THREADS"] = old
    p = predict.Predictor(model_dir["mf"], context=ctx)
    yield p
    p.close()
    ctx.close()


def pairs_of(wl):
    return list(wl.query_seqs), [g.replace("-", "") for g in wl.gapped_target], list(wl.coords)


def test_structures_equal_flat_submit_and_upload(mf, wl):
    got = mf.submit_structures(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords, 10.0, 2).wait()
    ps = batching.pack_structures(wl.gapped_query, wl.gapped_target, wl.coords)
    sb, so = predict._pack_checked(wl.query_seqs)
    flat = np.empty((N, mf.n_terms), np.float32)
    job = C.c_void_p()
    L = _lib.lib()
    _lib.check(L.mdf_path_submit(mf._handle, N, sb, _lib.lp(so), ps.coords.ctypes.data, _lib.lp(ps.coord_off), ps.q_aln, ps.t_aln,
                                 _lib.lp(ps.aln_off), float(bio_utils.threshold_sq(10.0)), 2, flat.ctypes.data, C.byref(job)))
    _lib.check(L.mdf_path_wait(job))
    b = mf.upload(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords)
    try:
        mf.run(b, 10.0, 2)
        resident = mf.fetch_scores(b)
    finally:
        b.close()
    assert np.abs(got - flat).max() < 1e-5
    assert np.abs(got - resident).max() < 1e-5


def test_contact_maps_equal_upload(mf, wl):
    """`_mdf_pyhost.cmap_ragged` on this context (as `bio_utils._packed_ragged` calls it on the default one)."""
    host = _lib.pyhost()
    fn = _lib.fn_addr("mdf_cmap_build_transfer_ragged")
    thr = float(bio_utils.threshold_sq(10.0))
    rc, poff, soff = host.cmap_ragged(fn, mf._ctx.handle.value, wl.gapped_query, None, None, thr, 2, 0, 0)
    _lib.check(rc)
    buf = np.empty(int(np.frombuffer(poff, np.int64)[-1]), np.uint32)
    rc, _, _ = host.cmap_ragged(fn, mf._ctx.handle.value, wl.gapped_query, wl.gapped_target, wl.coords, thr, 2, buf.ctypes.data,
                                buf.size)
    _lib.check(rc)
    b = mf.upload(wl.query_seqs, wl.gapped_query, wl.gapped_target, wl.coords)
    try:
        mf.run(b, 10.0, 2, upto=1)
        assert np.array_equal(np.frombuffer(poff, np.int64), b.packed_off)
        assert np.array_equal(np.frombuffer(soff, np.int64), b.seq_off)
        assert np.array_equal(buf, mf.fetch(b, "packed"))
    finally:
        b.close()


def test_pairs_equal_upload_pairs(mf, wl):
    qs, ts, cs = pairs_of(wl)
    s, nw, ln, nm = mf.forward_pairs(qs, ts, cs, B62, threshold=10.0, generated_contacts=2)
    b = mf.upload_pairs(qs, ts, cs, B62)
    try:
        nw2, ln2, nm2 = b.alignment()
        mf.run(b, 10.0, 2)
        resident = mf.fetch_scores(b)
    finally:
        b.close()
    assert np.array_equal(nw, nw2) and np.array_equal(ln, ln2) and np.array_equal(nm, nm2)
    assert np.abs(s - resident).max() < 1e-5


def test_first_bad_pair_across_threads(mf, wl):
    qs, ts, cs = pairs_of(wl)
    plant = lambda s: s[:2] + "J" + s[3:]              # 'J' is not in the BLOSUM62 alphabet
    bad_q, bad_t = list(qs), list(ts)
    bad_t[1500] = plant(bad_t[1500])
    bad_q[1900] = plant(bad_q[1900])
    with pytest.raises(ValueError, match="target 1500 holds 'J'"):
        mf.submit_pairs(bad_q, bad_t, cs, B62)
    with pytest.raises(ValueError, match="query 1900 holds 'J'"):
        mf.submit_pairs(bad_q, ts, cs, B62)
    # the context still works after the failed submits
    s = mf.forward_pairs(qs[:300], ts[:300], cs[:300], B62, threshold=10.0, generated_contacts=2)[0]
    assert s.shape == (300, mf.n_terms) and np.isfinite(s).all()
