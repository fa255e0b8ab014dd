/*
 * _mdf_pyhost: CPython glue between Python lists and the ragged entry points of libmdf_b200.
 *
 * The reference's pipeline holds, per alignment, a few Python strings and one small NumPy array (pipeline.py:476-481,
 * alignment.py:65-150).  Joining / concatenating 16k of them in Python costs more than the GPU needs for the whole path
 * (measured: 115 ms of packing against a 68 ms step), so this module only collects the POINTERS - the UTF-8 buffer of each str,
 * the data pointer of each float32 [rows, 3] array - and hands them to mdf_path_submit_ragged, which packs them into pinned
 * memory on worker threads with the GIL released.  No arithmetic happens here.
 *
 *   submit_ragged(fn_addr, model_addr, seqs, gapped_query, gapped_target, coords, thr2, gen, scores_addr) -> (rc, job_addr)
 *   submit_pairs(fn_addr, model_addr, queries, targets, coords, matrix_addr, alphabet, ...) -> (rc, job_addr)
 *   submit_sequences(fn_addr, model_addr, seqs, scores_addr) -> (rc, job_addr)
 *   pointers(strings) -> (bytes ptr-array, bytes len-array)      [used for the alignment / ingest entry points]
 *   cmap_ragged(fn_addr, ctx_addr, gapped_query, gapped_target, coords, thr2, gen, out_addr, out_words) -> (rc, packed_off, seq_off)
 *
 * Errors: a str that is not ASCII raises UnicodeEncodeError like predict.pyx:19; a coordinate item that is not a C-contiguous
 * float32 [rows, 3] buffer raises TypeError naming the item (the Python wrapper converts and retries).
 */
#define PY_SSIZE_T_CLEAN
#include <Python.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct mdf_model mdf_model;
typedef struct mdf_job mdf_job;
typedef int (*submit_ragged_fn)(mdf_model *, int, const char *const *, const int *, const float *const *, const int *,
                                const char *const *, const char *const *, const int *, float, int, float *, mdf_job **);

/* borrowed pointer to the bytes of item `o` (str: ASCII only; bytes accepted) */
static int text_of(PyObject *o, const char **ptr, Py_ssize_t *len, const char *what, Py_ssize_t i)
{
    if (PyUnicode_Check(o)) {
        if (!PyUnicode_IS_ASCII(o)) {
            PyObject *b = PyUnicode_AsASCIIString(o);      /* raises UnicodeEncodeError with the offending position */
            Py_XDECREF(b);
            if (!PyErr_Occurred()) PyErr_Format(PyExc_ValueError, "%s[%zd] is not ASCII", what, i);
            return -1;
        }
        *ptr = PyUnicode_AsUTF8AndSize(o, len);            /* for ASCII strings: the string's own buffer, no copy */
        return *ptr ? 0 : -1;
    }
    if (PyBytes_Check(o)) {
        *ptr = PyBytes_AS_STRING(o);
        *len = PyBytes_GET_SIZE(o);
        return 0;
    }
    PyErr_Format(PyExc_TypeError, "%s[%zd] must be str or bytes", what, i);
    return -1;
}

/* data pointer and row count of coordinate item i (a C-contiguous float32 [rows, 3] buffer, kept in views[*nviews] until released) */
static int coords_of(PyObject *c, Py_buffer *views, Py_ssize_t *nviews, Py_ssize_t i, const float **ptr, int *rows)
{
    Py_buffer *v = &views[*nviews];
    if (PyObject_GetBuffer(c, v, PyBUF_C_CONTIGUOUS | PyBUF_FORMAT) < 0) {
        PyErr_Clear();
        PyErr_Format(PyExc_TypeError, "coords[%zd] is not a C-contiguous buffer", i);
        return -1;
    }
    ++*nviews;
    const char *f = v->format ? v->format : "";
    if (*f == '<' || *f == '=' || *f == '@') ++f;
    if (strcmp(f, "f") != 0 || v->itemsize != 4 || v->ndim != 2 || v->shape[1] != 3) {
        PyErr_Format(PyExc_TypeError, "coords[%zd] is not a float32 array of shape (Lt, 3)", i);
        return -1;
    }
    *ptr = (const float *)v->buf;
    *rows = (int)v->shape[0];
    return 0;
}

enum { TEXT, SAME_LEN, COORDS };      /* SAME_LEN: text items as long as those of the column before (paired alignment strings) */

/* One argument of n items, collected into pointer / length arrays: str or bytes items (their buffers and lengths), or coordinate
 * items (their float32 data and row counts, with the buffer views held until release) */
typedef struct {
    const char *name;
    int kind;
    PyObject *obj, *fast;
    const void **ptr;
    int *len;
    Py_buffer *views;
    Py_ssize_t nviews;
} Column;

/* Collects k columns that must hold the same number *n of items (else ValueError `mismatch`; OverflowError `too_long` for an item
 * of 2^31 characters or more).  Returns -1 with an exception set on failure; release() the columns in either case. */
static int collect(Column *c, int k, const char *mismatch, const char *too_long, Py_ssize_t *n)
{
    char msg[64];
    for (int j = 0; j < k; ++j) {
        snprintf(msg, sizeof msg, "%s must be a sequence", c[j].name);
        if (!(c[j].fast = PySequence_Fast(c[j].obj, msg))) return -1;
    }
    *n = PySequence_Fast_GET_SIZE(c[0].fast);
    for (int j = 1; j < k; ++j)
        if (PySequence_Fast_GET_SIZE(c[j].fast) != *n) {
            PyErr_SetString(PyExc_ValueError, mismatch);
            return -1;
        }
    for (int j = 0; j < k; ++j) {
        c[j].ptr = malloc(sizeof(void *) * (*n + 1));
        c[j].len = malloc(sizeof(int) * (*n + 1));
        if (c[j].kind == COORDS) c[j].views = calloc((size_t)*n + 1, sizeof(Py_buffer));
        if (!c[j].ptr || !c[j].len || (c[j].kind == COORDS && !c[j].views)) {
            PyErr_NoMemory();
            return -1;
        }
    }
    for (Py_ssize_t i = 0; i < *n; ++i)
        for (int j = 0; j < k; ++j) {
            Column *col = &c[j];
            PyObject *o = PySequence_Fast_GET_ITEM(col->fast, i);
            if (col->kind == COORDS) {
                const float *data;
                if (coords_of(o, col->views, &col->nviews, i, &data, &col->len[i]) < 0) return -1;
                col->ptr[i] = data;
                continue;
            }
            const char *text;
            Py_ssize_t len;
            if (text_of(o, &text, &len, col->name, i) < 0) return -1;
            if (col->kind == SAME_LEN && len != c[j - 1].len[i]) {
                PyErr_Format(PyExc_ValueError, "alignment %zd: query and target alignments differ in length", i);
                return -1;
            }
            if (len > INT32_MAX) {
                PyErr_SetString(PyExc_OverflowError, too_long);
                return -1;
            }
            col->ptr[i] = text;
            col->len[i] = (int)len;
        }
    return 0;
}

static void release(Column *c, int k)
{
    for (int j = 0; j < k; ++j) {
        for (Py_ssize_t i = 0; i < c[j].nviews; ++i) PyBuffer_Release(&c[j].views[i]);
        free(c[j].views);
        free(c[j].ptr);
        free(c[j].len);
        Py_XDECREF(c[j].fast);
    }
}

static PyObject *submit_ragged(PyObject *self, PyObject *args)
{
    unsigned long long fn_addr, model_addr, scores_addr;
    PyObject *seqs, *gq, *gt, *coords;
    double thr2;
    int gen;
    if (!PyArg_ParseTuple(args, "KKOOOOdiK", &fn_addr, &model_addr, &seqs, &gq, &gt, &coords, &thr2, &gen, &scores_addr)) return NULL;
    Column c[4] = {{"seqs", TEXT, seqs}, {"gapped_query", TEXT, gq}, {"gapped_target", SAME_LEN, gt}, {"coords", COORDS, coords}};
    Py_ssize_t n;
    PyObject *result = NULL;
    if (collect(c, 4, "seqs, gapped_query, gapped_target and coords must have the same length", "sequence too long", &n) == 0) {
        mdf_job *job = NULL;
        int rc;
        submit_ragged_fn fn = (submit_ragged_fn)(uintptr_t)fn_addr;
        Py_BEGIN_ALLOW_THREADS
        rc = fn((mdf_model *)(uintptr_t)model_addr, (int)n, (const char *const *)c[0].ptr, c[0].len, (const float *const *)c[3].ptr,
                c[3].len, (const char *const *)c[1].ptr, (const char *const *)c[2].ptr, c[1].len, (float)thr2, gen,
                (float *)(uintptr_t)scores_addr, &job);
        Py_END_ALLOW_THREADS
        result = Py_BuildValue("iK", rc, (unsigned long long)(uintptr_t)job);
    }
    release(c, 4);
    return result;
}

typedef int (*submit_pairs_fn)(mdf_model *, int, const char *const *, const int *, const char *const *, const int *, const float *const *,
                               const int *, const int8_t *, const char *, int, int, int, float, int, float *, int32_t *, int32_t *, int32_t *,
                               char *, const int64_t *, int *, mdf_job **);

/* submit_pairs(fn_addr, model_addr, queries, targets, coords, matrix_addr, alphabet, gap_open, gap_extend, thr2, gen, scores_addr,
 *              nw_score_addr, aln_len_addr, n_match_addr, ops_addr, ops_off_addr, ops_len_addr) -> (rc, job_addr)
 * the pairs twin of submit_ragged: calls mdf_path_submit_pairs with the GIL released (ops_addr == 0: no alignment strings) */
static PyObject *submit_pairs(PyObject *self, PyObject *args)
{
    unsigned long long fn_addr, model_addr, matrix_addr, scores_addr, nw_addr, len_addr, match_addr, ops_addr, ops_off_addr, ops_len_addr;
    PyObject *queries, *targets, *coords;
    const char *alphabet;
    Py_ssize_t A;
    int gap_open, gap_extend, gen;
    double thr2;
    if (!PyArg_ParseTuple(args, "KKOOOKy#iidiKKKKKKK", &fn_addr, &model_addr, &queries, &targets, &coords, &matrix_addr, &alphabet, &A,
                          &gap_open, &gap_extend, &thr2, &gen, &scores_addr, &nw_addr, &len_addr, &match_addr, &ops_addr, &ops_off_addr,
                          &ops_len_addr))
        return NULL;
    Column c[3] = {{"queries", TEXT, queries}, {"targets", TEXT, targets}, {"coords", COORDS, coords}};
    Py_ssize_t n;
    PyObject *result = NULL;
    if (collect(c, 3, "queries, targets and coords must have the same length", "sequence too long", &n) == 0) {
        mdf_job *job = NULL;
        int rc;
        submit_pairs_fn fn = (submit_pairs_fn)(uintptr_t)fn_addr;
        Py_BEGIN_ALLOW_THREADS
        rc = fn((mdf_model *)(uintptr_t)model_addr, (int)n, (const char *const *)c[0].ptr, c[0].len, (const char *const *)c[1].ptr,
                c[1].len, (const float *const *)c[2].ptr, c[2].len, (const int8_t *)(uintptr_t)matrix_addr, alphabet, (int)A, gap_open,
                gap_extend, (float)thr2, gen, (float *)(uintptr_t)scores_addr, (int32_t *)(uintptr_t)nw_addr,
                (int32_t *)(uintptr_t)len_addr, (int32_t *)(uintptr_t)match_addr, (char *)(uintptr_t)ops_addr,
                (const int64_t *)(uintptr_t)ops_off_addr, (int *)(uintptr_t)ops_len_addr, &job);
        Py_END_ALLOW_THREADS
        result = Py_BuildValue("iK", rc, (unsigned long long)(uintptr_t)job);
    }
    release(c, 3);
    return result;
}

typedef struct mdf_cnn_model mdf_cnn_model;
typedef int (*submit_sequences_fn)(mdf_cnn_model *, int, const char *const *, const int *, float *, mdf_job **);

/* submit_sequences(fn_addr, model_addr, seqs, scores_addr) -> (rc, job_addr)
 * the sequence-only DeepCNN branch: calls mdf_cnn_submit_ragged with the GIL released */
static PyObject *submit_sequences(PyObject *self, PyObject *args)
{
    unsigned long long fn_addr, model_addr, scores_addr;
    PyObject *seqs;
    if (!PyArg_ParseTuple(args, "KKOK", &fn_addr, &model_addr, &seqs, &scores_addr)) return NULL;
    Column c[1] = {{"seqs", TEXT, seqs}};
    Py_ssize_t n;
    PyObject *result = NULL;
    if (collect(c, 1, "", "sequence too long", &n) == 0) {
        mdf_job *job = NULL;
        int rc;
        submit_sequences_fn fn = (submit_sequences_fn)(uintptr_t)fn_addr;
        Py_BEGIN_ALLOW_THREADS
        rc = fn((mdf_cnn_model *)(uintptr_t)model_addr, (int)n, (const char *const *)c[0].ptr, c[0].len, (float *)(uintptr_t)scores_addr,
                &job);
        Py_END_ALLOW_THREADS
        result = Py_BuildValue("iK", rc, (unsigned long long)(uintptr_t)job);
    }
    release(c, 1);
    return result;
}

/* pointers(list of str / bytes) -> (ptr-array as bytes [n x 8], int32 length array as bytes [n x 4]); the pointers stay valid as
 * long as the list's items live */
static PyObject *pointers(PyObject *self, PyObject *arg)
{
    PyObject *f = PySequence_Fast(arg, "expected a sequence of str / bytes");
    if (!f) return NULL;
    const Py_ssize_t n = PySequence_Fast_GET_SIZE(f);
    PyObject *pb = PyBytes_FromStringAndSize(NULL, n * (Py_ssize_t)sizeof(char *)), *lb = PyBytes_FromStringAndSize(NULL, n * 4);
    if (!pb || !lb) { Py_XDECREF(pb); Py_XDECREF(lb); Py_DECREF(f); return NULL; }
    const char **pp = (const char **)PyBytes_AS_STRING(pb);
    int *ll = (int *)PyBytes_AS_STRING(lb);
    for (Py_ssize_t i = 0; i < n; ++i) {
        Py_ssize_t len;
        if (text_of(PySequence_Fast_GET_ITEM(f, i), &pp[i], &len, "item", i) < 0 || len > INT32_MAX) {
            if (!PyErr_Occurred()) PyErr_SetString(PyExc_OverflowError, "string too long");
            Py_DECREF(pb); Py_DECREF(lb); Py_DECREF(f);
            return NULL;
        }
        ll[i] = (int)len;
    }
    Py_DECREF(f);
    return Py_BuildValue("NN", pb, lb);
}

typedef struct mdf_ctx mdf_ctx;
typedef int (*cmap_ragged_fn)(mdf_ctx *, int, const float *const *, const int *, const char *const *, const char *const *, const int *,
                              float, int, uint32_t *, size_t, int64_t *, int64_t *);

/* cmap_ragged(fn_addr, ctx_addr, gapped_query, gapped_target, coords, thr2, gen, out_addr, out_capacity_words)
 *   -> (rc, packed_off bytes [n+1 x int64], seq_off bytes [n+1 x int64])
 * out_addr == 0: offsets only (coords / gapped_target may be None then).  Calls mdf_cmap_build_transfer_ragged with the GIL
 * released. */
static PyObject *cmap_ragged(PyObject *self, PyObject *args)
{
    unsigned long long fn_addr, ctx_addr, out_addr, out_cap;
    PyObject *gq, *gt, *coords;
    double thr2;
    int gen;
    if (!PyArg_ParseTuple(args, "KKOOOdiKK", &fn_addr, &ctx_addr, &gq, &gt, &coords, &thr2, &gen, &out_addr, &out_cap)) return NULL;
    /* out_addr == 0: sizes only, from the query alignments alone */
    const int k = out_addr == 0 ? 1 : 3;
    Column c[3] = {{"gapped_query", TEXT, gq}, {"gapped_target", SAME_LEN, gt}, {"coords", COORDS, coords}};
    Py_ssize_t n;
    PyObject *result = NULL, *poff = NULL, *soff = NULL;
    if (collect(c, k, "gapped_query, gapped_target and coords must have the same length", "alignment too long", &n) == 0) {
        poff = PyBytes_FromStringAndSize(NULL, (n + 1) * 8);
        soff = PyBytes_FromStringAndSize(NULL, (n + 1) * 8);
    }
    if (poff && soff) {
        int rc;
        cmap_ragged_fn fn = (cmap_ragged_fn)(uintptr_t)fn_addr;
        int64_t *po = (int64_t *)PyBytes_AS_STRING(poff), *so = (int64_t *)PyBytes_AS_STRING(soff);
        Py_BEGIN_ALLOW_THREADS
        rc = fn((mdf_ctx *)(uintptr_t)ctx_addr, (int)n, (const float *const *)c[2].ptr, c[2].len, (const char *const *)c[0].ptr,
                (const char *const *)c[1].ptr, c[0].len, (float)thr2, gen, (uint32_t *)(uintptr_t)out_addr, (size_t)out_cap, po, so);
        Py_END_ALLOW_THREADS
        result = Py_BuildValue("iOO", rc, poff, soff);
    }
    Py_XDECREF(poff);
    Py_XDECREF(soff);
    release(c, k);
    return result;
}

static PyMethodDef methods[] = {
    {"cmap_ragged", cmap_ragged, METH_VARARGS, "collect per-alignment pointers and call mdf_cmap_build_transfer_ragged (GIL released)"},
    {"submit_ragged", submit_ragged, METH_VARARGS, "collect per-protein pointers and call mdf_path_submit_ragged (GIL released)"},
    {"submit_pairs", submit_pairs, METH_VARARGS, "collect per-pair pointers and call mdf_path_submit_pairs (GIL released)"},
    {"submit_sequences", submit_sequences, METH_VARARGS, "collect per-sequence pointers and call mdf_cnn_submit_ragged (GIL released)"},
    {"pointers", pointers, METH_O, "pointer / length arrays of a list of str or bytes"},
    {NULL, NULL, 0, NULL}};

static struct PyModuleDef moddef = {PyModuleDef_HEAD_INIT, "_mdf_pyhost", "list -> pointer-array glue for libmdf_b200", -1, methods};

PyMODINIT_FUNC PyInit__mdf_pyhost(void) { return PyModule_Create(&moddef); }
