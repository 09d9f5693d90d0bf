/* mctq_pyext.c -- CPython front door to the hottest C-ABI entry points (module `_mctq_fast`).
 *
 * ctypes spends ~4 us per call converting 11-14 arguments; for the 0.6 MB activation of BASELINE config 1 that is as long
 * as the kernel itself.  These METH_FASTCALL wrappers parse plain ints / floats and call straight into libmctq_sm100.so
 * (linked with rpath $ORIGIN; same symbols, same argument order as include/mctq.h, stream last).  Pure plumbing: no
 * arithmetic, no device work of its own.  The package works without it (ctypes path), only slower per call.
 */
#define PY_SSIZE_T_CLEAN
#include <Python.h>
#include <stdint.h>

#include "mctq.h"

static inline void* as_ptr(PyObject* o) {
    if (o == Py_None) return NULL;
    return (void*)(uintptr_t)PyLong_AsUnsignedLongLong(o);
}
static inline int64_t as_i64(PyObject* o) { return (int64_t)PyLong_AsLongLong(o); }
static inline int as_int(PyObject* o) { return (int)PyLong_AsLong(o); }

#define NEED(n)                                                                              \
    if (nargs != (n)) {                                                                      \
        PyErr_Format(PyExc_TypeError, "expected %d arguments, got %zd", (n), nargs);         \
        return NULL;                                                                         \
    }
#define FINISH(rc)                                   \
    if (PyErr_Occurred()) return NULL;               \
    return PyLong_FromLong((long)(rc));

/* (x, y, codes, n, dtype, scale, zp, qmin, qmax, code_mode, stream) */
static PyObject* py_fq_affine_scalar(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(11)
    const void* x = as_ptr(a[0]);
    void* y = as_ptr(a[1]);
    void* codes = as_ptr(a[2]);
    const int64_t n = as_i64(a[3]);
    const int dtype = as_int(a[4]);
    const float scale = (float)PyFloat_AsDouble(a[5]);
    const int zp = as_int(a[6]), qmin = as_int(a[7]), qmax = as_int(a[8]), code_mode = as_int(a[9]);
    void* st = as_ptr(a[10]);
    if (PyErr_Occurred()) return NULL;
    int rc = mctq_fq_affine_scalar(x, y, codes, n, dtype, scale, zp, qmin, qmax, code_mode, st);
    FINISH(rc)
}

/* (x, x2, y, n, dtype, pre_op, scale, zp, qmin, qmax, stream) */
static PyObject* py_fq_affine_scalar_pre(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(11)
    const void* x = as_ptr(a[0]);
    const void* x2 = as_ptr(a[1]);
    void* y = as_ptr(a[2]);
    const int64_t n = as_i64(a[3]);
    const int dtype = as_int(a[4]), pre = as_int(a[5]);
    const float scale = (float)PyFloat_AsDouble(a[6]);
    const int zp = as_int(a[7]), qmin = as_int(a[8]), qmax = as_int(a[9]);
    void* st = as_ptr(a[10]);
    if (PyErr_Occurred()) return NULL;
    int rc = mctq_fq_affine_scalar_pre(x, x2, y, n, dtype, pre, scale, zp, qmin, qmax, st);
    FINISH(rc)
}

/* (x, y, codes, n, dtype, scale_dev, zp_dev, C, inner, elem_offset, qmin, qmax, code_mode, stream) */
static PyObject* py_fq_affine(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(14)
    int rc = mctq_fq_affine(as_ptr(a[0]), as_ptr(a[1]), as_ptr(a[2]), as_i64(a[3]), as_int(a[4]), (const float*)as_ptr(a[5]),
                            (const int32_t*)as_ptr(a[6]), as_i64(a[7]), as_i64(a[8]), as_i64(a[9]), as_int(a[10]), as_int(a[11]),
                            as_int(a[12]), as_ptr(a[13]));
    FINISH(rc)
}

/* (x, y, codes, n, dtype, prepared_dev, C, inner, elem_offset, qmin, qmax, code_mode, stream) */
static PyObject* py_fq_affine_prepared(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(13)
    int rc = mctq_fq_affine_prepared(as_ptr(a[0]), as_ptr(a[1]), as_ptr(a[2]), as_i64(a[3]), as_int(a[4]), as_ptr(a[5]), as_i64(a[6]),
                                     as_i64(a[7]), as_i64(a[8]), as_int(a[9]), as_int(a[10]), as_int(a[11]), as_ptr(a[12]));
    FINISH(rc)
}

/* (x, y, idx, n, dtype, prepared_dev, K, bw, is_signed, C, inner, elem_offset, idx_mode, stream) */
static PyObject* py_fq_lut_prepared(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(14)
    int rc = mctq_fq_lut_prepared(as_ptr(a[0]), (float*)as_ptr(a[1]), as_ptr(a[2]), as_i64(a[3]), as_int(a[4]), as_ptr(a[5]), as_int(a[6]),
                                  as_int(a[7]), as_int(a[8]), as_i64(a[9]), as_i64(a[10]), as_i64(a[11]), as_int(a[12]), as_ptr(a[13]));
    FINISH(rc)
}

/* (sites_host_ptr, n_sites, stream) */
static PyObject* py_fq_affine_scalar_multi(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(3)
    int rc = mctq_fq_affine_scalar_multi((const MctqSiteDesc*)as_ptr(a[0]), as_int(a[1]), as_ptr(a[2]));
    FINISH(rc)
}

/* (desc_host_ptr, out_features, in_features, x, x_dtype, M, bias, y, stream) */
static PyObject* py_packed_linear(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(9)
    int rc = mctq_packed_linear((const MctqPackedDesc*)as_ptr(a[0]), as_i64(a[1]), as_i64(a[2]), as_ptr(a[3]), as_int(a[4]),
                                as_i64(a[5]), as_ptr(a[6]), as_ptr(a[7]), as_ptr(a[8]));
    FINISH(rc)
}

/* (desc_host_ptr, out_features, in_features, x, x_dtype, M, bias, y, lut_quotients_host, stream) */
static PyObject* py_packed_linear_batched(PyObject* self, PyObject* const* a, Py_ssize_t nargs) {
    NEED(10)
    int rc = mctq_packed_linear_batched((const MctqPackedDesc*)as_ptr(a[0]), as_i64(a[1]), as_i64(a[2]), as_ptr(a[3]),
                                        as_int(a[4]), as_i64(a[5]), as_ptr(a[6]), as_ptr(a[7]), (const float*)as_ptr(a[8]),
                                        as_ptr(a[9]));
    FINISH(rc)
}

static PyMethodDef methods[] = {
    {"fq_affine_scalar", (PyCFunction)(void (*)(void))py_fq_affine_scalar, METH_FASTCALL, "mctq_fq_affine_scalar"},
    {"fq_affine_scalar_pre", (PyCFunction)(void (*)(void))py_fq_affine_scalar_pre, METH_FASTCALL, "mctq_fq_affine_scalar_pre"},
    {"fq_affine", (PyCFunction)(void (*)(void))py_fq_affine, METH_FASTCALL, "mctq_fq_affine"},
    {"fq_affine_prepared", (PyCFunction)(void (*)(void))py_fq_affine_prepared, METH_FASTCALL, "mctq_fq_affine_prepared"},
    {"fq_lut_prepared", (PyCFunction)(void (*)(void))py_fq_lut_prepared, METH_FASTCALL, "mctq_fq_lut_prepared"},
    {"fq_affine_scalar_multi", (PyCFunction)(void (*)(void))py_fq_affine_scalar_multi, METH_FASTCALL, "mctq_fq_affine_scalar_multi"},
    {"packed_linear", (PyCFunction)(void (*)(void))py_packed_linear, METH_FASTCALL, "mctq_packed_linear"},
    {"packed_linear_batched", (PyCFunction)(void (*)(void))py_packed_linear_batched, METH_FASTCALL, "mctq_packed_linear_batched"},
    {NULL, NULL, 0, NULL}};

static struct PyModuleDef moddef = {PyModuleDef_HEAD_INIT, "_mctq_fast", "CPython front door to libmctq_sm100.so", -1, methods};

PyMODINIT_FUNC PyInit__mctq_fast(void) { return PyModule_Create(&moddef); }
