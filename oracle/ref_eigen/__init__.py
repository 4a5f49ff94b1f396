"""ctypes wrapper of oracle/_ref/libregenie_ref_eigen*.so (TEST INFRASTRUCTURE ONLY: tests/, bench.py's CPU arms).

The library is our C++/Eigen/OpenMP restatement of the reference's level-0 and score-test arithmetic
(regenie_ref_eigen.cpp, reference file:line in its header), compiled against the reference's vendored Eigen 3.4.0 by
oracle/build_native.py."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_REF = os.path.join(os.path.dirname(_HERE), "_ref")
_lib = None
_variant = None

_u8p = ctypes.POINTER(ctypes.c_uint8)
_f64p = ctypes.POINTER(ctypes.c_double)
_i64p = ctypes.POINTER(ctypes.c_int64)


def _cpu_has(flag):
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    return flag in line.split()
    except OSError:
        pass
    return False


def available():
    return any(os.path.exists(os.path.join(_REF, n)) for n in ("libregenie_ref_eigen.so", "libregenie_ref_eigen_avx2.so"))


def lib():
    global _lib, _variant
    if _lib is not None:
        return _lib
    names = ["libregenie_ref_eigen.so"]
    if _cpu_has("avx2") and _cpu_has("fma") and os.environ.get("RG_REF_EIGEN_ISA", "") != "sse2":
        names.insert(0, "libregenie_ref_eigen_avx2.so")
    for n in names:
        p = os.path.join(_REF, n)
        if os.path.exists(p):
            _lib = ctypes.CDLL(p)
            _variant = n
            break
    if _lib is None:
        raise OSError("oracle/_ref/libregenie_ref_eigen*.so not built (python -m oracle.build_native)")
    _lib.rge_build_info.restype = ctypes.c_char_p
    _lib.rge_max_threads.restype = ctypes.c_int
    return _lib


def build_info():
    return lib().rge_build_info().decode()


def max_threads():
    return int(lib().rge_max_threads())


def default_threads():
    """Eigen's OpenMP GEMM stops scaling (and then collapses) well before 128 threads on a bs x bs result: measured on
    the 128-thread GPU host, one N=100k block takes 94 s with 128 threads against ~7 s with 8.  Callers that do not
    calibrate (the parity tests) use at most 32."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(32, n))


def _p(a, t):
    return a.ctypes.data_as(t)


def l0_block_kfold(bed_rows, N, in_analysis, X, Y, mask, fold_sizes, lam, neff, n_analyzed, threads=0, ref_first=False):
    """One level-0 block through the Eigen restatement.  Returns (W [P][N x R], phase seconds [4])."""
    bed_rows = np.ascontiguousarray(bed_rows, dtype=np.uint8)
    bs, stride = bed_rows.shape
    X = np.asfortranarray(X, dtype=np.float64); Y = np.asfortranarray(Y, dtype=np.float64)
    mask = np.asfortranarray(mask, dtype=np.uint8)
    ia = np.ascontiguousarray(in_analysis, dtype=np.uint8)
    fs = np.ascontiguousarray(fold_sizes, dtype=np.int64)
    lam = np.ascontiguousarray(lam, dtype=np.float64); neff = np.ascontiguousarray(neff, dtype=np.float64)
    C, P, R = X.shape[1], Y.shape[1], len(lam)
    W = np.zeros((P, R, N), dtype=np.float64)
    ph = np.zeros(4)
    rc = lib().rge_l0_block_kfold(_p(bed_rows, _u8p), ctypes.c_int64(stride), ctypes.c_int32(bs), ctypes.c_int64(N),
                                  _p(ia, _u8p), ctypes.c_int32(1 if ref_first else 0), _p(X, _f64p), ctypes.c_int32(C),
                                  _p(Y, _f64p), _p(mask, _u8p), ctypes.c_int32(P), _p(fs, _i64p), ctypes.c_int32(len(fs)),
                                  _p(lam, _f64p), ctypes.c_int32(R), _p(neff, _f64p), ctypes.c_int64(int(n_analyzed)),
                                  ctypes.c_int32(threads or default_threads()), _p(W, _f64p), _p(ph, _f64p))
    if rc != 0:
        raise ValueError("SNP %d has low variance" % (rc - 1))
    return [W[p].T for p in range(P)], ph


def s2_block_qt_bed(bed_rows, N, in_analysis, X, res, mask, YtX, scf_sv, n_analyzed, min_mac=5.0, threads=0):
    bed_rows = np.ascontiguousarray(bed_rows, dtype=np.uint8)
    bs, stride = bed_rows.shape
    X = np.asfortranarray(X, dtype=np.float64); res = np.asfortranarray(res, dtype=np.float64)
    mask = np.asfortranarray(mask, dtype=np.uint8); YtX = np.asfortranarray(YtX, dtype=np.float64)
    ia = np.ascontiguousarray(in_analysis, dtype=np.uint8)
    scf = np.ascontiguousarray(scf_sv, dtype=np.float64)
    C, P = X.shape[1], res.shape[1]
    out = np.zeros((bs, 4 + 5 * P))
    lib().rge_s2_block_qt_bed(_p(bed_rows, _u8p), ctypes.c_int64(stride), ctypes.c_int32(bs), ctypes.c_int64(N), _p(ia, _u8p),
                              _p(X, _f64p), ctypes.c_int32(C), _p(res, _f64p), _p(mask, _u8p), ctypes.c_int32(P),
                              _p(YtX, _f64p), _p(scf, _f64p), ctypes.c_int64(int(n_analyzed)), ctypes.c_double(min_mac),
                              ctypes.c_int32(threads or default_threads()), _p(out, _f64p))
    return out


def s2_block_bt_probs(probs, ploidy_missing, N, in_analysis, gsm, XG, yres, min_mac=5.0, threads=0):
    probs = np.ascontiguousarray(probs, dtype=np.uint8); pm = np.ascontiguousarray(ploidy_missing, dtype=np.uint8)
    bs = probs.shape[0]
    ia = np.ascontiguousarray(in_analysis, dtype=np.uint8)
    gsm = np.ascontiguousarray(gsm, dtype=np.float64).ravel(); yres = np.ascontiguousarray(yres, dtype=np.float64).ravel()
    XG = np.asfortranarray(XG, dtype=np.float64)
    out = np.zeros((bs, 4))
    lib().rge_s2_block_bt_probs(_p(probs, _u8p), _p(pm, _u8p), ctypes.c_int32(bs), ctypes.c_int64(N), _p(ia, _u8p),
                                _p(gsm, _f64p), _p(XG, _f64p), ctypes.c_int32(XG.shape[1]), _p(yres, _f64p),
                                ctypes.c_double(min_mac), ctypes.c_int32(threads or default_threads()), _p(out, _f64p))
    return out
