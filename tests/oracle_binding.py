"""ctypes binding of oracle/liboracle_synth.so (the CPU restatement). TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from parseoggvorbis_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
_LIB = None
_REF = None

IMDCT_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_float))


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(ORACLE_DIR, "liboracle_synth.so")
        srcs = [os.path.join(ORACLE_DIR, f) for f in ("synth_oracle.c", "vorbis_mdct.c")]
        if not os.path.exists(path) or os.path.getmtime(path) < max(map(os.path.getmtime, srcs)):
            subprocess.check_call(["make", "-C", ORACLE_DIR, "port"], stdout=subprocess.DEVNULL)
        L = C.CDLL(path)
        L.por_inverse_db_table.restype = C.POINTER(C.c_float)
        L.por_floor1_unwrap.restype = C.c_uint32
        L.por_floor1_db.restype = C.c_uint32
        L.por_residue_apply.restype = C.c_uint32
        L.por_synth_batch.restype = C.c_int
        L.por_synth_batch_ex.restype = C.c_int
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def inverse_db_table():
    return np.ctypeslib.as_array(lib().por_inverse_db_table(), shape=(256,)).copy()


def floor1_neighbors(xs):
    xs = np.ascontiguousarray(xs, np.uint16)
    lo = np.zeros(len(xs), np.int32)
    hi = np.zeros(len(xs), np.int32)
    lib().por_floor1_neighbors(_p(xs, C.c_uint16), len(xs), _p(lo, C.c_int), _p(hi, C.c_int))
    return lo, hi


def floor1_curve(xs, multiplier, ys, n):
    """-> (status, final_ys, step2_flag, floor[n] uint32, floor_outputs[n] float32)"""
    xs = np.ascontiguousarray(xs, np.uint16)
    ys = np.ascontiguousarray(ys, np.uint32)
    posts = len(xs)
    fy = np.zeros(posts, np.uint32)
    flag = np.zeros(posts, np.uint8)
    st = lib().por_floor1_unwrap(_p(xs, C.c_uint16), posts, int(multiplier), _p(ys, C.c_uint32),
                                 _p(fy, C.c_uint32), _p(flag, C.c_uint8))
    fl = np.zeros(n, np.uint32)
    lib().por_floor1_render(_p(xs, C.c_uint16), posts, int(multiplier), _p(fy, C.c_uint32), _p(flag, C.c_uint8),
                            C.c_uint32(n), _p(fl, C.c_uint32))
    out = np.zeros(n, np.float32)
    st |= lib().por_floor1_db(_p(fl, C.c_uint32), C.c_uint32(n), _p(out, C.c_float))
    return st, fy, flag.astype(bool), fl, out


def inverse_coupling(mag, ang):
    mag = np.array(mag, np.float32)
    ang = np.array(ang, np.float32)
    lib().por_inverse_coupling(_p(mag, C.c_float), _p(ang, C.c_float), C.c_uint32(len(mag)))
    return mag, ang


def imdct(x, kind="closed"):
    x = np.ascontiguousarray(x, np.float32)
    n = 2 * len(x)
    out = np.zeros(n, np.float32)
    fn = lib().por_imdct_closed if kind == "closed" else lib().por_imdct_fast
    fn(_p(x, C.c_float), C.c_uint32(n), _p(out, C.c_float))
    return out


def vorbis_imdct(x):
    """libvorbis' mdct_backward (oracle/vorbis_mdct.c), the reference's own transform: bit for bit on its dumps."""
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros(2 * len(x), np.float32)
    lib().por_vorbis_mdct_backward(C.c_int(len(out)), _p(x, C.c_float), _p(out, C.c_float))
    return out


def window(bs0, bs1, blockflag, prev, nxt):
    n = bs1 if blockflag else bs0
    out = np.zeros(n, np.float32)
    lib().por_window(C.c_uint32(bs0), C.c_uint32(bs1), int(blockflag), int(prev), int(nxt), _p(out, C.c_float))
    return out


def reference_lib():
    """The UNMODIFIED reference as a shared library (oracle/_ref/libparseoggvorbis_ref.so), or None."""
    global _REF
    if _REF is None:
        path = os.path.join(ORACLE_DIR, "_ref", "libparseoggvorbis_ref.so")
        if not os.path.exists(path):
            return None
        _REF = C.CDLL(path)
    return _REF


class _MdctLookup(C.Structure):  # src/mdct.h:87-97
    _fields_ = [("n", C.c_int), ("log2n", C.c_int), ("trig", C.c_void_p), ("bitrev", C.c_void_p),
                ("scale", C.c_float)]


_ref_plans = {}


def reference_imdct(x):
    """mdct_backward of the reference itself (src/mdct.h:105), as a black box."""
    ref = reference_lib()
    x = np.ascontiguousarray(x, np.float32)
    n = 2 * len(x)
    if n not in _ref_plans:
        l = _MdctLookup()
        ref.mdct_init(C.byref(l), n)
        _ref_plans[n] = l
    out = np.zeros(n, np.float32)
    ref.mdct_backward(C.byref(_ref_plans[n]), _p(x, C.c_float), _p(out, C.c_float))
    return out


def _ref_imdct_cb():
    """The reference's mdct_backward as the oracle's IMDCT callback: a C function of the oracle library that calls straight
    into oracle/_ref (no Python in the loop, so threads of the CPU baseline really run side by side)."""
    ref = reference_lib()
    L = lib()
    L.por_bind_reference_mdct.argtypes = [C.c_void_p, C.c_void_p]
    L.por_bind_reference_mdct.restype = None
    L.por_bind_reference_mdct(C.cast(ref.mdct_init, C.c_void_p), C.cast(ref.mdct_backward, C.c_void_p))
    return C.cast(L.por_imdct_reference, IMDCT_FN)


def dump_mdct_pairs(*goldens):
    """(n, input, output) of every IMDCT in reference dumps: after_envelope in, pcm_after_mdct out."""
    for g in goldens:
        oh = of = 0
        for n in g["blocksize"]:
            n = int(n)
            for _ in range(int(g["channels"])):
                yield n, g["after_envelope"][oh:oh + n // 2], g["pcm_after_mdct"][of:of + n]
                oh += n // 2
                of += n


def golden_imdct(*goldens):
    """An IMDCT callback that answers with the transforms stored in the reference dumps `goldens`, looked up by input
    vector (+0.0 and -0.0 alike): with it the oracle's window and overlap-add run on the reference's own mdct_backward
    output for those streams. An input the dumps do not hold comes back as NaN, so a comparison with the dump fails."""
    def key(n, x):
        return n, (x + np.float32(0)).tobytes()
    table = {key(n, x): y for n, x, y in dump_mdct_pairs(*goldens)}

    def cb(user, n, x, out):
        y = table.get(key(n, np.ctypeslib.as_array(x, shape=(n // 2,))))
        C.memmove(out, (y if y is not None else np.full(n, np.nan, np.float32)).ctypes.data, 4 * n)
    return IMDCT_FN(cb)


def _imdct_kind(imdct):
    """-> (kind, callback) for por_synth_batch*: "closed", "fast", "reference" (oracle/_ref) or a golden_imdct callback."""
    if isinstance(imdct, IMDCT_FN):
        return 2, imdct
    kind = {"closed": 0, "fast": 1, "reference": 2}[imdct]
    return kind, _ref_imdct_cb() if kind == 2 else C.cast(None, IMDCT_FN)


def synth_batch(setups, batch: abi.Batch, imdct="fast", capture=False):
    """Run the whole-batch oracle. setups: list of abi.Setup. Returns (pcm, status[, captures])."""
    csetups = [s.to_c() for s in setups]
    arr = (abi.pov_setup * len(csetups))(*[c.c for c in csetups])
    cb = batch.to_c()
    pcm = np.zeros(int(batch.pcm_floats), np.float32)
    status = np.zeros(len(batch.packets), np.uint32)
    kind, fn = _imdct_kind(imdct)
    if not capture:
        rc = lib().por_synth_batch(arr, len(csetups), C.byref(cb), kind, fn, None, _p(pcm, C.c_float),
                                   _p(status, C.c_uint32))
        assert rc == 0, rc
        return pcm, status
    nmax = max(max(s.blocksize) for s in setups)
    Cmax = max(s.channels for s in setups)
    P = len(batch.packets)
    ares = np.zeros((P, Cmax, nmax), np.float32)
    aenv = np.zeros((P, Cmax, nmax), np.float32)
    mdct = np.zeros((P, Cmax, nmax), np.float32)
    assert len(setups) == 1, "capture mode assumes one setup (fixed channel count)"
    rc = lib().por_synth_batch_ex(arr, len(csetups), C.byref(cb), kind, fn, None, _p(pcm, C.c_float),
                                  _p(status, C.c_uint32), _p(ares, C.c_float), _p(aenv, C.c_float),
                                  _p(mdct, C.c_float), C.c_uint32(nmax))
    assert rc == 0, rc
    return pcm, status, dict(after_residue=ares, after_envelope=aenv, pcm_after_mdct=mdct)


def snr_db(test, ref):
    test = np.asarray(test, np.float64)
    ref = np.asarray(ref, np.float64)
    err = ((test - ref) ** 2).sum()
    sig = (ref ** 2).sum()
    if err == 0:
        return float("inf")
    if sig == 0:
        return float("-inf")
    return 10 * np.log10(sig / err)


def synth_batch_raw(csetup, cbatch, imdct="fast", capture=False):
    """Whole-batch oracle on raw ctypes structs (one setup), e.g. straight from the host front-end."""
    kind, fn = _imdct_kind(imdct)
    pcm = np.zeros(int(cbatch.pcm_floats), np.float32)
    P = int(cbatch.n_packets)
    status = np.zeros(P, np.uint32)
    arr = (abi.pov_setup * 1)(csetup)
    if not capture:
        rc = lib().por_synth_batch(arr, 1, C.byref(cbatch), kind, fn, None, _p(pcm, C.c_float), _p(status, C.c_uint32))
        assert rc == 0, rc
        return pcm, status
    nmax = int(csetup.blocksize[1])
    Cn = int(csetup.channels)
    ares = np.zeros((P, Cn, nmax), np.float32)
    aenv = np.zeros((P, Cn, nmax), np.float32)
    mdct = np.zeros((P, Cn, nmax), np.float32)
    rc = lib().por_synth_batch_ex(arr, 1, C.byref(cbatch), kind, fn, None, _p(pcm, C.c_float), _p(status, C.c_uint32),
                                  _p(ares, C.c_float), _p(aenv, C.c_float), _p(mdct, C.c_float), C.c_uint32(nmax))
    assert rc == 0, rc
    return pcm, status, dict(after_residue=ares, after_envelope=aenv, pcm_after_mdct=mdct)
