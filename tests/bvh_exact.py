"""Layouts and exact checks shared by the node-by-node audits of the refit kernels (test_gpu_refit_kernels.py) and of the creation-time
builder (test_gpu_bvh_build.py): the ctypes layouts of MeshDev, BuildResult and RefitArgs, the refit module's loader, bit-level float
comparison, and the exact-arithmetic bound check of quantised child boxes."""
import ctypes as C
import os
from fractions import Fraction

import numpy as np

QSTEP_MAX = np.float32(2.0e6)                  # RBRT_QSTEP_MAX (common.cuh)
UNUSED_WORD = 0x0000FFFF                       # unused slot: lo 65535, hi 0 on every axis ...
DUMMY_REF = 0xFFFFFFFF                         # ... and the leaf ref make_leaf_ref(0, 1)
NAN_BITS = 0x7FFFFFFF


# ---------------------------------------------------------------- struct layouts restated from common.cuh / bvh_build.cuh
class MeshDevC(C.Structure):
    _fields_ = [("lo", C.c_float * 3), ("hi", C.c_float * 3), ("tri_base", C.c_uint32), ("n_tris", C.c_uint32), ("node_base", C.c_uint32),
                ("root_ref", C.c_int32), ("nrm_base", C.c_uint32), ("elem", C.c_uint32), ("qorg", C.c_float * 3), ("qstep", C.c_float * 3)]


class BuildResultC(C.Structure):
    _fields_ = [("live_nodes", C.c_uint32), ("depth", C.c_uint32), ("error", C.c_uint32), ("pad", C.c_uint32)]


class RefitArgsC(C.Structure):                 # update.cuh
    _fields_ = [("raw", C.c_void_p), ("n_all", C.c_uint64), ("n_eff", C.c_uint32), ("pad_rel", C.c_float), ("mesh", C.c_void_p),
                ("tris", C.c_void_p), ("normals", C.c_void_p), ("nodes", C.c_void_p), ("res", C.c_void_p)]


UPD = os.environ.get("RBRT_GPU_UPDATE_LIB") or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rbrt_b200",
                                                            "librbrt_gpu_update.so")


def update_lib():
    """librbrt_gpu_update.so with the signatures of rbrt_update_scratch_bytes and rbrt_update_refit(const RefitArgs*, scratch, stream)."""
    lib = C.CDLL(UPD)
    lib.rbrt_update_scratch_bytes.restype, lib.rbrt_update_scratch_bytes.argtypes = C.c_size_t, [C.c_uint64]
    lib.rbrt_update_refit.restype, lib.rbrt_update_refit.argtypes = C.c_int, [C.POINTER(RefitArgsC), C.c_void_p, C.c_void_p]
    return lib


def bitseq(a, b):
    """Bit-identical float32 arrays; a NaN matches any NaN (the GPU writes the canonical 0x7FFFFFFF, the host propagates payloads)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def exact_diff(v, org):
    """v - org for float32 arrays, exactly, as float64 where that is exact (TwoSum error zero), else as Fractions (object array)."""
    a, c = v.astype(np.float64), -np.float64(org)
    s = a + c
    bp = s - a
    err = (a - (s - bp)) + (c - bp)
    if np.all(err[np.isfinite(s)] == 0):
        return s
    out = s.astype(object)
    for i in np.nonzero(err != 0)[0]:
        out[i] = Fraction(float(v[i])) - Fraction(float(org))
    return out


def check_bounds(words, rows, slots, clo, chi, step, org):
    """Used slots (node `rows[i]`, slot `slots[i]`) of a [n, 16] uint32 node array whose children have the float boxes clo[i] / chi[i]
    (the union of the subtree's padded triangle boxes): the decoded bounds contain the box with a margin of >= 63/64 step, and are
    <= 3 steps away from it; an axis on which the box is NaN gets [0, 0].  Axes whose step the traversal does not read (step above
    RBRT_QSTEP_MAX: NaN qstep) are skipped.  Returns the number of bounds checked."""
    checked = 0
    for ax in range(3):
        w = words[rows, 3 * slots + ax].astype(np.int64)
        qlo, qhi = w & 0xFFFF, w >> 16
        nan = np.isnan(clo[:, ax]) | np.isnan(chi[:, ax])
        both = np.isnan(clo[:, ax]) & np.isnan(chi[:, ax])
        assert (qlo[both] == 0).all() and (qhi[both] == 0).all(), "an all-NaN box must get the build's [0, 0] words"
        if not step[ax] <= QSTEP_MAX:
            continue
        ok = ~nan
        st = np.float64(step[ax])
        dlo, dhi = exact_diff(clo[ok, ax], org[ax]), exact_diff(chi[ok, ax], org[ax])
        ql, qh = qlo[ok].astype(np.float64), qhi[ok].astype(np.float64)
        margin = 63.0 / 64.0
        # (q +- 63/64) * step and (q +- 3) * step are exact in float64 (q < 2^17, step has 24 significant bits)
        # at the ends of the grid (q = 0 or 65535: only where the 8 steps of slack vanished in the rounding of qorg, a flat axis with
        # pad_rel = 0) the bound can only be the box itself
        bad_lo = ~(((ql + margin) * st <= dlo) | ((ql == 0) & (0.0 <= dlo))) | ~((ql + 3.0) * st >= dlo)
        bad_hi = ~(((qh - margin) * st >= dhi) | ((qh == 65535) & (qh * st >= dhi))) | ~((qh - 3.0) * st <= dhi)
        assert not bad_lo.any(), (f"axis {ax}: {int(bad_lo.sum())} lower bounds not outside the box by a step, or looser than 3; first child "
                                  f"{np.nonzero(bad_lo)[0][0]}: q {ql[bad_lo][0]} box {clo[ok, ax][bad_lo][0]!r} org {org[ax]!r} step {step[ax]!r}")
        assert not bad_hi.any(), (f"axis {ax}: {int(bad_hi.sum())} upper bounds not outside the box by a step, or looser than 3; first child "
                                  f"{np.nonzero(bad_hi)[0][0]}: q {qh[bad_hi][0]} box {chi[ok, ax][bad_hi][0]!r} org {org[ax]!r} step {step[ax]!r}")
        checked += int(ok.sum())
    return checked
