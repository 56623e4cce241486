"""
ctypes binding of ``libmdh_b200.so`` (C ABI: ``include/mdh_b200.h``).

There is NO CPU fallback: if the shared library is missing or cannot be loaded,
:func:`lib` raises.  Build it with ``make -C mdhelper_b200/csrc`` (or
``__graft_entry__.build()``).
"""

from __future__ import annotations

import ctypes
import pathlib

import numpy as np

import os

_HERE = pathlib.Path(__file__).resolve().parent
# MDH_B200_LIB lets a profiling session A/B another build of the same ABI
LIB_PATH = pathlib.Path(os.environ.get("MDH_B200_LIB", _HERE / "libmdh_b200.so"))

MDH_OK, MDH_EINVAL, MDH_ECUDA, MDH_ESTATE, MDH_ENOMEM = 0, -1, -2, -3, -4
MDH_HOST, MDH_DEVICE = 0, 1
RDF_MODES = {"auto": 0, "allpairs": 1, "cells": 2}
HIST_MODES = {"auto": 0, "warp_atomic": 1, "lane_private": 2}
FILTER_MODES = {"auto": 0, "off": 1, "on": 2, "audit": 3}
WRAP_MODES = {"auto": 0, "never": 1, "always": 2}
SQ_MODES = {"auto": 0, "lattice_fp64": 1, "general_fp64": 3, "lattice_fp32": 4,
            "lattice_dmma": 5}

_i32, _i64, _f64 = ctypes.c_int, ctypes.c_int64, ctypes.c_double
_p = ctypes.c_void_p

# name -> (restype, argtypes); every symbol include/mdh_b200.h declares
SIGNATURES = {
    "mdh_abi_version": (_i32, []),
    "mdh_last_error": (ctypes.c_char_p, []),
    "mdh_ctx_create": (_i32, [_i32, _p, ctypes.POINTER(_p)]),
    "mdh_ctx_destroy": (_i32, [_p]),
    "mdh_sync": (_i32, [_p]),
    "mdh_last_kernel_ms": (_i32, [_p, ctypes.POINTER(ctypes.c_float),
                                  ctypes.POINTER(ctypes.c_float)]),
    "mdh_kernel_time": (_i32, [_p, _i32, ctypes.POINTER(_f64), ctypes.POINTER(_i64),
                               ctypes.POINTER(_f64), ctypes.POINTER(_i64)]),
    "mdh_launch_count": (_i32, [_p, ctypes.POINTER(_i64)]),
    "mdh_rdf_configure": (_i32, [_p, _i64, _i64, _i32, _i32, _p, _f64, _f64, _i64,
                                 _i64, _i32, _i32, _i32]),
    "mdh_rdf_accumulate": (_i32, [_p, _p, _i64, _p, _i64, _i32, _p, _i32]),
    "mdh_rdf_accumulate_triclinic": (_i32, [_p, _p, _i64, _p, _i64, _i32, _p, _i32]),
    "mdh_rdf_triclinic_grid": (_i32, [_p, _f64, _i64, _p, ctypes.POINTER(_f64)]),
    "mdh_rdf_cells_grid": (_i32, [_p, _f64, _i64, _i32, _p, ctypes.POINTER(_f64)]),
    "mdh_rdf_filter_window": (_i32, [_i32, _f64, _f64, _i32, _i32, _i32, _f64, _i32, _p, _p,
                                     _p, _p, _p]),
    "mdh_rdf_triclinic_filter_window": (_i32, [_i32, _f64, _f64, _f64, _i32, _p, _p, _p, _p]),
    "mdh_rdf_triclinic_cells_filter_window": (_i32, [_i32, _f64, _f64, _f64, _i32, _p, _p]),
    "mdh_rdf_fetch": (_i32, [_p, _p]),
    "mdh_rdf_reset": (_i32, [_p]),
    "mdh_rdf_counts_device": (_i32, [_p, ctypes.POINTER(_p)]),
    "mdh_rdf_pair_evaluations": (_i32, [_p, ctypes.POINTER(_i64)]),
    "mdh_rdf_set_filter": (_i32, [_p, _i32]),
    "mdh_rdf_set_prewrap": (_i32, [_p, _i32]),
    "mdh_rdf_filter_stats": (_i32, [_p, _p]),
    "mdh_rdf_bin_lookup": (_i32, [_p, _p]),
    "mdh_rdf_bin_guess_audit": (_i32, [_p, _p]),
    "mdh_rdf_filter_modes": (_i32, [_p, _p]),
    "mdh_rdf_filter_unclamped": (_i32, [_p, _p]),
    "mdh_rdf_filter_cleanx": (_i32, [_p, _p]),
    "mdh_rdf_filter_triclinic": (_i32, [_p, _p]),
    "mdh_sq_configure": (_i32, [_p, _i64, _i32, _p, _i32, _p, _p, _p, _i32, _p, _i32]),
    "mdh_sq_set_cell": (_i32, [_p, _p]),
    "mdh_sq_accumulate": (_i32, [_p, _p, _i64, _i32, _i32]),
    "mdh_sq_accumulate_f64": (_i32, [_p, _p, _i64, _i32, _i32]),
    "mdh_sq_fetch": (_i32, [_p, _p]),
    "mdh_sq_kernel": (_i32, [_p, _p]),
    "mdh_sq_tiling": (_i32, [_p, _p]),
    "mdh_sq_plan": (_i32, [_i32, _p, _p, _p, _p]),
    "mdh_sq_plan_items": (_i32, [_i32, _p, _p, _p, _i64, _p]),
    "mdh_sq_reset": (_i32, [_p]),
    "mdh_sq_accum_device": (_i32, [_p, ctypes.POINTER(_p)]),
    "mdh_sq_fetch_rho": (_i32, [_p, _p]),
    "mdh_com_configure": (_i32, [_p, _i32, _i64, _i64, _p, _p]),
    "mdh_com_reduce": (_i32, [_p, _i32, _p, _i64, _i32, _i32, _p, _i64]),
    "mdh_com_reduce_f64": (_i32, [_p, _i32, _p, _i64, _i32, _i32, _p, _i64]),
    "mdh_sq_configure_chains": (_i32, [_p, _i64, _i64]),
    "mdh_isf_configure": (_i32, [_p, _i32, _i32, _i64]),
    "mdh_isf_accumulate": (_i32, [_p, _p, _i64, _i32, _i32]),
    "mdh_isf_accumulate_f64": (_i32, [_p, _p, _i64, _i32, _i32]),
    "mdh_stage_plan": (_i32, [_i32, _f64, _f64, _p, _i32, _p]),
    "mdh_isf_fetch": (_i32, [_p, _p, _p]),
}

_LIB = None


def lib() -> ctypes.CDLL:
    """Loads ``libmdh_b200.so``; raises if it has not been built."""
    global _LIB
    if _LIB is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} not found: the CUDA library has not been built "
                "(run `make -C mdhelper_b200/csrc`). mdhelper_b200 has no CPU "
                "fallback."
            )
        L = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.mdh_abi_version() != 1:
            raise RuntimeError("libmdh_b200.so ABI version mismatch")
        _LIB = L
    return _LIB


def check(rc: int) -> None:
    """Maps an ``MDH_E*`` return code to the reference-style Python exception."""
    if rc == MDH_OK:
        return
    msg = lib().mdh_last_error().decode(errors="replace")
    if rc == MDH_EINVAL:
        raise ValueError(msg)
    if rc == MDH_ENOMEM:
        raise MemoryError(msg)
    raise RuntimeError(f"libmdh_b200 error {rc}: {msg}")


def _ptr(a):
    """Address of a numpy array, a torch tensor or a raw integer address."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return int(a)
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()          # torch.Tensor


def sq_plan(lattice_n) -> dict:
    """Work decomposition of the DMMA structure-factor kernel for the lattice indices
    ``lattice_n`` (``[n_q, 3]``), computed on the host without a device: tiling statistics,
    how often every wavevector is covered (must be once) and violations of the table
    layout's column-pairing rule (must be none)."""
    ln = np.ascontiguousarray(lattice_n, dtype=np.int32).reshape(-1, 3)
    stats = (ctypes.c_int64 * 6)()
    cover = np.zeros(len(ln), dtype=np.int32)
    bad = ctypes.c_int32(0)
    check(lib().mdh_sq_plan(len(ln), ln.ctypes.data, stats, cover.ctypes.data,
                            ctypes.byref(bad)))
    return {"items": stats[0], "tiles": stats[1], "max_scheduler_tiles": stats[2],
            "schedulers": stats[3], "warps_per_block": stats[4], "smem_bytes": stats[5],
            "coverage": cover, "pair_rule_violations": bad.value}


def sq_plan_items(lattice_n) -> dict:
    """Per-warp report of both lattice plans for ``lattice_n`` (``mdh_sq_plan_items``; no
    device needed): ``mma`` is ``[items, 4]`` of ``(nt0, nt1, t0, padding)`` per warp item
    of the DMMA kernel -- ``(nt0, nt1)`` names the ``sq_mma_consume`` instance it runs --,
    ``lattice_r`` the number of nz terms ``R`` per warp of the scalar kernel (0: padding)."""
    ln = np.ascontiguousarray(lattice_n, dtype=np.int32).reshape(-1, 3)
    counts = np.zeros(2, dtype=np.int64)
    check(lib().mdh_sq_plan_items(len(ln), ln.ctypes.data, None, None, 0, counts.ctypes.data))
    cap = int(counts.max())
    mma = np.zeros((cap, 4), dtype=np.int32)
    r = np.zeros(cap, dtype=np.int32)
    check(lib().mdh_sq_plan_items(len(ln), ln.ctypes.data, mma.ctypes.data, r.ctypes.data,
                                  cap, counts.ctypes.data))
    return {"mma": mma[:counts[0]], "lattice_r": r[:counts[1]]}


def stage_plan(n_frames: int, bytes_per_frame: float, copy_over_kernel: float = 0.0) -> list:
    """Frames per piece of a host batch (``mdh_stage_plan``; no device needed): the copy of
    piece k+1 runs beside the kernels of piece k.  ``copy_over_kernel``: measured copy time
    over kernel time per frame, 0 when unknown."""
    pieces = (ctypes.c_int32 * max(1, int(n_frames)))()
    n = ctypes.c_int32(0)
    check(lib().mdh_stage_plan(int(n_frames), float(bytes_per_frame), float(copy_over_kernel),
                               pieces, len(pieces), ctypes.byref(n)))
    return list(pieces[:n.value])


def triclinic_grid(cell, r_hi: float, n_max: int):
    """Cell-list grid of one triclinic frame (``mdh_rdf_triclinic_grid``; no device
    needed): ``(cells per axis, margin M)`` for the lower-triangular ``cell`` (3x3, float32)
    and cut-off ``r_hi``; the cells are ``(0, 0, 0)`` when fewer than 3 fit on some axis.
    Every cell's perpendicular width is at least ``r_hi + M``."""
    m = np.ascontiguousarray(cell, dtype=np.float32).reshape(9)
    nc = np.zeros(3, dtype=np.int32)
    margin = _f64(0.0)
    check(lib().mdh_rdf_triclinic_grid(m.ctypes.data, float(r_hi), int(n_max), nc.ctypes.data,
                                       ctypes.byref(margin)))
    return tuple(int(v) for v in nc), margin.value


def cells_grid(cell, r_hi: float, n_max: int, drop_axis=None):
    """Cell-list grid of one frame for any cell and ``drop_axis`` (``mdh_rdf_cells_grid``; no
    device needed): ``(cells per axis, margin M)``.  A diagonal ``cell`` gets the grid of the
    orthorhombic cell list, any other the triclinic one; one cell along a dropped axis,
    ``(0, 0, 0)`` when fewer than 3 fit on a kept axis.  Raises ``ValueError`` where the
    cell list is not offered: a triclinic cell with ``drop_axis`` 0 or 1, or ``drop_axis`` 2
    with ``c_z < r_hi + M``."""
    m = np.ascontiguousarray(cell, dtype=np.float32).reshape(9)
    nc = np.zeros(3, dtype=np.int32)
    margin = _f64(0.0)
    check(lib().mdh_rdf_cells_grid(m.ctypes.data, float(r_hi), int(n_max),
                                   -1 if drop_axis is None else int(drop_axis), nc.ctypes.data,
                                   ctypes.byref(margin)))
    return tuple(int(v) for v in nc), margin.value


FILTER_LAYOUT_FIELDS = ("k", "scale", "offbase", "cbits", "span", "lg", "cb", "hslots", "lo",
                        "unclamped", "sb", "lower")
FILTER_FRAME_FIELDS = ("offm", "wlim", "halfbox", "unclamped", "mu")


def filter_window(n_bins: int, r_lo: float, r_hi: float, box, ext1, ext2=None, *,
                  drop_axis=None, ipt: int = 4, filter_occ: int = 2,
                  sqrt_err: float = 2.0 ** -22) -> dict:
    """Layout and per-frame windows of the fp32 RDF filter (``mdh_rdf_filter_window``; no
    device needed).  ``box``: ``[n_frames, 3]``; ``ext1`` / ``ext2``: ``[n_frames, 6]``
    float32 extents {min x, y, z, max x, y, z} of the two groups (``ext2=None``: one group).
    Returns ``{"clamped": layout, "allpairs": layout, "frames": [{"allpairs": window,
    "cells": window}, ...]}`` with the fields of ``FILTER_LAYOUT_FIELDS`` and
    ``FILTER_FRAME_FIELDS`` (integers as ``int``; ``scale``, ``offbase``, ``offm``, ``mu`` as
    ``float``).  Raises ``ValueError`` when the configuration is not eligible for the filter."""
    b = np.ascontiguousarray(box, dtype=np.float32).reshape(-1, 3)
    nf = len(b)
    e1 = np.ascontiguousarray(ext1, dtype=np.float32).reshape(nf, 6)
    e2 = None if ext2 is None else np.ascontiguousarray(ext2, dtype=np.float32).reshape(nf, 6)
    lay = np.zeros((2, 12), np.float64)
    fr = np.zeros((nf, 2, 5), np.float64)
    check(lib().mdh_rdf_filter_window(int(n_bins), float(r_lo), float(r_hi),
                                      -1 if drop_axis is None else int(drop_axis), int(ipt),
                                      int(filter_occ), float(sqrt_err), nf, b.ctypes.data,
                                      e1.ctypes.data, _ptr(e2), lay.ctypes.data,
                                      fr.ctypes.data))

    def typed(names, vals):
        return {n: (float(v) if n in ("scale", "offbase", "offm", "mu") else int(v))
                for n, v in zip(names, vals)}
    return {"clamped": typed(FILTER_LAYOUT_FIELDS, lay[0]),
            "allpairs": typed(FILTER_LAYOUT_FIELDS, lay[1]),
            "frames": [{"allpairs": typed(FILTER_FRAME_FIELDS, fr[f, 0]),
                        "cells": typed(FILTER_FRAME_FIELDS, fr[f, 1])} for f in range(nf)]}


TRI_FILTER_FIELDS = ("eligible", "R", "delta", "mu", "reach", "offm", "wlim", "k")


def triclinic_filter_window(n_bins: int, r_lo: float, r_hi: float, cell, ext1, ext2=None, *,
                            sqrt_err: float = 2.0 ** -22) -> list:
    """Per-frame parameters of the triclinic fp32 RDF filter
    (``mdh_rdf_triclinic_filter_window``; no device needed).  ``cell``: ``[n_frames, 3, 3]``
    lower-triangular cell matrices; ``ext1`` / ``ext2``: ``[n_frames, 6]`` float32 extents
    {min x, y, z, max x, y, z} of the two groups after the wrap into the cell (``ext2=None``:
    one group).  Returns one dict per frame with the fields of ``TRI_FILTER_FIELDS``
    (``eligible``, ``wlim``, ``k`` as ``int``, the others as ``float``).  Raises ``ValueError``
    when the configuration is not eligible for the filter or a cell is invalid."""
    c = np.ascontiguousarray(cell, dtype=np.float32).reshape(-1, 9)
    nf = len(c)
    e1 = np.ascontiguousarray(ext1, dtype=np.float32).reshape(nf, 6)
    e2 = None if ext2 is None else np.ascontiguousarray(ext2, dtype=np.float32).reshape(nf, 6)
    fr = np.zeros((nf, 8), np.float64)
    check(lib().mdh_rdf_triclinic_filter_window(int(n_bins), float(r_lo), float(r_hi),
                                                float(sqrt_err), nf, c.ctypes.data,
                                                e1.ctypes.data, _ptr(e2), fr.ctypes.data))
    return [{n: (int(v) if n in ("eligible", "wlim", "k") else float(v))
             for n, v in zip(TRI_FILTER_FIELDS, fr[f])} for f in range(nf)]


TRI_CELLS_FILTER_FIELDS = ("eligible", "A", "a", "mu", "offm", "wlim", "k")


def triclinic_cells_filter_window(n_bins: int, r_lo: float, r_hi: float, cell, *,
                                  sqrt_err: float = 2.0 ** -22) -> list:
    """Per-frame parameters of the fp32 filter of the triclinic cell list
    (``mdh_rdf_triclinic_cells_filter_window``; no device needed).  ``cell``:
    ``[n_frames, 3, 3]`` lower-triangular cell matrices; the bound depends on the cell alone.
    Returns one dict per frame with the fields of ``TRI_CELLS_FILTER_FIELDS`` (``eligible``,
    ``wlim``, ``k`` as ``int``, the others as ``float``).  Raises ``ValueError`` when the
    configuration is not eligible for the filter or a cell is invalid."""
    c = np.ascontiguousarray(cell, dtype=np.float32).reshape(-1, 9)
    nf = len(c)
    fr = np.zeros((nf, 7), np.float64)
    check(lib().mdh_rdf_triclinic_cells_filter_window(int(n_bins), float(r_lo), float(r_hi),
                                                      float(sqrt_err), nf, c.ctypes.data,
                                                      fr.ctypes.data))
    return [{n: (int(v) if n in ("eligible", "wlim", "k") else float(v))
             for n, v in zip(TRI_CELLS_FILTER_FIELDS, fr[f])} for f in range(nf)]


class Context:
    """
    One device, one stream (``mdh_ctx``).  ``stream=None`` uses torch's current
    stream on that device so that torch events and NCCL collectives order
    correctly against the kernels.
    """

    def __init__(self, device: int = 0, stream=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("mdhelper_b200 needs a CUDA device (B200, sm_100a); "
                               "there is no CPU fallback.")
        self._lib = lib()
        self.device = int(device)
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        if not stream:
            # torch's default stream has the handle 0, which the C ABI reads as "create a
            # stream of your own" -- work queued there would not be ordered against torch
            # events, uploads on side streams or NCCL.  cudaStreamLegacy (1) names the
            # default stream explicitly.
            stream = 1
        h = _p()
        check(self._lib.mdh_ctx_create(self.device, _p(stream), ctypes.byref(h)))
        self._h = h
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            self._lib.mdh_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    def sync(self):
        check(self._lib.mdh_sync(self._h))
        self._keep.clear()

    def last_kernel_ms(self):
        a, b = ctypes.c_float(), ctypes.c_float()
        check(self._lib.mdh_last_kernel_ms(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def kernel_time(self, reset: bool = False):
        """``(rdf_ms, rdf_calls, sq_ms, sq_calls)`` since the last reset."""
        a, b, na, nb = _f64(), _f64(), _i64(), _i64()
        check(self._lib.mdh_kernel_time(self._h, int(reset), ctypes.byref(a),
                                        ctypes.byref(na), ctypes.byref(b),
                                        ctypes.byref(nb)))
        return a.value, na.value, b.value, nb.value

    def launch_count(self) -> int:
        n = _i64()
        check(self._lib.mdh_launch_count(self._h, ctypes.byref(n)))
        return n.value

    # ---- seam #1 ----
    def rdf_configure(self, n1, n2, same_group, thresholds_sq, r_lo, r_hi, *,
                      exclusion=None, drop_axis=None, mode="auto", hist="auto"):
        thr = np.ascontiguousarray(thresholds_sq, dtype=np.float64)
        e1, e2 = (0, 0) if exclusion is None else (int(exclusion[0]), int(exclusion[1]))
        check(self._lib.mdh_rdf_configure(
            self._h, int(n1), int(n2), int(bool(same_group)), len(thr) - 1,
            thr.ctypes.data, float(r_lo), float(r_hi), e1, e2,
            -1 if drop_axis is None else int(drop_axis),
            RDF_MODES[mode], HIST_MODES[hist]))
        self._n_bins = len(thr) - 1

    def rdf_accumulate(self, pos1, stride1, pos2, stride2, box, n_frames, *,
                       device=False, keepalive=None):
        box = np.ascontiguousarray(box, dtype=np.float32)
        if box.shape != (n_frames, 3):
            raise ValueError("box must have shape (n_frames, 3)")
        check(self._lib.mdh_rdf_accumulate(
            self._h, _ptr(pos1), int(stride1), _ptr(pos2), int(stride2),
            MDH_DEVICE if device else MDH_HOST, box.ctypes.data, int(n_frames)))
        if keepalive is not None:
            self._keep.append(keepalive)

    def rdf_accumulate_triclinic(self, pos1, stride1, pos2, stride2, cell, n_frames, *,
                                 device=False, keepalive=None):
        """Triclinic cells: ``cell`` is ``[n_frames, 3, 3]`` (lower-triangular matrices)."""
        cell = np.ascontiguousarray(cell, dtype=np.float32)
        if cell.shape != (n_frames, 3, 3):
            raise ValueError("cell must have shape (n_frames, 3, 3)")
        check(self._lib.mdh_rdf_accumulate_triclinic(
            self._h, _ptr(pos1), int(stride1), _ptr(pos2), int(stride2),
            MDH_DEVICE if device else MDH_HOST, cell.ctypes.data, int(n_frames)))
        if keepalive is not None:
            self._keep.append(keepalive)

    def rdf_fetch(self) -> np.ndarray:
        out = np.empty(self._n_bins, dtype=np.int64)
        check(self._lib.mdh_rdf_fetch(self._h, out.ctypes.data))
        self._keep.clear()
        return out

    def rdf_reset(self):
        check(self._lib.mdh_rdf_reset(self._h))

    def rdf_set_filter(self, mode: str = "auto"):
        """fp32 filter of the all-pairs kernel: ``auto``, ``off``, ``on``, ``audit``.  It
        covers triclinic cells on the all-pairs path as well; frames whose ``r_max`` plus the
        error bound does not fit inside half the shortest of a_x, b_y, c_z (or with
        non-finite coordinates) are declined and take the 27-image fp64 arithmetic.  On the
        triclinic cell list, frames with a "far" coordinate, non-finite coordinates or a bound
        that is not small against a bin are declined and take the fp64 arithmetic of the
        cell list."""
        check(self._lib.mdh_rdf_set_filter(self._h, FILTER_MODES[mode]))

    def rdf_set_prewrap(self, mode: str = "auto"):
        """Coordinates outside the cell: ``auto`` (as the reference: moved into the cell in
        float32 whenever MDAnalysis would pick its grid search), ``never``, ``always``."""
        check(self._lib.mdh_rdf_set_prewrap(self._h, WRAP_MODES[mode]))

    def rdf_filter_stats(self) -> dict:
        out = np.zeros(12, dtype=np.int64)
        check(self._lib.mdh_rdf_filter_stats(self._h, out[:6].ctypes.data))
        check(self._lib.mdh_rdf_filter_modes(self._h, out[6:8].ctypes.data))
        check(self._lib.mdh_rdf_filter_unclamped(self._h, out[8:9].ctypes.data))
        check(self._lib.mdh_rdf_filter_cleanx(self._h, out[9:10].ctypes.data))
        check(self._lib.mdh_rdf_filter_triclinic(self._h, out[10:].ctypes.data))
        return dict(zip(("deferred_entries", "inline_entries", "audit_violations",
                         "audit_uncertain_pairs", "declined_frames", "eligible",
                         "halfbox_frames", "rint_frames", "unclamped_frames",
                         "cleanx_pairs", "triclinic_frames", "triclinic_exact_pairs"),
                        (int(v) for v in out)))

    def rdf_bin_lookup(self) -> dict:
        """Which bin lookup the configured run uses (``fast``: the branch-free guess, else the
        binary search) and the disagreements of its configure-time self-check."""
        out = np.zeros(2, dtype=np.int64)
        check(self._lib.mdh_rdf_bin_lookup(self._h, out.ctypes.data))
        return {"fast": int(out[0]), "selfcheck_bad": int(out[1])}

    def rdf_bin_guess_audit(self) -> dict:
        """The bin guess of the configured thresholds checked for every d2 >= 0, inf and NaN
        (``mdh_rdf_bin_guess_audit``): classes checked, disagreements, the bits of the
        smallest bad d2 (-1: none) and its fast slot minus its exact slot."""
        out = np.zeros(4, dtype=np.int64)
        check(self._lib.mdh_rdf_bin_guess_audit(self._h, out.ctypes.data))
        return dict(zip(("classes", "bad", "first_bits", "slot_diff"), (int(v) for v in out)))

    def rdf_pair_evaluations(self) -> int:
        n = _i64()
        check(self._lib.mdh_rdf_pair_evaluations(self._h, ctypes.byref(n)))
        return n.value

    # ---- seam #2 ----
    def sq_configure(self, n_total, group_offsets, wavevectors, pairs, *,
                     lattice_n=None, lattice_b=None, mode="auto"):
        goff = np.ascontiguousarray(group_offsets, dtype=np.int64)
        wv = np.ascontiguousarray(wavevectors, dtype=np.float64)
        pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        ln = lb = None
        if lattice_n is not None:
            ln = np.ascontiguousarray(lattice_n, dtype=np.int32)
            lb = np.ascontiguousarray(lattice_b, dtype=np.float64)
            if ln.shape != wv.shape or lb.shape != (3,):
                raise ValueError("lattice_n must match wavevectors; lattice_b is (3,)")
        # an unchanged configuration (run() after run() on the same object) only needs its
        # accumulator cleared, not the work items rebuilt and uploaded
        key = (int(n_total), goff.tobytes(), wv.tobytes(), pr.tobytes(),
               None if ln is None else ln.tobytes(), None if lb is None else lb.tobytes(), mode)
        if key == getattr(self, "_sq_key", None):
            check(self._lib.mdh_sq_reset(self._h))
            return
        self._sq_key = None
        check(self._lib.mdh_sq_configure(
            self._h, int(n_total), len(goff) - 1, goff.ctypes.data, len(wv),
            wv.ctypes.data, _ptr(ln), _ptr(lb), len(pr), pr.ctypes.data,
            SQ_MODES[mode]))
        self._sq_key = key
        self._sq_shape = (len(pr), len(wv))
        self._sq_nrho = 1 if (pr < 0).any() else len(goff) - 1

    def sq_set_cell(self, cell):
        """Coordinates enter the Fourier sums as fractional coordinates of ``cell`` (the
        ``[3, 3]`` lower-triangular cell matrix, or ``None`` to clear it); the configured
        wavevectors are then ``k = q H^T`` (``mdh_sq_set_cell``)."""
        h = None if cell is None else np.ascontiguousarray(cell, dtype=np.float64).reshape(9)
        check(self._lib.mdh_sq_set_cell(self._h, _ptr(h)))
        if h is not None and getattr(self, "_sq_key", None) is not None:
            # the reset shortcut of sq_configure must not reuse a context whose cell differs
            self._sq_key = (self._sq_key, h.tobytes())

    def sq_accumulate(self, pos, stride, n_frames, *, device=False, keepalive=None,
                      f64=False):
        """``f64``: ``pos`` holds float64 coordinates (``stride`` in doubles)."""
        fn = self._lib.mdh_sq_accumulate_f64 if f64 else self._lib.mdh_sq_accumulate
        check(fn(
            self._h, _ptr(pos), int(stride),
            MDH_DEVICE if device else MDH_HOST, int(n_frames)))
        if keepalive is not None:
            self._keep.append(keepalive)

    def sq_fetch(self) -> np.ndarray:
        out = np.empty(self._sq_shape, dtype=np.float64)
        check(self._lib.mdh_sq_fetch(self._h, out.ctypes.data))
        self._keep.clear()
        return out

    def sq_kernel(self) -> str:
        """Name of the kernel strategy the current configuration runs."""
        m = ctypes.c_int(0)
        check(self._lib.mdh_sq_kernel(self._h, ctypes.byref(m)))
        return {v: k for k, v in SQ_MODES.items()}[m.value]

    def sq_tiling(self) -> dict:
        """Tiling statistics of the DMMA lattice kernel (zeros for the other kernels)."""
        st = (ctypes.c_int64 * 4)()
        check(self._lib.mdh_sq_tiling(self._h, st))
        return {"items": st[0], "tiles": st[1], "max_scheduler_tiles": st[2],
                "schedulers": st[3]}

    def sq_reset(self):
        check(self._lib.mdh_sq_reset(self._h))

    # ---- centres of mass of consecutive atom runs ----
    def com_configure(self, slot: int, starts, masses):
        st = np.ascontiguousarray(starts, dtype=np.int64)
        m = np.ascontiguousarray(masses, dtype=np.float64)
        check(self._lib.mdh_com_configure(self._h, int(slot), len(m), len(st) - 1,
                                          st.ctypes.data, m.ctypes.data))

    def com_reduce(self, slot: int, pos, stride, n_frames, out_device, out_stride, *,
                   device=False, f64=False):
        """``f64``: ``out_device`` is a float64 buffer (``out_stride`` in doubles)."""
        fn = self._lib.mdh_com_reduce_f64 if f64 else self._lib.mdh_com_reduce
        check(fn(self._h, int(slot), _ptr(pos), int(stride),
                 MDH_DEVICE if device else MDH_HOST, int(n_frames),
                 _ptr(out_device), int(out_stride)))

    def sq_configure_chains(self, n_chains: int, n_monomers: int):
        """Single-chain mode: ``sq_accumulate`` adds sum over chains of |rho_chain|^2."""
        self._sq_key = None                      # C-side state now differs from a plain configure
        check(self._lib.mdh_sq_configure_chains(self._h, int(n_chains), int(n_monomers)))

    # ---- intermediate scattering function (after sq_configure) ----
    def isf_configure(self, n_lags: int, incoherent: bool, max_frames: int):
        check(self._lib.mdh_isf_configure(self._h, int(n_lags), int(bool(incoherent)),
                                          int(max_frames)))
        self._isf = (int(n_lags), bool(incoherent))

    def isf_accumulate(self, pos, stride, n_frames, *, device=False, keepalive=None,
                       f64=False):
        fn = self._lib.mdh_isf_accumulate_f64 if f64 else self._lib.mdh_isf_accumulate
        check(fn(
            self._h, _ptr(pos), int(stride),
            MDH_DEVICE if device else MDH_HOST, int(n_frames)))
        if keepalive is not None:
            self._keep.append(keepalive)

    def isf_fetch(self):
        """``(cisf[n_lags, n_pairs, n_q], iisf[n_lags, n_rho, n_q] or None)``, raw sums."""
        n_lags, inc = self._isf
        n_pairs, n_q = self._sq_shape
        cisf = np.empty((n_lags, n_pairs, n_q), dtype=np.float64)
        iisf = np.empty((n_lags, self._sq_nrho, n_q), dtype=np.float64) if inc else None
        check(self._lib.mdh_isf_fetch(self._h, cisf.ctypes.data, _ptr(iisf)))
        self._keep.clear()
        return cisf, iisf

    def sq_fetch_rho(self) -> np.ndarray:
        out = np.empty((self._sq_nrho, self._sq_shape[1]), dtype=np.complex128)
        check(self._lib.mdh_sq_fetch_rho(self._h, out.ctypes.data))
        return out
