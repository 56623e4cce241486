"""GPU: every compiled instance of the fp32 RDF filter on pairs at bin edges.

Group 1 holds random centres, group 2 each centre's partner at e +- t w (bin edge e, t in
[0, 4], w the frame's window half-width; _filter_model.edge_pairs, the generator of the CPU
test test_host_filter_window.py).  One batch holds a half-box frame the all-pairs kernel runs
unclamped, a half-box frame of a large box it runs clamped, an unwrapped frame (rint form)
and a frame it declines.  Every MDH_TUNE setting that selects other kernel instances runs on
a fresh context (filter_occ persists in one): ipt=2 / occ=3 / occ=4 (the all-pairs filter
instances and the IPT 2 exact kernels), fast=0 (slot_search in the exact kernels and in the
re-evaluation) and cipt=2 (the IPT 2 cell-pair instances), each over exclusions x r_lo > 0
(LOWER) x same / two groups.  arith="audit" must find no violation; "auto" and "off" must
give the oracle's counts.  Then the bin-count edges: 4095 and 4965 bins all-pairs (4966 is
refused), and the two cell-list sizes where the sub-bins drop to 0 and where the candidate
buffer is halved.
"""
import os

import numpy as np
import pytest

import _filter_model as fm

pytestmark = pytest.mark.gpu

ALLPAIRS_TUNES = ["", "ipt=2", "occ=3", "occ=4", "ipt=2,occ=3", "ipt=2,occ=4", "fast=0"]
N = 1536                      # particles per group and frame


def _lib():
    from mdhelper_b200 import _lib
    return _lib


def _thr(n_bins, rr):
    from mdhelper_b200.analysis._binning import squared_thresholds
    return squared_thresholds(n_bins, rr)


def _fit(rng, c, p, n):
    """Exactly n pairs: a random subset, or all of them repeated."""
    idx = rng.choice(len(c), n, replace=len(c) < n)
    return c[idx], p[idx]


def _frame(rng, box, n_bins, rr, kinds, region, n_shift=0, w=None):
    box = np.asarray(box, np.float32)
    edges = fm.edge_sample(n_bins, *rr, rng, n_max=40)
    if w is None:
        e = np.array([0.0] * 3 + [float(np.max(region))] * 3, np.float32)
        win = _lib().filter_window(n_bins, rr[0], rr[1], box[None], e[None])
        w = fm.window_distance(win["allpairs"], win["frames"][0]["allpairs"],
                               n_bins / (rr[1] - rr[0]))
    c, p = fm.edge_pairs(rng, box, edges, w, kinds, region, n_shift=n_shift)
    return _fit(rng, c, p, N)


def allpairs_batch(n_bins, rr, seed):
    """[F, N, 3] centres and partners and [F, 3] boxes: unclamped half-box, clamped half-box,
    rint, declined."""
    rng = np.random.default_rng(seed)
    b0 = np.array([11.0, 12.5, 13.25], np.float32)
    big = np.array([400.0, 380.0, 390.0], np.float32)
    frames = [
        _frame(rng, b0, n_bins, rr, ("inside", "axis", "h", "box", "1.5box", "d2"),
               1.5 * b0 * (1 - 2.0 ** -22)),
        _frame(rng, big, n_bins, rr, ("inside", "axis"), np.full(3, 3 * rr[1])),
        _frame(rng, b0, n_bins, rr, ("unwrap", "inside"), 40 * b0, n_shift=30),
    ]
    far = (rng.random((N, 3)) * (b0 * 2.0 ** 21)).astype(np.float32)
    frames.append((far, far + np.float32(0.5)))
    c = np.stack([f[0] for f in frames])
    p = np.stack([f[1] for f in frames])
    return c, p, np.stack([b0, big, b0, b0])


def _oracle(c, p, boxes, n_bins, rr, same, excl):
    from oracle import reference_port as rp
    out = np.zeros(n_bins, np.int64)
    for f in range(len(c)):
        dims = np.array(list(boxes[f]) + [90, 90, 90], np.float32)
        q = c[f] if same else p[f]
        out += rp.radial_histogram(c[f], q, n_bins, rr, dims, exclusion=excl,
                                   method="bruteforce")
    return out


def _run(tune, c, p, boxes, n_bins, rr, same, excl, arith, mode="allpairs"):
    L = _lib()
    old = os.environ.get("MDH_TUNE")
    os.environ["MDH_TUNE"] = tune
    ctx = L.Context(0)
    try:
        ctx.rdf_set_filter(arith)
        ctx.rdf_set_prewrap("never")
        n = c.shape[1]
        ctx.rdf_configure(n, n, same, _thr(n_bins, rr), rr[0], rr[1], exclusion=excl,
                          mode=mode)
        ctx.rdf_accumulate(c, 3 * n, None if same else p, 3 * n, boxes, len(c))
        return ctx.rdf_fetch(), ctx.rdf_filter_stats()
    finally:
        ctx.close()
        if old is None:
            os.environ.pop("MDH_TUNE", None)
        else:
            os.environ["MDH_TUNE"] = old


# (n_bins, range): the batch layout is unclamped for the first, LOWER (r_lo > 0, clamped
# layout) for the second
CONFIGS = [(201, (0.0, 14.5)), (100, (1.0, 4.5))]
_BATCH, _WANT = {}, {}


def _batch(ci):
    if ci not in _BATCH:
        _BATCH[ci] = allpairs_batch(*CONFIGS[ci], seed=100 + ci)
    return _BATCH[ci]


def _want(ci, same, excl):
    key = (ci, same, excl)
    if key not in _WANT:
        c, p, boxes = _batch(ci)
        _WANT[key] = _oracle(c, p, boxes, *CONFIGS[ci], same, excl)
    return _WANT[key]


def test_batch_layouts():
    """The batches reach the layouts and bodies the GPU cases assert."""
    for ci, (lower, unclamped) in enumerate([(0, 1), (1, 0)]):
        c, p, boxes = _batch(ci)
        e1 = np.stack([fm.extents(c[f], p[f])[0] for f in range(len(c))])
        e2 = np.stack([fm.extents(c[f], p[f])[1] for f in range(len(c))])
        w = _lib().filter_window(*CONFIGS[ci][:1], *CONFIGS[ci][1], boxes, e1, e2)
        assert w["allpairs"]["lower"] == lower
        fr = [f["allpairs"] for f in w["frames"]]
        assert [f["halfbox"] for f in fr[:3]] == [1, 1, 0]
        assert [f["unclamped"] for f in fr] == [unclamped, 0, 0, 0]
        assert [f["wlim"] > 0 for f in fr] == [True, True, True, False]


@pytest.mark.parametrize("tune", ALLPAIRS_TUNES)
def test_allpairs_instances(tune):
    for ci, (n_bins, rr) in enumerate(CONFIGS):
        c, p, boxes = _batch(ci)
        for same in (False, True):
            for excl in (None, (3, 3)):
                want = _want(ci, same, excl)
                assert want.sum() > 0
                for arith in ("audit", "auto", "off"):
                    got, st = _run(tune, c, p, boxes, n_bins, rr, same, excl, arith)
                    where = (tune, ci, same, excl, arith, st)
                    assert np.array_equal(got, want), where
                    if arith == "off":
                        continue
                    assert st["eligible"] == 1 and st["deferred_entries"] > 0, where
                    assert st["halfbox_frames"] == 2 and st["rint_frames"] == 1, where
                    assert st["declined_frames"] == 1, where
                    assert st["unclamped_frames"] == (1 - ci), where
                    if arith == "audit":
                        assert st["audit_violations"] == 0, where
                        assert st["audit_uncertain_pairs"] > 0, where


def cells_batch(n_bins, rr, seed):
    """Frames for the cell list: coordinates within one box and within 1.5 boxes."""
    rng = np.random.default_rng(seed)
    b = np.array([15.0, 15.5, 16.25], np.float32)
    kinds = ("inside", "axis", "box", "d2")
    f0 = _frame(rng, b, n_bins, rr, kinds, b * (1 - 2.0 ** -22))
    f1 = _frame(rng, b, n_bins, rr, kinds + ("1.5box",), 1.5 * b * (1 - 2.0 ** -22))
    return np.stack([f0[0], f1[0]]), np.stack([f0[1], f1[1]]), np.stack([b, b])


@pytest.mark.parametrize("tune", ["", "cipt=2"])
def test_cell_list_instances(tune):
    for n_bins, rr in [(150, (0.0, 4.5)), (150, (0.5, 4.5))]:
        c, p, boxes = cells_batch(n_bins, rr, 7)
        for same in (False, True):
            for excl in (None, (3, 3)):
                want = _oracle(c, p, boxes, n_bins, rr, same, excl)
                assert want.sum() > 0
                for arith in ("audit", "auto", "off"):
                    got, st = _run(tune, c, p, boxes, n_bins, rr, same, excl, arith,
                                   mode="cells")
                    where = (tune, rr, same, excl, arith, st)
                    assert np.array_equal(got, want), where
                    if arith != "off":
                        assert st["eligible"] == 1 and st["declined_frames"] == 0, where
                        assert st["deferred_entries"] > 0, where
                        assert st["audit_violations"] == 0, where


@pytest.mark.parametrize("n_bins", [4095, 4965])
@pytest.mark.parametrize("tune", ["", "ipt=2"])
def test_allpairs_bin_count_edges(n_bins, tune):
    """k = 9, the coarsest fixed point, and 4965 bins, the most the warp-atomic histogram
    accepts (pair_smem_bytes<WARP_ATOMIC, 4>: 40 n + 33832 <= 227 KB, whatever the ipt)."""
    rr = (0.0, 6.0)
    c, p, boxes = allpairs_batch(n_bins, rr, seed=n_bins)
    c, p, boxes = c[:3], p[:3], boxes[:3]
    want = _oracle(c, p, boxes, n_bins, rr, False, None)
    for arith in ("audit", "auto"):
        got, st = _run(tune, c, p, boxes, n_bins, rr, False, None, arith)
        assert np.array_equal(got, want), (tune, arith, st)
        assert st["eligible"] == 1 and st["audit_violations"] == 0, st
        assert st["halfbox_frames"] == 2 and st["rint_frames"] == 1, st


def test_4966_bins_are_refused():
    L = _lib()
    ctx = L.Context(0)
    try:
        with pytest.raises(ValueError):
            ctx.rdf_configure(10, 10, True, _thr(4966, (0.0, 5.0)), 0.0, 5.0)
    finally:
        ctx.close()


# cell-pair kernel sizing, restated from rdf_cells.cu (kCpWarps = 6, kCpSlack = 32,
# kCpListCap = 64, two resident blocks)
def cp_smem_bytes(n_bins, sb, cap):
    a16 = lambda x: (x + 15) // 16 * 16
    return (256 + a16(8 * (n_bins + 1)) + 6 * 2 * (cap + 32) * 16 +
            4 * 6 * (((n_bins + 2) << sb) + 32) + 4 * 6 * 64 + 8 * 6 * 2 * 32)


def cellpair_sub_bins(n_bins, sb_max, cap):
    for sb in range(sb_max, -1, -1):
        if cp_smem_bytes(n_bins, sb, cap) <= 224 * 1024 // 2:
            return sb
    return 0 if cp_smem_bytes(n_bins, 0, cap) <= 224 * 1024 else -1


def cell_plan(n1, n2, same, box, r_hi, n_bins):
    """(first cap, final cap, sub-bins) as rdf_cells_accumulate chooses them."""
    nc, _ = _lib().cells_grid(np.diag(box).astype(np.float32), r_hi, max(n1, n2))
    ncell = int(np.prod(nc))
    expect = n1 / ncell + (13.0 if same else 27.0) * n2 / ncell
    cap = int(expect + 6.0 * np.sqrt(expect) + 24.0)
    cap = min(1024, max(96, (cap + 31) // 32 * 32))
    cap0 = cap
    sb = cellpair_sub_bins(n_bins, 2, cap)
    while sb < 0 and cap > 96:
        cap = max(96, cap // 2 // 32 * 32)
        sb = cellpair_sub_bins(n_bins, 2, cap)
    return cap0, cap, sb, nc


def _cell_edge_run(n_bins, rr, box, n, same, excl, seed):
    rng = np.random.default_rng(seed)
    box = np.asarray(box, np.float32)
    c, p = _frame(rng, box, n_bins, rr, ("inside", "axis", "box"), box * (1 - 2.0 ** -22))
    # fill up to n particles per group with random ones
    idx = rng.choice(len(c), min(len(c), n // 2), replace=False)
    fill = lambda a: np.concatenate(
        [a[idx], (rng.random((n - len(idx), 3)) * box).astype(np.float32)])
    c, p = fill(c)[None], fill(p)[None]
    want = _oracle(c, p, box[None], n_bins, rr, same, excl)
    got, st = _run("", c, p, box[None], n_bins, rr, same, excl, "audit", mode="cells")
    assert np.array_equal(got, want), st
    assert st["eligible"] == 1 and st["audit_violations"] == 0 and st["declined_frames"] == 0
    assert st["deferred_entries"] > 0, st


@pytest.mark.parametrize("same,excl", [(False, None), (True, (3, 3))])
def test_cell_list_without_sub_bins(same, excl):
    """About 2000 bins at ordinary density: the per-warp histograms fit only without
    sub-bins (sb = 0)."""
    n_bins, rr, box, n = 2000, (0.0, 4.0), (40.0, 40.0, 40.0), 6000
    cap0, cap, sb, _ = cell_plan(n, n, same, box, rr[1], n_bins)
    assert cap0 == cap and sb == 0, (cap0, cap, sb)
    _cell_edge_run(n_bins, rr, box, n, same, excl, seed=2000)


@pytest.mark.parametrize("same,excl", [(False, (3, 3)), (True, None)])
def test_cell_list_with_halved_buffers(same, excl):
    """Three cells per axis holding thousands of particles: the buffers start at 1024
    candidates, where not even sb = 0 fits, and are halved (more cells take the long-list
    path)."""
    n_bins, rr, box, n = 1000, (0.0, 3.0), (9.5, 9.5, 9.5), 3000
    cap0, cap, sb, nc = cell_plan(n, n, same, box, rr[1], n_bins)
    assert nc == (3, 3, 3)
    assert cap0 == 1024 and cellpair_sub_bins(n_bins, 2, 1024) < 0
    assert cap < cap0 and sb >= 0, (cap0, cap, sb)
    _cell_edge_run(n_bins, rr, box, n, same, excl, seed=1000)
