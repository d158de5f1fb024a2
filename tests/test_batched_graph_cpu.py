"""Batched cross-camera graphs from camera layouts, the parts that need no GPU: the segment layout helper against a brute-force
count, its rejection of malformed layouts, and every ValueError of TrackletGraph.from_cameras(ptr=) raised before device work."""
import numpy as np
import pytest

import gcn_mtmc_b200 as m


class DeviceTouched(Exception):
    pass


def layout(seg_ptr, graph_seg):
    """(E, seg_ebase) from the library's host helper; E = -1 for a malformed layout."""
    sp = np.ascontiguousarray(seg_ptr, dtype=np.int32)
    gs = np.ascontiguousarray(graph_seg, dtype=np.int32)
    eb = np.zeros(max(sp.size, 1), dtype=np.int64)
    E = m._lib.lib().mpn_cross_camera_batched_layout(sp.ctypes.data, sp.size - 1, gs.ctypes.data, gs.size - 1, eb.ctypes.data)
    return int(E), eb


def segments(cams, ptr):
    """(seg_ptr, graph_seg) of a batch: one segment per (graph, camera)."""
    first = np.zeros(cams.size, dtype=bool)
    first[ptr[:-1]] = True
    starts = np.flatnonzero(first | np.r_[True, cams[1:] != cams[:-1]])
    return np.r_[starts, cams.size], np.searchsorted(starts, ptr)


def ragged_batch(rng, n_graphs):
    """Graphs of 1..8 cameras with non-contiguous ids drawn from 0..19 (so cameras are missing from some graphs), 1..30 nodes
    per camera."""
    cams, sizes = [], []
    for _ in range(n_graphs):
        ids = np.sort(rng.choice(20, size=int(rng.integers(1, 9)), replace=False))
        c = np.repeat(ids, rng.integers(1, 31, size=ids.size))
        cams.append(c)
        sizes.append(c.size)
    return np.concatenate(cams), np.cumsum([0] + sizes)


def brute_force(cams, ptr):
    """Every row's degree counted node by node: E and the first edge of every row."""
    gid = np.repeat(np.arange(ptr.size - 1), np.diff(ptr))
    deg = np.array([np.sum((gid == gid[r]) & (cams != cams[r])) for r in range(cams.size)], dtype=np.int64)
    return int(deg.sum()), np.r_[0, np.cumsum(deg)]


@pytest.mark.parametrize("seed", range(6))
def test_layout_helper_matches_brute_force_on_ragged_batches(seed):
    rng = np.random.default_rng(seed)
    cams, ptr = ragged_batch(rng, int(rng.integers(1, 12)))
    seg_ptr, graph_seg = segments(cams, ptr)
    E, seg_ebase = layout(seg_ptr, graph_seg)
    E_bf, row_start = brute_force(cams, ptr)
    assert E == E_bf
    assert np.array_equal(seg_ebase, row_start[seg_ptr])
    per_graph = 0
    for g in range(ptr.size - 1):                     # the single-graph count, graph by graph
        cp = np.ascontiguousarray(seg_ptr[graph_seg[g]:graph_seg[g + 1] + 1] - ptr[g], dtype=np.int32)
        per_graph += m._lib.lib().mpn_cross_camera_edges(cp.ctypes.data, cp.size - 1)
    assert per_graph == E


def test_layout_helper_counts_a_uniform_batch():
    G, n, C = 2000, 300, 4
    seg_ptr = np.arange(G * C + 1) * (n // C)
    graph_seg = np.arange(G + 1) * C
    E, seg_ebase = layout(seg_ptr, graph_seg)
    assert E == G * 67500 and seg_ebase[C] == 67500 and seg_ebase[-1] == E


@pytest.mark.parametrize("seg_ptr, graph_seg", [
    ([1, 3, 6], [0, 2]),                 # nodes do not start at 0
    ([0, 3, 3, 6], [0, 3]),              # empty segment
    ([0, 4, 3, 6], [0, 3]),              # decreasing
    ([0, 3, 6], [1, 2]),                 # segments do not start at 0
    ([0, 3, 6], [0, 1]),                 # graph_seg does not end at n_segs
    ([0, 3, 6], [0, 2, 2]),              # empty graph
    ([0, 3, 6], [0, 2, 1]),              # graphs out of order
    ([0], [0, 0]),                       # no segment
    ([0, 3, 6], [0]),                    # no graph
])
def test_layout_helper_rejects_malformed_layouts(seg_ptr, graph_seg):
    assert layout(seg_ptr, graph_seg)[0] == -1


def test_layout_helper_null_arguments():
    sp = np.array([0, 3, 6], dtype=np.int32)
    gs = np.array([0, 2], dtype=np.int32)
    lib = m._lib.lib()
    assert lib.mpn_cross_camera_batched_layout(None, 2, gs.ctypes.data, 1, None) == -1
    assert lib.mpn_cross_camera_batched_layout(sp.ctypes.data, 2, None, 1, None) == -1
    assert lib.mpn_cross_camera_batched_layout(sp.ctypes.data, 2, gs.ctypes.data, 1, None) == 18     # seg_ebase is optional


@pytest.fixture
def no_device(monkeypatch):
    """Any step past the host-side checks raises DeviceTouched."""
    def touched(*a, **k):
        raise DeviceTouched()
    monkeypatch.setattr(m._lib, "require_device", touched)


@pytest.mark.parametrize("cams, ptr, kw, match", [
    ([0, 1, 0, 1, 0, 1], [0, 4, 6], {}, "grouped by ascending camera id within every graph"),
    ([0, 1, 1, 0, 2, 3], [0, 4, 6], {}, "grouped by ascending camera id within every graph"),
    ([0, 1, 0, 1, 0, 1], [0, 2, 2, 6], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [1, 2, 6], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [0, 2, 5], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [0, 4, 2, 6], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [[0, 2, 6]], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [0.0, 2.0, 6.0], {}, "strictly increasing"),
    ([0, 1, 0, 1, 0, 1], [0], {}, "strictly increasing"),
    ([0, 1, 2, 5, 0, 1], [0, 3, 4, 6], {}, "at least 2 nodes and 2 edges"),       # a graph of one node
    ([0, 1, 2, 3, 3, 3], [0, 3, 6], {}, "at least 2 nodes and 2 edges"),          # one camera: no edge
    ([0, 1, 0, 1, 0, 1], [0, 2, 4, 6], {"row_block": (0, 2)}, "cannot be row-sharded"),
])
def test_from_cameras_ptr_value_errors_before_device_work(no_device, cams, ptr, kw, match):
    with pytest.raises(ValueError, match=match):
        m.TrackletGraph.from_cameras(np.array(cams), "cuda:0", ptr=ptr, **kw)


def test_from_cameras_ptr_edge_count_limit(no_device):
    cams = np.r_[np.repeat([0, 1], 33000), [0, 1]]                     # 2 * 33000^2 > 2^31 edges in the first graph
    with pytest.raises(ValueError, match="2\\^31"):
        m.TrackletGraph.from_cameras(cams, "cuda:0", ptr=[0, 66000, 66002])


@pytest.mark.parametrize("cams, ptr", [
    ([0, 1, 0, 1, 0, 1], [0, 2, 4, 6]),          # a camera id may drop at a graph boundary
    ([2, 5, 7, 7, 0, 9], np.array([0, 4, 6])),
    ([0, 1, 2, 3], [0, 4]),                       # one graph: the single-graph path
])
def test_from_cameras_ptr_valid_layouts_reach_the_device(no_device, cams, ptr):
    with pytest.raises(DeviceTouched):
        m.TrackletGraph.from_cameras(np.array(cams), "cuda:0", ptr=ptr)

