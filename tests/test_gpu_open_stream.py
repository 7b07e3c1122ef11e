"""Open streams (the causal feed), causal window, range-restricted batches, result delivery to unaligned pinned buffers.
Everything through the C ABI, checked against the CPU oracle (``oracle.Fast``).  Needs a B200."""
import ctypes as C
import threading

import numpy as np
import pytest

import oracle
from instaslice_b200 import engine as E
from instaslice_b200 import tables, workloads as W

pytestmark = pytest.mark.gpu


def _inventory(G, seed):
    rng = W.SplitMix64(seed)
    node_off = W.node_offsets(G // 8, 8)
    occ = ((rng.next(G) & rng.next(G)) & np.uint64(0x7F)).astype(np.uint8)
    return rng, node_off, occ


def _causal_batches(rng, ref, n_batches, n, n_profiles, min_age):
    """Batches whose FREEs name allocations placed at least ``min_age`` batches earlier; returns [(requests, oracle results)]."""
    out, aged, young = [], [], []
    for b in range(n_batches):
        while young and young[0][0] <= b - min_age:
            aged.extend(young.pop(0)[1])
        req = W.alloc_requests((rng.next(n) % np.uint64(n_profiles)).astype(np.uint8))
        for _ in range(min(len(aged), n // 3)):
            g, s, z = aged.pop(int(rng.next1() % len(aged)))
            req[int(rng.next1() % n)] = (g, 0, E.OP_FREE, s, z)
        res = ref.place(req)
        placed = res[(req["op"] == E.OP_ALLOC) & (res["status"] == E.ST_PLACED)]
        young.append((b, [(int(r["gpu"]), int(r["start"]), int(r["size"])) for r in placed]))
        out.append((req, res))
    return out


@pytest.mark.parametrize("G,n,window", [(65536, 20000, 1), (65536, 30000, 3), (4096, 3000, 2), (512, 700, 4)])
def test_open_stream_matches_oracle_batch_by_batch(G, n, window):
    """Submit with at most ``window`` batches in flight (batch b is composed only after batch b - window was waited for), results and
    final occupancy byte-identical to the oracle run batch after batch."""
    rows = E.make_profiles(tables.H100_80GB)
    rng, node_off, occ = _inventory(G, 5 + window)
    ref = oracle.Fast(node_off, rows)
    ref.load(occ)
    n_batches = 10
    batches = _causal_batches(rng, ref, n_batches, n, len(rows), window)
    eng = E.Engine(max_gpus=G, max_batch=n_batches * 65536)
    eng.load_profiles(rows)
    eng.load_inventory(node_off, occ)
    h_in = E.PinnedArray(n_batches * n, E.REQUEST_DTYPE)
    h_out = E.PinnedArray(n_batches * n, E.RESULT_DTYPE)
    h_out.array[:] = np.zeros(1, dtype=E.RESULT_DTYPE)[0]
    eng.stream_open(n_batches)
    with pytest.raises(E.EngineError):                       # the stream owns the engine
        eng.place_batch(batches[0][0])
    tickets = []
    for b, (req, want) in enumerate(batches):
        if b >= window:
            eng.stream_wait(tickets[b - window])
            assert np.array_equal(h_out.array[(b - window) * n:(b - window + 1) * n], batches[b - window][1]), b - window
        h_in.array[b * n:(b + 1) * n] = req
        tickets.append(eng.stream_submit_ptr(n, h_in.ptr + 8 * b * n, h_out.ptr + 8 * b * n))
    for b in range(n_batches):
        eng.stream_wait(tickets[b])
        assert np.array_equal(h_out.array[b * n:(b + 1) * n], batches[b][1]), b
    eng.stream_close()
    assert np.array_equal(eng.read_occupancy(), ref.occupancy())
    # the engine is usable again, and a second stream on the same engine works
    eng.load_inventory(node_off, occ)
    eng.stream_open(2)
    t0 = eng.stream_submit_ptr(n, h_in.ptr, h_out.ptr)
    eng.stream_wait(t0)
    assert np.array_equal(h_out.array[:n], batches[0][1])
    eng.stream_close()
    h_in.free(); h_out.free()
    eng.close()


def test_open_stream_closed_without_or_with_partial_use():
    rows = E.make_profiles(tables.H100_80GB)
    rng, node_off, occ = _inventory(2048, 3)
    eng = E.Engine(max_gpus=2048, max_batch=4 * 65536)
    eng.load_profiles(rows)
    eng.load_inventory(node_off, occ)
    eng.stream_open(4)
    eng.stream_close()                                       # never launched
    assert np.array_equal(eng.read_occupancy(), occ)
    eng.stream_open(4)
    with pytest.raises(E.EngineError):                       # pageable result buffer: the kernel could not write it
        req = W.alloc_requests(np.zeros(10, dtype=np.uint8))
        eng._check(eng._lib.isl_stream_submit(eng._h, 10, req.ctypes.data_as(C.c_void_p), np.zeros(10, dtype=E.RESULT_DTYPE).ctypes.data_as(C.c_void_p), None), "submit")
    eng.stream_close()
    eng.close()


def test_causal_window_on_device_resident_stream():
    """isl_set_causal_window only delays chunks; the results stay those of batch-after-batch resolution."""
    rows = E.make_profiles(tables.H100_80GB)
    rng, node_off, occ = _inventory(65536, 9)
    ref = oracle.Fast(node_off, rows)
    ref.load(occ)
    batches = _causal_batches(rng, ref, 8, 40000, len(rows), 2)
    for window in (1, 2, 5):
        eng = E.Engine(max_gpus=65536, max_batch=8 * 65536)
        eng.load_profiles(rows)
        eng.load_inventory(node_off, occ)
        eng.set_causal_window(window)
        got = eng.place_stream([b[0] for b in batches])
        for i, (g_, (_, w)) in enumerate(zip(got, batches)):
            assert np.array_equal(g_, w), (window, i)
        assert np.array_equal(eng.read_occupancy(), ref.occupancy())
        eng.close()


def test_stream_results_into_pinned_buffer_that_is_only_8_byte_aligned():
    """The delivering CTA writes 16-byte vectors; a destination offset by one record must still be correct (8-byte path)."""
    rows = E.make_profiles(tables.H100_80GB)
    rng, node_off, occ = _inventory(65536, 13)
    ref = oracle.Fast(node_off, rows)
    ref.load(occ)
    batches = _causal_batches(rng, ref, 4, 30001, len(rows), 1)
    total = sum(len(b[0]) for b in batches)
    sizes = np.array([len(b[0]) for b in batches], dtype=np.uint32)
    h_in = E.PinnedArray(total + 2, E.REQUEST_DTYPE)
    h_out = E.PinnedArray(total + 2, E.RESULT_DTYPE)
    for shift in (1, 0):
        h_in.array[shift:shift + total] = np.concatenate([b[0] for b in batches])
        h_out.array[:] = np.zeros(1, dtype=E.RESULT_DTYPE)[0]
        eng = E.Engine(max_gpus=65536, max_batch=1 << 18)
        eng.load_profiles(rows)
        eng.load_inventory(node_off, occ)
        eng.place_stream_ptr(sizes, h_in.ptr + 8 * shift, h_out.ptr + 8 * shift, device=False)
        assert np.array_equal(h_out.array[shift:shift + total], np.concatenate([b[1] for b in batches])), shift
        assert np.array_equal(eng.read_occupancy(), ref.occupancy())
        eng.close()
    h_in.free(); h_out.free()


def test_place_batch_range_is_one_node_scan_and_is_thread_safe():
    """isl_place_batch_range == findDeviceForASlice on one node's GPUs (:240-262); two threads hammering different nodes never see each
    other's restriction and the engine's own partition is untouched."""
    rows = E.make_profiles(tables.A100_40GB)
    G = 64
    node_off = W.node_offsets(8, 8)
    eng = E.Engine(max_gpus=G, max_batch=1 << 12)
    eng.load_profiles(rows)
    eng.load_inventory(node_off, np.zeros(G, dtype=np.uint8))
    p1g = tables.profile_index(tables.A100_40GB, "1g.5gb")
    errors = []

    def worker(node, count):
        lo, hi = int(node_off[node]), int(node_off[node + 1])
        for i in range(count):
            res = eng.place_batch_range(lo, hi, W.alloc_requests(np.array([p1g], dtype=np.uint8)))
            g, st = int(res["gpu"][0]), int(res["status"][0])
            want_gpu = lo + i // 7
            if st != E.ST_PLACED or g != want_gpu or int(res["start"][0]) != i % 7:
                errors.append((node, i, g, st))

    th = [threading.Thread(target=worker, args=(n, 56)) for n in (1, 6)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors[:5]
    occ = eng.read_occupancy()
    assert (occ[8:16] == 0x7F).all() and (occ[48:56] == 0x7F).all() and occ[:8].sum() == 0 and occ[16:48].sum() == 0 and occ[56:].sum() == 0
    # node 1 is full now: the range call reports the reference's error, a whole-inventory call places on node 0
    res = eng.place_batch_range(8, 16, W.alloc_requests(np.array([p1g], dtype=np.uint8)))
    assert int(res["status"][0]) == E.ST_NO_CAPACITY and int(res["start"][0]) == E.START_NONE
    res = eng.place_batch(W.alloc_requests(np.array([p1g], dtype=np.uint8)))
    assert (int(res["gpu"][0]), int(res["start"][0])) == (0, 0)
    # larger batches through the range call vs the oracle restricted by hand
    rng = W.SplitMix64(4)
    eng.load_inventory(node_off, np.zeros(G, dtype=np.uint8))
    ref = oracle.Fast(W.node_offsets(2, 8), E.make_profiles(tables.A100_40GB))
    ref.load(np.zeros(16, dtype=np.uint8))
    req = W.alloc_requests((rng.next(300) % np.uint64(len(rows))).astype(np.uint8))
    got = eng.place_batch_range(24, 40, req)
    want = ref.place(req)
    want["gpu"][want["status"] == E.ST_PLACED] += 24
    assert np.array_equal(got, want)
    with pytest.raises(E.EngineError):
        eng.place_batch_range(40, 24, req)
    eng.close()

