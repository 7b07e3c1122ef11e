"""Tables with all ISL_MAX_PROFILES = 16 profile names, through every kernel instantiation, against the CPU oracle.

With exactly 16 names loaded the engine runs the ``kP15`` instantiations of ``k_pipeline`` (a real key of profile 15 at in-chunk index
65535 has all-ones t / profile fields, like an exhausted lane's INF), and the number of (table, profile, start) candidates picks K, the
32-lane candidate slots of ``k_pipeline`` / ``k_chain`` / ``k_small``: K = 1 up to 32 candidates, 2 up to 64, 4 up to 128.  The tables
below sit on those boundaries, and every test asserts the K and the path it claims to reach, so that a table edit that moves a case to
another instantiation fails instead of passing quietly.  Results of every batch and the final occupancy must equal ``oracle.Fast``.

The GPU tests are marked one by one: the oracle checks on the same tables at the end of the file run on any machine.
"""
import os

import numpy as np
import pytest

import oracle
from instaslice_b200 import engine as E
from instaslice_b200 import tables, workloads as W

gpu = pytest.mark.gpu

P15 = 15
BAD_IDS = (16, 17, 31, 127, 254, 255)       # profile ids past the table: ST_BAD_PROFILE, as the oracle's `p >= P`
CHUNK = 65536                               # requests per commit chunk (kChunk)
LOG_CAP = 8 * 512                           # decisions a 512-GPU segment can log (kLogCap)
Q_CAP = CHUNK + 32 * 16                     # per-profile queues of a chunk, each padded to 32 entries (kQCap)


# ---- tables -------------------------------------------------------------------------------------------------------------------

def _named(prefix, spec):
    """[(size, starts)] -> table rows named prefix00..prefix15."""
    return [("%s%02d" % (prefix, i), size, list(starts), i) for i, (size, starts) in enumerate(spec)]


# sizes 1, 2 and 4 only, and starts that are legal under both quirk sets: the same candidate count for quirks 3 and 0
_K1_32 = [(1, [0, 1, 2, 3, 4, 5, 6]), (2, [0, 2, 4]), (4, [0]), (4, [2]), (2, [4, 0]), (1, [7]), (1, [3, 5]), (2, [2]),
          (4, [1]), (1, [6, 0]), (2, [1, 3]), (4, [3]), (1, [2, 5]), (2, [5]), (1, [4, 1]), (2, [0, 2, 4])]
_K2_33 = _K1_32[:15] + [(2, [4, 2, 0, 5])]


def _four(p):
    """Four legal starts for row p, rotated through the pool of its size so that the rows differ."""
    size = (1, 2, 4)[p % 3]
    pool = {1: [7, 0, 3, 5, 1, 6, 2, 4], 2: [0, 2, 4, 1, 3, 5], 4: [0, 1, 2, 3]}[size]
    r = p % len(pool)
    return size, (pool[r:] + pool[:r])[:4]


_K2_64 = [_four(p) for p in range(16)]                                  # profile 15: size 1
_K4_65 = _K2_64[:15] + [(1, [6, 7, 0, 2, 4])]
_K4_128 = [(1, [(3 * p + 5 * j) % 8 for j in range(8)]) for p in range(16)]   # every row a permutation of 0..7

# QUIRKS_FIXED is where this table is meant to bite: sizes 3, 5, 6 and 7 are placeable there, starts run past slot 7 (never candidates),
# start orders are scrambled, and two size-1 rows name start 7
HOSTILE = [("h1a", 1, [7, 3, 0, 5], 0), ("h2a", 2, [6, 0, 3, 7], 1), ("h3a", 3, [5, 0, 2, 6], 2), ("h4a", 4, [4, 1, 5], 3),
           ("h5a", 5, [3, 0, 4], 4), ("h6a", 6, [2, 0, 3], 5), ("h7a", 7, [1, 0, 2], 6), ("h8a", 8, [0, 1], 7),
           ("h1b", 1, [0, 1, 2, 3, 4, 5, 6, 7], 8), ("h3b", 3, [0, 3], 9), ("h5b", 5, [0], 10), ("h2b", 2, [1, 5, 3], 11),
           ("h6b", 6, [1], 12), ("h7b", 7, [0], 13), ("h4b", 4, [0, 2, 4], 14), ("h1c", 1, [5, 7], 15)]

# A100-40GB + H100-80GB + A30-24GB have 14 names; a fourth node type adds two.  "2g.20gb" is 2 slices on H100 and 4 here, "1g.10gb"
# is 2 slices on A100 and 1 on H100; profile 15 ("x1g.7") exists on the fourth node type only.
CUSTOM = [("1g.5gb", 1, [7, 6, 5], 0), ("x3g.30gb", 3, [5, 0], 21), ("2g.20gb", 4, [0, 4], 1), ("x1g.7", 1, [7, 3], 22)]

# full decision log: under quirks 3 rows 0..13 (sizes 3, 5, 6, 7) are never candidates, so the table has 11 candidates and the pipeline
# may use 512-GPU segments; profile 15 takes all 8 slices of a GPU one by one
_LOG = [((3, 5, 6, 7)[p % 4], [0]) for p in range(14)] + [(2, [0, 2, 4]), (1, [7, 0, 1, 2, 3, 4, 5, 6])]

# name -> (tables, {quirks: candidates})
CASES = {
    "k1_32": ([_named("a", _K1_32)], {3: 32, 0: 32}),
    "k2_33": ([_named("b", _K2_33)], {3: 33, 0: 33}),
    "k2_64": ([_named("c", _K2_64)], {3: 64, 0: 64}),
    "k4_65": ([_named("d", _K4_65)], {3: 65, 0: 65}),
    "k4_128": ([_named("e", _K4_128)], {3: 128, 0: 128}),
    "hostile": ([HOSTILE], {3: 22, 0: 40}),
    "hetero": ([tables.A100_40GB, tables.H100_80GB, tables.A30_24GB, CUSTOM], {3: 43, 0: 52}),
    "log": ([_named("l", _LOG)], {3: 11}),
    # one name short of 16: the kP15 = false instantiations at the same K, and id 15 is past the table
    "k1_15names": ([_named("f", _K1_32[:15])], {3: 29, 0: 29}),
    "k2_15names": ([_named("g", _K2_64[:15])], {3: 60, 0: 60}),
    "k4_15names": ([_named("h", _K4_128[:15])], {3: 120, 0: 120}),
}


def slots(n_cand):
    return 1 if n_cand <= 32 else (2 if n_cand <= 64 else 4)


def profile_rows(case):
    """isl_profile records: [16] for one table, [n_tables][16] for a heterogeneous set."""
    tabs = CASES[case][0]
    return E.make_profiles(tabs[0]) if len(tabs) == 1 else E.make_profile_tables(tabs)[1]


def count_candidates(rows, quirks):
    """(table, profile, start) triples the search can ever return: a start counts when it is legal on an empty GPU as the only start
    of its row (what load_tables counts with candidate_mask)."""
    flat = np.ascontiguousarray(rows, dtype=E.PROFILE_DTYPE).reshape(-1)
    n = 0
    for r in range(len(flat)):
        for k in range(int(flat[r]["n_starts"])):
            one = flat[r:r + 1].copy()
            one["n_starts"] = 1
            one["starts"][0, 0] = flat[r]["starts"][k]
            n += oracle.start_for(one[0], quirks, 0) != E.START_NONE
    return n


class Cluster:
    """One of the CASES on n_nodes x gpn GPUs (node types drawn at random for a heterogeneous set)."""

    def __init__(self, case, quirks, n_nodes, gpn=8, seed=1):
        self.case, self.quirks = case, quirks
        self.rows = profile_rows(case)
        self.n_tables = 1 if self.rows.ndim == 1 else self.rows.shape[0]
        assert self.rows.shape[-1] == (15 if case.endswith("15names") else E.MAX_PROFILES)
        self.node_off = W.node_offsets(n_nodes, gpn)
        self.G = n_nodes * gpn
        rng = W.SplitMix64(seed)
        self.node_table = None if self.n_tables == 1 else (rng.next(n_nodes) % np.uint64(self.n_tables)).astype(np.uint8)
        self.n_cand = count_candidates(self.rows, quirks)
        assert self.n_cand == CASES[case][1][quirks], (case, quirks, self.n_cand)
        self.K = slots(self.n_cand)

    def oracle(self, occ, policy=E.POLICY_FIRST_FIT):
        ref = oracle.Fast(self.node_off, self.rows, self.quirks, policy=policy, node_table=self.node_table)
        ref.load(occ)
        return ref

    def engine(self, occ, flags=0, spec=None, policy=E.POLICY_FIRST_FIT, max_batch=1 << 18):
        eng = E.Engine(max_gpus=max(4096, self.G), max_batch=max_batch, policy=policy, quirks=self.quirks, flags=flags)
        if spec is not None:
            eng.set_speculation(spec)
        if self.n_tables == 1:
            eng.load_profiles(self.rows)
        else:
            eng.load_profile_tables(self.rows)
        eng.load_inventory(self.node_off, occ)
        if self.node_table is not None:
            eng.set_node_tables(self.node_table)
        return eng


# ---- workloads ----------------------------------------------------------------------------------------------------------------

def draw_profiles(rng, n, p15_percent=30):
    """n profile ids: p15_percent of them profile 15, about 1 % from BAD_IDS, the rest uniform over 0..15."""
    r = rng.next(n)
    prof = (r % np.uint64(16)).astype(np.uint8)
    prof[(r >> np.uint64(20)) % np.uint64(100) < np.uint64(p15_percent)] = P15
    bad = (r >> np.uint64(40)) % np.uint64(100) == 0
    prof[bad] = np.array(BAD_IDS, dtype=np.uint8)[((r >> np.uint64(48)) % np.uint64(len(BAD_IDS)))[bad].astype(np.int64)]
    return prof


def churn(rng, ref, sizes, p15_percent=30):
    """Batches of the given sizes: ALLOCs from draw_profiles, FREEs of live allocations, a NOOP; expected results from ``ref``."""
    batches, wants, live = [], [], []
    for n in sizes:
        req = W.alloc_requests(draw_profiles(rng, n, p15_percent))
        for _ in range(min(len(live), n // 4)):
            g, s, z = live.pop(int(rng.next1() % len(live)))
            req[int(rng.next1() % n)] = (g, 0, E.OP_FREE, s, z)
        if n >= 4:
            req[int(rng.next1() % n)] = (0, 0, E.OP_NOOP, 0, 0)
        res = ref.place(req)
        live.extend((int(r["gpu"]), int(r["start"]), int(r["size"])) for r in res[(req["op"] == E.OP_ALLOC) & (res["status"] == E.ST_PLACED)])
        batches.append(req)
        wants.append(res)
    return batches, wants


def assert_profile_15_places_and_runs_out(batches, wants):
    """The workload itself reaches both outcomes of profile 15, and the unknown ids."""
    req, res = np.concatenate(batches), np.concatenate(wants)
    alloc = req["op"] == E.OP_ALLOC
    st15 = res["status"][alloc & (req["profile"] == P15)]
    assert (st15 == E.ST_PLACED).any() and (st15 == E.ST_NO_CAPACITY).any()
    bad = alloc & (req["profile"] >= 16)
    assert bad.any() and (res["status"][bad] == E.ST_BAD_PROFILE).all()


def place_all(eng, batches, wants, final):
    for i, (req, want) in enumerate(zip(batches, wants)):
        got = eng.place_batch(req)
        bad = np.flatnonzero(got != want)
        assert len(bad) == 0, (i, bad[:5], got[bad[:5]], want[bad[:5]], req[bad[:5]])
    assert np.array_equal(eng.read_occupancy(), final)


def chunks(n):
    return (n + CHUNK - 1) // CHUNK


# Every path resolves a call in a known number of launches: k_few or k_small 1; the single chain 1 (prepare) + 5 per chunk (partition,
# two sweep kernels, chain, commit); the segment pipeline 3 (prepare, partition, the pipeline).  A pipeline that could not launch and fell
# back to the chunk-by-chunk path shows up here.
def expected_launches(path, sizes):
    if path in ("few", "small"):
        return len(sizes)
    if path == "chain":
        return sum(1 + 5 * chunks(n) for n in sizes)
    return 3 * len(sizes)


PATH_FLAGS = {"chain": E.FLAG_NO_PIPELINE | E.FLAG_NO_SMALL, "pipe": E.FLAG_FORCE_PIPELINE, "spec": E.FLAG_FORCE_PIPELINE}
PATH_SPEC = {"chain": None, "pipe": E.SPEC_OFF, "spec": E.SPEC_ON}


def run_path(cl, path, occ, batches, wants, final, policy=E.POLICY_FIRST_FIT, flags=0, inspect=None):
    """Place ``batches`` on a fresh engine forced onto ``path``; assert results, occupancy and the path reached.  ``inspect(eng)`` runs
    before the engine is closed."""
    eng = cl.engine(occ, flags=PATH_FLAGS[path] | flags, spec=PATH_SPEC[path], policy=policy)
    l0 = eng.stats()["kernel_launches"]
    place_all(eng, batches, wants, final)
    st = eng.stats()
    assert st["kernel_launches"] - l0 == expected_launches(path, [len(b) for b in batches]), (path, st)
    if path == "spec":
        assert st["spec_chunks"] >= len(batches), st
    else:
        assert st["spec_chunks"] == 0, st
    if inspect:
        inspect(eng)
    eng.close()
    return st


# ---- 1 + 2: every path with profile 15 live -----------------------------------------------------------------------------------

ALL_TABLES = [("k1_32", 3, 1), ("k1_32", 0, 1), ("k2_33", 3, 2), ("k2_33", 0, 2), ("k2_64", 3, 2), ("k2_64", 0, 2),
              ("k4_65", 3, 4), ("k4_65", 0, 4), ("k4_128", 3, 4), ("k4_128", 0, 4), ("hostile", 0, 2), ("hostile", 3, 1),
              ("hetero", 3, 2), ("hetero", 0, 2)]


@gpu
@pytest.mark.parametrize("case,quirks,K", ALL_TABLES)
def test_small_batches_k_few_and_k_small(case, quirks, K):
    """Batches of 1..8 requests (k_few) and of up to 1024 (k_small) on 256 GPUs that run full; the same batches again with
    ISL_NO_FEW=1, so that k_small resolves the short ones too."""
    cl = Cluster(case, quirks, 32, seed=7 + quirks)
    assert cl.K == K
    rng = W.SplitMix64(100 + K + quirks + len(case))
    occ = ((rng.next(cl.G) | rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ)
    sizes = [1 + int(rng.next1() % 8) for _ in range(40)] + [1024, 300, 8, 700, 64, 65, 5]
    batches, wants = churn(rng, ref, sizes, p15_percent=40)
    assert_profile_15_places_and_runs_out(batches, wants)
    for no_few in ("", "1"):
        os.environ.pop("ISL_NO_FEW", None)
        if no_few:
            os.environ["ISL_NO_FEW"] = "1"
        try:
            eng = cl.engine(occ)
            l0 = eng.stats()["kernel_launches"]
            place_all(eng, batches, wants, ref.occupancy())
            assert eng.stats()["kernel_launches"] - l0 == expected_launches("small", sizes)
            eng.close()
        finally:
            os.environ.pop("ISL_NO_FEW", None)


@gpu
@pytest.mark.parametrize("case,quirks,K", ALL_TABLES)
def test_chain_pipeline_and_speculative_rounds(case, quirks, K):
    """The single chain, the plain pipeline and the speculative rounds on 4096 GPUs, one batch of two chunks among them: all 12
    k_pipeline instantiations run across the parametrisation (kP15 = true here, kP15 = false in the rest of the suite)."""
    cl = Cluster(case, quirks, 512, seed=11 + quirks)
    assert cl.K == K
    rng = W.SplitMix64(200 + K + quirks + len(case))
    occ = ((rng.next(cl.G) & rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ)
    batches, wants = churn(rng, ref, [3000, 70000, 9000, 40])
    assert_profile_15_places_and_runs_out(batches, wants)
    for path in ("chain", "pipe", "spec"):
        run_path(cl, path, occ, batches, wants, ref.occupancy())


@gpu
@pytest.mark.parametrize("case,quirks,K", [("k1_15names", 0, 1), ("k2_15names", 3, 2), ("k4_15names", 0, 4)])
def test_fifteen_names_chain_pipeline_and_speculative_rounds(case, quirks, K):
    """The same workload shape with 15 names: the kP15 = false pipeline at each K, side by side with the kP15 = true runs above, and
    id 15 is one past the table."""
    cl = Cluster(case, quirks, 512, seed=15)
    assert cl.K == K
    rng = W.SplitMix64(250 + K + quirks)
    occ = ((rng.next(cl.G) & rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ)
    batches, wants = churn(rng, ref, [3000, 70000, 40])
    req, res = np.concatenate(batches), np.concatenate(wants)
    alloc = req["op"] == E.OP_ALLOC
    assert (alloc & (req["profile"] == P15)).any() and (res["status"][alloc & (req["profile"] >= 15)] == E.ST_BAD_PROFILE).all()
    for path in ("chain", "pipe", "spec"):
        run_path(cl, path, occ, batches, wants, ref.occupancy())


@gpu
@pytest.mark.parametrize("case,quirks", [("k1_32", 3), ("k4_128", 0), ("hostile", 0), ("hetero", 3)])
def test_scan_mode_with_only_profile_15(case, quirks):
    """A chunk whose only placeable profile is 15 is committed by the sweep kernels in scan mode, without a chain."""
    cl = Cluster(case, quirks, 64, seed=3)
    rng = W.SplitMix64(17 + quirks)
    occ = ((rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ)
    batches, wants, live = [], [], []
    for n in (700, 5000, 70000):
        prof = np.full(n, P15, dtype=np.uint8)
        prof[::97] = np.resize(np.array(BAD_IDS, dtype=np.uint8), len(prof[::97]))
        req = W.alloc_requests(prof)
        for _ in range(min(len(live), 50)):
            g, s, z = live.pop(int(rng.next1() % len(live)))
            req[int(rng.next1() % n)] = (g, 0, E.OP_FREE, s, z)
        res = ref.place(req)
        live.extend((int(r["gpu"]), int(r["start"]), int(r["size"])) for r in res[(req["op"] == E.OP_ALLOC) & (res["status"] == E.ST_PLACED)])
        batches.append(req)
        wants.append(res)
    assert_profile_15_places_and_runs_out(batches, wants)
    eng = cl.engine(occ, flags=E.FLAG_NO_PIPELINE | E.FLAG_NO_SMALL)
    place_all(eng, batches, wants, ref.occupancy())
    st = eng.stats()
    placed = sum(int((w["status"] == E.ST_PLACED).sum()) for w in wants)
    assert st["scan_placed"] == placed > 0, st
    assert st["chain_steps"] == 0, st
    eng.close()


@gpu
@pytest.mark.parametrize("case,quirks,K", [("k1_32", 3, 1), ("k4_128", 0, 4)])
@pytest.mark.parametrize("window", [1, 3])
def test_device_stream_with_causal_window(case, quirks, K, window):
    """Device-side stream of churn batches with a causal window: AUTO runs the speculative rounds for windows 1..3."""
    import torch
    cl = Cluster(case, quirks, 1024, seed=5)
    assert cl.K == K
    rng = W.SplitMix64(300 + window + K)
    occ = ((rng.next(cl.G) | rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)      # dense enough that profile 15 runs out
    ref = cl.oracle(occ)
    n_batches = 6
    batches, wants = churn(rng, ref, [12000] * n_batches)
    assert_profile_15_places_and_runs_out(batches, wants)
    sizes = np.array([len(b) for b in batches], dtype=np.uint32)
    d_in = torch.from_numpy(np.concatenate(batches).view(np.int64).copy()).cuda()
    d_out = torch.empty_like(d_in)
    eng = cl.engine(occ)
    eng.set_causal_window(window)
    torch.cuda.synchronize()
    eng.place_stream_ptr(sizes, d_in.data_ptr(), d_out.data_ptr(), device=True)
    eng.synchronize()
    got = d_out.cpu().numpy().view(E.RESULT_DTYPE)
    want = np.concatenate(wants)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, (bad[:5], got[bad[:5]], want[bad[:5]])
    assert np.array_equal(eng.read_occupancy(), ref.occupancy())
    assert eng.stats()["spec_chunks"] == n_batches
    eng.close()


@gpu
def test_open_stream_strictly_causal_speculative():
    """An open stream with the rounds on: batch b frees what batch b - 1 placed."""
    cl = Cluster("k2_64", 3, 1024, seed=9)
    assert cl.K == 2
    rng = W.SplitMix64(77)
    occ = ((rng.next(cl.G) | rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)       # dense enough that profile 15 runs out
    ref = cl.oracle(occ)
    n, n_batches = 12000, 5
    eng = cl.engine(occ, spec=E.SPEC_ON, max_batch=n_batches * CHUNK)
    h_in = E.PinnedArray(n_batches * n, E.REQUEST_DTYPE)
    h_out = E.PinnedArray(n_batches * n, E.RESULT_DTYPE)
    eng.stream_open(n_batches)
    live, st15 = [], []
    for b in range(n_batches):
        req = W.alloc_requests(draw_profiles(rng, n, 40))
        for _ in range(min(len(live), n // 2)):
            g, s, z = live.pop(int(rng.next1() % len(live)))
            req[int(rng.next1() % n)] = (g, 0, E.OP_FREE, s, z)
        h_in.array[b * n:(b + 1) * n] = req
        t = eng.stream_submit_ptr(n, h_in.ptr + 8 * b * n, h_out.ptr + 8 * b * n)
        eng.stream_wait(t)
        got = h_out.array[b * n:(b + 1) * n].copy()
        want = ref.place(req)
        bad = np.flatnonzero(got != want)
        assert len(bad) == 0, (b, bad[:5], got[bad[:5]], want[bad[:5]])
        live.extend((int(r["gpu"]), int(r["start"]), int(r["size"])) for r in got[(req["op"] == E.OP_ALLOC) & (got["status"] == E.ST_PLACED)])
        st15.extend(got["status"][(req["op"] == E.OP_ALLOC) & (req["profile"] == P15)])
    eng.stream_close()
    assert np.array_equal(eng.read_occupancy(), ref.occupancy())
    assert E.ST_PLACED in st15 and E.ST_NO_CAPACITY in st15
    assert eng.stats()["spec_chunks"] == n_batches
    h_in.free(); h_out.free()
    eng.close()


@gpu
def test_two_ranks_on_one_gpu_speculative():
    """A partitioned inventory over two engines in one process, the rounds on, records exchanged through each other's memory."""
    import torch
    from instaslice_b200 import dist as D
    cl = Cluster("k4_128", 3, 512, seed=13)
    assert cl.K == 4
    rng = W.SplitMix64(999)
    G = cl.G
    occ0 = ((rng.next(G) | rng.next(G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ0)
    batches, want = churn(rng, ref, [3000 + 2000 * b for b in range(5)])
    assert_profile_15_places_and_runs_out(batches, want)
    sizes = np.array([len(b) for b in batches], dtype=np.uint32)
    n_ops = int(sizes.sum())
    d_in = torch.from_numpy(np.concatenate(batches).view(np.int64).copy()).cuda()
    n_ranks = 2
    bounds = D.all_bounds(G, n_ranks, align=64)
    cuts = [lo for lo, _ in bounds] + [G]
    engines = []
    for lo, hi in bounds:
        eng = cl.engine(occ0, max_batch=1 << 16)
        eng.ipc_inbox_handle(); eng.ipc_spec_handle()          # allocate the shared buffers
        engines.append(eng)
    for r, eng in enumerate(engines):
        eng.connect_local(engines[r + 1] if r + 1 < n_ranks else None, has_prev=r > 0)
        eng.connect_owner_local(engines[0] if r > 0 else None)
        eng.set_ring_world(n_ranks)
        eng.connect_spec_local(n_ranks, r, engines, cuts)
        eng.set_causal_window(1)
        eng.set_speculation(E.SPEC_ON)
    torch.cuda.synchronize()
    for eng, (lo, hi) in zip(engines, bounds):
        eng.load_inventory(cl.node_off, occ0)
        eng.set_partition(lo, hi)
    for eng in engines:
        eng.place_stream_partitioned(sizes, d_in.data_ptr(), eng.device_results(), 1)
    for eng in engines:
        eng.synchronize()

    class _View:            # torch view of the owner's engine-owned result array (no copy)
        __cuda_array_interface__ = {"shape": (n_ops,), "typestr": "<i8", "data": (engines[0].device_results(), False), "version": 3}
    got = torch.as_tensor(_View(), device="cuda").cpu().numpy().view(E.RESULT_DTYPE)
    want = np.concatenate(want)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, (bad[:5], got[bad[:5]], want[bad[:5]])
    occ = np.concatenate([eng.read_occupancy()[lo:hi] for eng, (lo, hi) in zip(engines, bounds)])
    assert np.array_equal(occ, ref.occupancy())
    assert engines[-1].stats()["spec_chunks"] >= len(batches)
    for eng in engines:
        eng.close()


# ---- 3: chunk edges -----------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case,K", [("k1_32", 1), ("k4_128", 4)])
@pytest.mark.parametrize("n", [65535, 65536, 65537, 131077])
def test_batch_sizes_around_the_chunk(case, K, n):
    cl = Cluster(case, 3, 1024, seed=21)
    assert cl.K == K
    rng = W.SplitMix64(n + K)
    occ = ((rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ)
    batches, wants = churn(rng, ref, [n], p15_percent=50)
    assert_profile_15_places_and_runs_out(batches, wants)
    for path in ("chain", "pipe", "spec"):
        run_path(cl, path, occ, batches, wants, ref.occupancy())


def _last_of_chunk_is_profile_15(n_chunks):
    """n_chunks full chunks.  Each starts with three requests of every other profile, then NOOPs, then a tail of 300 profile-15 requests
    that ends on the chunk's last index (in-chunk t = 65535).  Free GPUs [0, 32) take the others and the head of the tail; [32, 2048) are
    full, so the tail walks across them with nothing to decide; [2048, 4096) are free and take the rest."""
    req = np.zeros(n_chunks * CHUNK, dtype=E.REQUEST_DTYPE)
    req["op"] = E.OP_NOOP
    req["handle"] = np.arange(len(req), dtype=np.uint32)
    for c in range(n_chunks):
        base = c * CHUNK
        others = np.repeat(np.arange(15, dtype=np.uint8), 3)
        req["op"][base:base + len(others)] = E.OP_ALLOC
        req["profile"][base:base + len(others)] = others
        req["op"][base + CHUNK - 300:base + CHUNK] = E.OP_ALLOC
        req["profile"][base + CHUNK - 300:base + CHUNK] = P15
    occ = np.zeros(4096, dtype=np.uint8)
    occ[32:2048] = 0xFF
    return req, occ


@gpu
@pytest.mark.parametrize("case,K", [("k1_32", 1), ("k2_64", 2), ("k4_128", 4)])
@pytest.mark.parametrize("n_chunks", [1, 2])
def test_profile_15_at_the_last_index_of_a_chunk(case, K, n_chunks):
    """A real key with t = 65535 and profile 15 has bits 11..30 all ones, as an exhausted lane's INF does: the pop test of the kP15
    instantiations must tell them apart while every other profile's queue is already exhausted."""
    cl = Cluster(case, 3, 512, seed=1)
    assert cl.K == K
    req, occ = _last_of_chunk_is_profile_15(n_chunks)
    ref = cl.oracle(occ)
    want = ref.place(req)
    for c in range(n_chunks):
        chunk_req, chunk_res = req[c * CHUNK:(c + 1) * CHUNK], want[c * CHUNK:(c + 1) * CHUNK]
        assert chunk_req["profile"][-1] == P15 and chunk_res["status"][-1] == E.ST_PLACED and chunk_res["gpu"][-1] >= 2048
        others = (chunk_req["op"] == E.OP_ALLOC) & (chunk_req["profile"] != P15)
        assert (chunk_res["status"][others] == E.ST_PLACED).all()       # their queues are exhausted long before t = 65535
    for path in ("chain", "pipe", "spec"):
        run_path(cl, path, occ, [req], [want], ref.occupancy())


@gpu
@pytest.mark.parametrize("case,quirks,K", [("k1_32", 3, 1), ("k2_64", 0, 2), ("k4_128", 3, 4)])
def test_worst_case_queue_padding(case, quirks, K):
    """A full chunk whose 16 per-profile counts are all 1 (mod 32): the padded queues take kQCap - 32 entries, the most a chunk can."""
    cl = Cluster(case, quirks, 1024, seed=2)
    assert cl.K == K
    rng = W.SplitMix64(31 + K)
    counts = np.full(16, 32 * 128 + 1)
    counts[int(rng.next1() % 16)] -= 32
    assert counts.sum() == CHUNK - 16 and (counts % 32 == 1).all()
    assert int(((counts + 31) // 32 * 32).sum()) == Q_CAP - 32
    prof = np.repeat(np.arange(16, dtype=np.uint8), counts)
    prof = prof[np.argsort(rng.next(len(prof)), kind="stable")]
    req = W.alloc_requests(np.concatenate([prof, np.zeros(16, dtype=np.uint8)]))
    occ = ((rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    tail = np.arange(CHUNK - 16, CHUNK)
    busy = np.flatnonzero(occ & 1)[:8]
    for i, g in zip(tail[:8], busy):
        req[i] = (g, 0, E.OP_FREE, 0, 1)
    req["op"][tail[8:]] = E.OP_NOOP
    assert len(req) == CHUNK and int((req["op"] == E.OP_ALLOC).sum()) == CHUNK - 16
    ref = cl.oracle(occ)
    want = ref.place(req)
    st15 = want["status"][(req["op"] == E.OP_ALLOC) & (req["profile"] == P15)]
    assert (st15 == E.ST_PLACED).any() and (st15 == E.ST_NO_CAPACITY).any()
    for path in ("chain", "pipe", "spec"):
        run_path(cl, path, occ, [req], [want], ref.occupancy())


# ---- 4: a full decision log ---------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("interleave", [False, True])
def test_full_decision_log(interleave):
    """Four whole 512-GPU segments of empty GPUs and a size-1 profile whose row names all 8 starts: every GPU takes 8 placements, so a
    stage logs exactly kLogCap decisions.  Interleaved: every fifth request is a 2-slice profile."""
    cl = Cluster("log", 3, 256, seed=4)
    assert cl.K == 1 and cl.G == 4 * 512
    occ = np.zeros(cl.G, dtype=np.uint8)
    n = 8 * cl.G + 1000
    prof = np.full(n, P15, dtype=np.uint8)
    if interleave:
        prof[::5] = 14
    prof[7::1001] = 3                       # a profile with no candidate under quirks 3: never placed
    req = W.alloc_requests(prof)
    ref = cl.oracle(occ)
    want = ref.place(req)
    placed = int((want["status"] == E.ST_PLACED).sum())
    assert (ref.occupancy() == 0xFF).all() and (want["status"][prof == 3] == E.ST_NO_CAPACITY).all()
    if not interleave:
        assert placed == 8 * cl.G
    os.environ["ISL_PIPE_SEGMENTS"] = "4"   # 512-GPU stages
    try:
        def per_stage(eng):         # decisions of every (chunk, stage) cell of the plain pipeline
            decisions = eng.read_trace()[:, :, 6]
            assert decisions.shape == (1, 4), decisions.shape
            assert int(decisions.sum()) == placed
            if not interleave:
                assert (decisions == LOG_CAP).all(), decisions

        for path in ("chain", "pipe", "spec"):
            st = run_path(cl, path, occ, [req], [want], ref.occupancy(), flags=E.FLAG_TRACE if path == "pipe" else 0,
                          inspect=per_stage if path == "pipe" else None)
            assert st["placed"] == placed
    finally:
        os.environ.pop("ISL_PIPE_SEGMENTS", None)


# ---- 5: policies and queries --------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case,quirks,K", [("k2_33", 0, 2), ("k4_128", 3, 4), ("hetero", 3, 2)])
def test_right_to_left_pipeline_and_speculative(case, quirks, K):
    cl = Cluster(case, quirks, 512, seed=8)
    assert cl.K == K
    rng = W.SplitMix64(41 + K)
    occ = ((rng.next(cl.G) & rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ, policy=E.POLICY_RIGHT_TO_LEFT)
    batches, wants = churn(rng, ref, [3000, 70000, 500])
    assert_profile_15_places_and_runs_out(batches, wants)
    for path in ("pipe", "spec"):
        run_path(cl, path, occ, batches, wants, ref.occupancy(), policy=E.POLICY_RIGHT_TO_LEFT)


@gpu
@pytest.mark.parametrize("policy", [E.POLICY_BEST_FIT, E.POLICY_MIN_FRAG])
@pytest.mark.parametrize("case,quirks", [("k1_32", 3), ("k4_128", 0), ("hostile", 0), ("hetero", 3)])
def test_best_fit_family(policy, case, quirks):
    cl = Cluster(case, quirks, 32, seed=6)
    rng = W.SplitMix64(51 + policy + quirks)
    occ = ((rng.next(cl.G) | rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    ref = cl.oracle(occ, policy=policy)
    batches, wants = churn(rng, ref, [7, 300, 900, 5])
    assert_profile_15_places_and_runs_out(batches, wants)
    eng = cl.engine(occ, policy=policy)
    place_all(eng, batches, wants, ref.occupancy())
    eng.close()


def capacity_by_hand(cl, occ):
    """Per profile: pods of that profile alone the inventory still takes — each GPU filled by repeating the reference's search with its
    own node's row."""
    rows = cl.rows.reshape(cl.n_tables, E.MAX_PROFILES)
    per_byte = np.zeros((cl.n_tables, E.MAX_PROFILES, 256), dtype=np.uint64)
    for t in range(cl.n_tables):
        for p in range(E.MAX_PROFILES):
            for o in range(256):
                cur, c = o, 0
                while (s := oracle.start_for(rows[t, p], cl.quirks, cur)) != E.START_NONE:
                    cur |= (((1 << int(rows[t, p]["size"])) - 1) << s) & 0xFF
                    c += 1
                per_byte[t, p, o] = c
    gtab = np.zeros(cl.G, dtype=np.int64)
    if cl.node_table is not None:
        gtab = np.repeat(cl.node_table.astype(np.int64), np.diff(cl.node_off.astype(np.int64)))
    return np.array([per_byte[gtab, p, occ].sum() for p in range(E.MAX_PROFILES)], dtype=np.uint64)


@gpu
@pytest.mark.parametrize("case,quirks", [("k1_32", 0), ("k4_128", 3), ("hostile", 0), ("hetero", 3), ("hetero", 0)])
def test_capacity_and_what_if(case, quirks):
    cl = Cluster(case, quirks, 256, seed=10)
    rng = W.SplitMix64(61 + quirks)
    occ = ((rng.next(cl.G) | rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    eng = cl.engine(occ)
    cap = eng.capacity()
    assert np.array_equal(cap, capacity_by_hand(cl, occ))
    assert cap[P15] > 0
    ref = cl.oracle(occ)
    plan = W.alloc_requests(draw_profiles(rng, 6000, 40))
    for i, g in enumerate(np.flatnonzero(occ & 1)[:150]):
        plan[3 * i] = (g, 0, E.OP_FREE, 0, 1)
    want = ref.place(plan)
    assert_profile_15_places_and_runs_out([plan], [want])
    got, before, after = eng.what_if(plan)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, (bad[:5], got[bad[:5]], want[bad[:5]])
    assert np.array_equal(before, cap)
    assert np.array_equal(after, capacity_by_hand(cl, ref.occupancy()))
    assert np.array_equal(eng.read_occupancy(), occ)            # the live state is back
    assert np.array_equal(eng.capacity(), cap)
    eng.close()


@gpu
@pytest.mark.parametrize("case,quirks", [("k4_128", 3), ("hostile", 0), ("k2_64", 0)])
def test_all_nodes_flag(case, quirks):
    """ISL_FLAG_ALL_NODES vs the structure-for-structure oracle with all_nodes=True on 16 nodes."""
    cl = Cluster(case, quirks, 16, seed=12)
    rng = W.SplitMix64(71 + quirks)
    occ = ((rng.next(cl.G) & rng.next(cl.G) & rng.next(cl.G)) & np.uint64(0xFF)).astype(np.uint8)
    f = oracle.Faithful(cl.node_off, cl.rows, quirks)
    f.load_occupancy_as_dangling(occ)
    eng = cl.engine(occ, flags=E.FLAG_ALL_NODES)
    st15 = []
    for rep in range(3):
        req = W.alloc_requests(draw_profiles(rng, 150, 40))
        want = f.place(req, all_nodes=True)
        got = eng.place_batch(req)
        bad = np.flatnonzero(got != want)
        assert len(bad) == 0, (rep, bad[:5], got[bad[:5]], want[bad[:5]])
        assert np.array_equal(eng.read_occupancy(), f.occupancy()), rep
        st15.extend(want["status"][req["profile"] == P15])
    assert E.ST_PLACED in st15 and E.ST_NO_CAPACITY in st15
    eng.close()


# ---- 6: profile ids past the table --------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("path", ["few", "small", "chain", "pipe", "spec", "best_fit"])
def test_ids_past_a_six_profile_table(path):
    """Ids 6..31, 127, 254 and 255 against the 6-profile H100 table on every path: no id may alias a real profile (e.g. through & 15)."""
    rows = E.make_profiles(tables.H100_80GB)
    rng = W.SplitMix64(81)
    G = 512
    node_off = W.node_offsets(G // 8, 8)
    occ = ((rng.next(G) & rng.next(G)) & np.uint64(0x7F)).astype(np.uint8)
    policy = E.POLICY_BEST_FIT if path == "best_fit" else E.POLICY_FIRST_FIT
    ref = oracle.Fast(node_off, rows, 3, policy=policy)
    ref.load(occ)
    ids = np.array(list(range(6, 32)) + [127, 254, 255], dtype=np.uint8)
    if path == "few":
        sizes = [8] * 12
    elif path == "small":
        sizes = [8] * 4 + [900]
    else:
        sizes = [3000, 70000] if path != "best_fit" else [900, 50]
    batches, wants, k = [], [], 0
    for n in sizes:
        prof = (rng.next(n) % np.uint64(6)).astype(np.uint8)
        pick = np.arange(n) % 2 == 1
        prof[pick] = ids[(k + np.arange(int(pick.sum()))) % len(ids)]     # every bad id at least once, even on the 8-request path
        k += int(pick.sum())
        req = W.alloc_requests(prof)
        res = ref.place(req)
        assert (res["status"][prof >= 6] == E.ST_BAD_PROFILE).all() and (res["status"][prof < 6] != E.ST_BAD_PROFILE).all()
        batches.append(req)
        wants.append(res)
    assert set(np.concatenate(batches)["profile"].tolist()) >= set(ids.tolist())
    if path in ("chain", "pipe", "spec"):
        flags, spec = PATH_FLAGS[path], PATH_SPEC[path]
    else:
        flags, spec = 0, None
    os.environ.pop("ISL_NO_FEW", None)
    if path == "small":
        os.environ["ISL_NO_FEW"] = "1"
    try:
        eng = E.Engine(max_gpus=4096, max_batch=1 << 18, policy=policy, flags=flags)
        if spec is not None:
            eng.set_speculation(spec)
        eng.load_profiles(rows)
        eng.load_inventory(node_off, occ)
        l0 = eng.stats()["kernel_launches"]
        place_all(eng, batches, wants, ref.occupancy())
        if path != "best_fit":
            assert eng.stats()["kernel_launches"] - l0 == expected_launches(path, sizes)
        if path == "spec":
            assert eng.stats()["spec_chunks"] >= len(sizes)
        eng.close()
    finally:
        os.environ.pop("ISL_NO_FEW", None)


# ---- CPU: the tables themselves and the oracle on them ------------------------------------------------------------------------

@pytest.mark.parametrize("case", sorted(CASES))
def test_candidate_counts_of_the_tables(case):
    """The counts each case claims (and so the K of every GPU test above), and the number of names."""
    for quirks, want in CASES[case][1].items():
        rows = profile_rows(case)
        assert rows.shape[-1] == (15 if case.endswith("15names") else E.MAX_PROFILES)
        assert count_candidates(rows, quirks) == want, (case, quirks)
    assert slots(32) == 1 and slots(33) == 2 and slots(64) == 2 and slots(65) == 4 and slots(128) == 4


def test_hetero_set_has_a_name_of_two_sizes_and_absent_names():
    names, rows = E.make_profile_tables(CASES["hetero"][0])
    assert len(names) == 16 and names[P15] == "x1g.7"
    sizes = [{int(rows[t, p]["size"]) for t in range(rows.shape[0]) if rows[t, p]["n_starts"]} for p in range(16)]
    assert any(len(s) > 1 for s in sizes)
    assert (rows["n_starts"] == 0).any(axis=0).all()            # every name is missing from at least one node type


@pytest.mark.parametrize("case", ["hostile", "k4_128", "hetero"])
@pytest.mark.parametrize("quirks", [3, 0])
def test_fast_oracle_agrees_with_faithful(case, quirks):
    """oracle.Fast (bitmask + cursors) against oracle.Faithful (the reference's structures) on the 16-name tables, random occupancy,
    frees of live allocations and ids past the table."""
    rows = profile_rows(case)
    rng = W.SplitMix64(91 + quirks + len(case))
    for trial in range(4):
        n_nodes = 2 + int(rng.next1() % 10)
        node_off = np.concatenate([[0], np.cumsum(1 + (rng.next(n_nodes) % np.uint64(4)).astype(np.int64))]).astype(np.uint32)
        G = int(node_off[-1])
        node_table = None if rows.ndim == 1 else (rng.next(n_nodes) % np.uint64(rows.shape[0])).astype(np.uint8)
        occ = ((rng.next(G) & rng.next(G)) & np.uint64(0xFF)).astype(np.uint8)
        fast = oracle.Fast(node_off, rows, quirks, node_table=node_table)
        fast.load(occ)
        faith = oracle.Faithful(node_off, rows, quirks, node_table=node_table)
        faith.load_occupancy_as_dangling(occ)
        live = []
        for batch in range(4):
            n = 5 + int(rng.next1() % 40)
            req = W.alloc_requests(draw_profiles(rng, n, 30))
            for i in range(n):
                if live and rng.next1() % 3 == 0:
                    g, s, z = live.pop(int(rng.next1() % len(live)))
                    req[i] = (g, 0, E.OP_FREE, s, z)
            a, b = fast.place(req), faith.place(req)
            assert np.array_equal(a, b), (case, quirks, trial, batch)
            assert np.array_equal(fast.occupancy(), faith.occupancy())
            live.extend((int(r["gpu"]), int(r["start"]), int(r["size"])) for r in a[(req["op"] == E.OP_ALLOC) & (a["status"] == E.ST_PLACED)])
