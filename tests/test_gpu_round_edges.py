"""The rounds engine at its size boundaries, against the C oracle bit for bit.

EGS_MODE_ROUNDS changes code path at sizes the benchmark configs never reach: more than RSMAX = 96 distinct shapes in
a batch (the host forms every round's set, only 96 cold shapes get a full evaluate, NEW options of shapes outside the
set must be dropped on nodes whose rows change), the resolver instantiations at 16/17 and 32/33 shapes, k_select's
shape groups of 32, scores near the int32 guard (cand_key packs them into the top half of a 64-bit key), clusters
above 296 CTAs x 4 warps x 128 nodes = 151 552 nodes (a warp then merges several chunks), node counts at the 32-node
group / 128-node chunk / 1024-node padding edges, and more than 4 096 shapes interned over a handle's life (the
per-slot observed flags and the option tables regrow).  Every case runs the rescan engine too and compares all six
per-pod outputs, the final rows and the option caches with the oracle."""
import threading

import numpy as np
import pytest

import oracle_c as oc

pytestmark = pytest.mark.gpu

FIELDS = ["node", "status", "alloc_mask", "fit_count", "fit_digest", "score_digest"]
RSMAX = 96                      # shapes per round set, csrc/egs_rounds.cuh
MAX_MEM = 1 << 25               # EGS_MAX_MEM_PER_GPU
MAX_CORE_LOAD = 1 << 20         # EGS_MAX_CORE_LOAD
SELECT_SPAN = 296 * 4 * 128     # k_select grid cap x warps per CTA x nodes per chunk


def _egs():
    import egs_b200
    return egs_b200


# ------------------------------------------------------------------------------------------------ batches and clusters
class Batch:
    """Pods as the C ABI takes them, with explicit uids (so that several batches on one handle stay distinct)."""

    def __init__(self, shapes, pick, uid0=1):
        c_off, units = [0], []
        for s in pick:
            units.extend(shapes[int(s)])
            c_off.append(len(units))
        self.c_off = np.array(c_off, np.int32)
        self.units = np.array(units, np.int32).reshape(-1, 3)
        self.uids = np.arange(uid0, uid0 + len(pick), dtype=np.uint64)
        self.shapes = [tuple(shapes[i]) for i in dict.fromkeys(int(s) for s in pick)]   # order of first appearance

    @property
    def n_pods(self):
        return len(self.c_off) - 1

    def split(self, at):
        k = int(self.c_off[at])
        a, b = Batch.__new__(Batch), Batch.__new__(Batch)
        a.c_off, a.units, a.uids = self.c_off[:at + 1].copy(), self.units[:k].copy(), self.uids[:at].copy()
        b.c_off, b.units, b.uids = self.c_off[at:] - k, self.units[k:].copy(), self.uids[at:].copy()
        for x in (a, b):
            x.shapes = list(dict.fromkeys(tuple(tuple(int(v) for v in x.units[j]) for j in range(x.c_off[p], x.c_off[p + 1]))
                                          for p in range(x.n_pods)))
        return a, b


def _nodes_random(rng, n):
    """Heterogeneous nodes (G in 1,2,4,8, per-GPU memory 16/40/80), half of them pre-loaded."""
    nodes = []
    for _ in range(n):
        g = int(rng.choice([1, 2, 4, 8]))
        m = int(rng.choice([16, 40, 80]))
        rows = None
        if rng.integers(0, 2):
            rows = ([int(rng.choice([100, 100, 60, 30, 0])) for _ in range(g)], [int(rng.integers(0, m + 1)) for _ in range(g)])
        nodes.append((g, m, rows))
    return nodes


def _oracle(policy, nodes):
    o = oc.OracleC(policy)
    for n, (g, m, rows) in enumerate(nodes):
        assert o.add_node(100 * g, m * g) == n
        if rows is not None:
            o.set_rows(n, rows[0], rows[1])
    return o


def _load(e, nodes):
    for n, (g, m, rows) in enumerate(nodes):
        assert e.node_set(n, g, m) == 0
        if rows is not None:
            assert e.state_load(n, rows[0], rows[1]) == 0


def _gpu(policy, nodes):
    e = _egs().Egs(policy, len(nodes))
    _load(e, nodes)
    return e


def _mixed_shapes(rng, D):
    """Exactly D distinct shapes of 1..4 containers mixing fractional, whole-GPU and {-1,-1,0} units; one fractional
    unit in nine asks for 40..90 memory units, which only some GPUs hold or none, and for D > 1 the first shape fits
    no GPU at all (81 memory units), so that pods also fail to fit."""
    out = [((50, 81, 0),)] if D > 1 else []
    seen = set(out)
    while len(out) < D:
        units = []
        for _ in range(int(rng.integers(1, 5))):
            k = rng.integers(0, 10)
            if k == 0:
                units.append((-1, -1, 0))
            elif k == 1:
                units.append((0, 0, int(rng.integers(1, 3))))
            elif k == 2:
                units.append((int(rng.choice([0, 25, 50])), int(rng.integers(40, 91)), 0))
            else:
                units.append((int(rng.choice([0, 5, 10, 25, 50])), int(rng.integers(1, 12)), 0))
        t = tuple(units)
        if t not in seen:
            seen.add(t)
            out.append(t)
    return out


def _order(rng, D, P, phased):
    """Shape index of every pod; every shape gets P // D or P // D + 1 pods.  Uniform: shuffled.  Phased: each pod's
    position follows its shape index plus a spread of 60 shapes, so a window of about 60 shapes slides over the list."""
    pick = np.resize(np.arange(D), P)
    if phased:
        return pick[np.argsort(pick + rng.uniform(0, 60, P), kind="stable")]
    return rng.permutation(pick)


# ------------------------------------------------------------------------------------------------ comparisons
def _assert_outputs(ref, got, what):
    for f in FIELDS:
        bad = np.argwhere(ref[f] != got[f])
        assert len(bad) == 0, f"{what}: {f} differs first at pod {bad[0][0]} (oracle {ref[f][bad[0][0]]}, got {got[f][bad[0][0]]})"


def _assert_rows(e, o, what):
    core, mem, gc, _ = e.state_dump(0, o.n_nodes)
    for i in range(o.n_nodes):
        rows = o.rows(i)
        got = [(int(core[i, g]), int(mem[i, g])) for g in range(int(gc[i]))]
        assert got == rows, f"{what}: rows of node {i}: {got} != oracle {rows}"


def _assert_caches(e, o, shapes, what):
    """Option cache of every shape on every node: presence, score and the GPU mask of each container."""
    n = o.n_nodes
    for sh in shapes:
        req = [tuple(u) for u in sh]
        v, sc, am = o.cache_dump(req, n)
        st, gsc, gam = e.option_dump(req, 0, n)
        pres = st == 1
        bad = np.argwhere(pres != v.astype(bool))
        assert len(bad) == 0, f"{what}: cache presence of {req} differs first on node {bad[0][0]} (state {st[bad[0][0]]})"
        k = np.nonzero(pres)[0]
        bad = k[gsc[k].astype(np.int64) != sc[k]]
        assert len(bad) == 0, f"{what}: cached score of {req} differs on node {bad[0]}: {gsc[bad[0]]} != {sc[bad[0]]}"
        bad = k[(gam[k, :len(req)] != am[k, :len(req)]).any(axis=1)]
        assert len(bad) == 0, f"{what}: cached GPUs of {req} differ on node {bad[0]}"


def _run_both(policy, nodes, batches, what, on_rounds=None):
    """Oracle, rescan and rounds over the same batch sequence, each engine on a fresh handle: the outputs of every
    batch, then the final rows and the caches of every shape must equal the oracle's.  Returns the oracle outputs."""
    o = _oracle(policy, nodes)
    refs = [o.schedule_batch(b.c_off, b.units.astype(np.int64), uids=b.uids) for b in batches]
    seen = list(dict.fromkeys(sh for b in batches for sh in b.shapes))
    for mode, name in ((1, "rescan"), (2, "rounds")):
        e = _gpu(policy, nodes)
        for i, b in enumerate(batches):
            got = e.schedule_batch(b.c_off, b.units, uids=b.uids, mode=mode)
            _assert_outputs(refs[i], got, f"{what} {name} batch {i}")
            if mode == 2 and on_rounds is not None:
                on_rounds(e, i)
        _assert_rows(e, o, f"{what} {name}")
        _assert_caches(e, o, seen, f"{what} {name}")
        e.close()
    return refs


def _cat(refs, f):
    return np.concatenate([r[f] for r in refs])


# ------------------------------------------------------------------------------------------------ A: shape-set sizes
D_SWEEP = [1, 16, 17, 32, 33, 64, 65, 96, 97, 200]


def _case_a(D, policy, phased, P=4000, n_nodes=1500):
    rng = np.random.default_rng(1000 * D + 10 * policy + phased)
    nodes = _nodes_random(rng, n_nodes)
    shapes = _mixed_shapes(rng, D)
    return nodes, shapes, Batch(shapes, _order(rng, D, P, phased))


@pytest.mark.parametrize("phased", [False, True], ids=["uniform", "phased"])
@pytest.mark.parametrize("policy", [0, 1], ids=["binpack", "spread"])
@pytest.mark.parametrize("D", D_SWEEP)
def test_shape_set_sweep(D, policy, phased):
    """D distinct shapes in one batch.  The phased order runs as two batches on one handle: the second starts with
    shapes the first already evaluated, so for D > 96 its cold-shape evaluate reaches past the first round set and the
    rounds leave NEW options of shapes outside the set on nodes whose rows then change."""
    eg = _egs()
    nodes, shapes, batch = _case_a(D, policy, phased)
    assert len(batch.shapes) == D
    batches = list(batch.split(batch.n_pods // 2)) if phased else [batch]
    if phased and D >= 2 * RSMAX:
        assert len(batches[1].shapes) > RSMAX            # the second batch runs host-formed round sets too

    def path(e, i):
        if i != 0:
            return
        d1 = len(batches[0].shapes)
        launches, _ = e.profile_get(eg.capi.EGS_K_EVALUATE)
        assert launches == min(d1, RSMAX), f"{launches} full-evaluate launches for {d1} cold shapes"
        if d1 > RSMAX:
            assert e.rounds_stats()["rounds"] >= -(-d1 // RSMAX)

    refs = _run_both(policy, nodes, batches, f"D={D} policy={policy} phased={phased}", on_rounds=path)
    if D >= 17 and policy == 0:
        st = _cat(refs, "status")
        assert (st == 1).any() and (st == 3).any(), "the batch must meet both no-fit pods and stale-option bind failures"


# ------------------------------------------------------------------------------------------------ B: shapes over a handle's life
def test_many_shapes_over_handle_life():
    """Ten batches on ONE handle (and one oracle), uids continuing, each re-using old shapes and adding about 500
    new single-container ones: the handle ends with more than 4 096 interned shapes (the option tables double
    several times, the per-slot observed flags regrow past 4 096); caches made by earlier batches must survive."""
    rng = np.random.default_rng(77)
    nodes = [(8, 80, None)] * 256
    pool = [((c, m, 0),) for c in range(101) for m in range(1, 81)]
    order = rng.permutation(len(pool))
    batches, known, uid = [], [], 1
    for i in range(10):
        new = [pool[int(j)] for j in order[i * 510:(i + 1) * 510]]
        old = [known[int(j)] for j in rng.integers(0, len(known), 150)] if known else []
        shapes = new + old
        pick = rng.permutation(len(shapes))
        b = Batch(shapes, pick, uid0=uid)
        uid += b.n_pods
        batches.append(b)
        known.extend(new)
    assert len(set(known)) > 4096
    for policy in (0, 1):
        o = _oracle(policy, nodes)
        es = {1: _gpu(policy, nodes), 2: _gpu(policy, nodes)}
        seen = []
        for i, b in enumerate(batches):
            ref = o.schedule_batch(b.c_off, b.units.astype(np.int64), uids=b.uids)
            seen = list(dict.fromkeys(seen + b.shapes))
            for mode, e in es.items():
                what = f"policy {policy} mode {mode} batch {i}"
                _assert_outputs(ref, e.schedule_batch(b.c_off, b.units, uids=b.uids, mode=mode), what)
                _assert_rows(e, o, what)
                _assert_caches(e, o, seen, what)
        assert len(seen) > 4096
        for e in es.values():
            e.close()


# ------------------------------------------------------------------------------------------------ C: guard-size values
def _case_c(n_nodes=400, P=2500):
    rng = np.random.default_rng(2025)
    nodes = []
    for _ in range(n_nodes):
        g = int(rng.choice([1, 2, 4, 8]))
        core, mem = [], []
        for _ in range(g):
            k = rng.integers(0, 6)
            mem.append(MAX_MEM if k < 2 else (0 if k == 2 else int(rng.integers(0, MAX_MEM + 1))))
            core.append(int(rng.choice([100, 100, 0, int(rng.integers(0, 101))])) if rng.integers(0, 40) else MAX_CORE_LOAD)
        nodes.append((g, MAX_MEM, (core, mem)))
    mems = [1, 1 << 20, 1 << 24, MAX_MEM - 1, MAX_MEM]
    cores = [0, 1, 50, 100]
    singles = [((c, m, 0),) for c in cores for m in mems]
    multi = [tuple((int(rng.choice(cores)), int(rng.choice(mems)), 0) for _ in range(int(rng.integers(2, 5)))) for _ in range(12)]
    shapes = list(dict.fromkeys(singles + multi))
    # mostly the small requests, so that the cluster does not fill at once
    w = np.array([8.0 if sh[0][1] <= 1 << 20 else 1.0 for sh in shapes])
    pick = np.concatenate([np.arange(len(shapes)), rng.choice(len(shapes), P - len(shapes), p=w / w.sum())])
    return nodes, Batch(shapes, rng.permutation(pick))


def test_guard_size_values():
    """Per-GPU memory up to EGS_MAX_MEM_PER_GPU = 2^25 and core rows up to EGS_MAX_CORE_LOAD: binpack scores of
    ~10^9 pass k_select -> k_merge -> k_resolve_mw (packed into cand_key) and the rescan engine; the full score
    vectors of a prefix match the oracle; one unit above the guard is refused."""
    eg = _egs()
    nodes, batch = _case_c()
    refs = _run_both(0, nodes, [batch], "guard")
    assert (refs[0]["status"] == 0).sum() > batch.n_pods // 4
    vec = 300
    o = _oracle(0, nodes)
    ref = o.schedule_batch(batch.c_off, batch.units.astype(np.int64), uids=batch.uids, vec_pods=vec)
    e = _gpu(0, nodes)
    got = e.schedule_batch_vec(batch.c_off, batch.units, vec, uids=batch.uids)
    _assert_outputs(ref, got, "guard vec")
    assert np.array_equal(ref["vec_fit"], got["vec_fit"])
    assert np.array_equal(ref["vec_score"], got["vec_score"])
    assert int(got["vec_score"].max()) > 5 * 10 ** 8, "scores near the int32 guard must be reached"
    # one over the guard: refused as a whole, nothing changes
    core0, mem0, _, _ = e.state_dump()
    with pytest.raises(eg.capi.EgsError) as ex:
        e.schedule_batch(np.array([0, 1], np.int32), np.array([[10, MAX_MEM + 1, 0]], np.int32), mode=2)
    assert ex.value.status == eg.capi.EGS_ERR_OVERFLOW_GUARD
    core1, mem1, _, _ = e.state_dump()
    assert np.array_equal(core0, core1) and np.array_equal(mem0, mem1)
    e.close()


# ------------------------------------------------------------------------------------------------ D: node-count edges
N_EDGES = [1, 2, 31, 32, 33, 127, 128, 129, 1023, 1024, 1025]


def _case_d(N, n_shapes):
    """Identical nodes (2 GPUs x 40): every score ties and node order alone decides; enough pods to fill them all."""
    rng = np.random.default_rng(N * 31 + n_shapes)
    nodes = [(2, 40, None)] * N
    if n_shapes == 1:
        shapes = [((30, 8, 0),)]                                  # 3 per GPU: 6 per node
        P = 6 * N + N // 4 + 3
    else:
        shapes = list(dict.fromkeys(tuple((int(rng.choice([5, 10, 20, 30, 45])), int(rng.integers(1, 9)), 0)
                                          for _ in range(int(rng.integers(1, 3)))) for _ in range(200)))[:n_shapes]
        shapes[-1] = ((0, 0, 1),)                                 # one whole-GPU shape
        P = 30 * N + 100                                          # most pods fail on stale options before nodes fill
    assert len(shapes) == n_shapes
    return nodes, Batch(shapes, _order(rng, n_shapes, P, False))


@pytest.mark.parametrize("n_shapes", [1, 20])
@pytest.mark.parametrize("policy", [0, 1], ids=["binpack", "spread"])
@pytest.mark.parametrize("N", N_EDGES)
def test_node_count_edges(N, policy, n_shapes):
    nodes, batch = _case_d(N, n_shapes)
    refs = _run_both(policy, nodes, [batch], f"N={N} policy={policy} shapes={n_shapes}")
    st = refs[0]["status"]
    assert (st == 1).any(), "every node must fill up"
    assert (refs[0]["node"] == N - 1).any(), "the last node must win a pod"


# ------------------------------------------------------------------------------------------------ E: large clusters
def _conservation(w, out, e):
    """Size-independent property: final rows == initial rows - sum of successful binds."""
    core = w.core.astype(np.int64).copy()
    mem = w.mem.astype(np.int64).copy()
    ok = out["status"] == 0
    assert ((out["node"] >= 0) == (out["status"] != 1)).all()
    for c in range(4):
        has = ok & (np.diff(w.c_off) > c)
        pods = np.nonzero(has)[0]
        m = out["alloc_mask"][pods, c]
        assert (np.bitwise_count(m) == 1).all()
        g = np.log2(m.astype(np.float64)).astype(np.int64)
        u = w.units[w.c_off[pods] + c]
        np.subtract.at(core, (out["node"][pods], g), u[:, 0])
        np.subtract.at(mem, (out["node"][pods], g), u[:, 1])
    dc, dm, _, _ = e.state_dump()
    assert np.array_equal(dc[:, :w.gpus], core) and np.array_equal(dm[:, :w.gpus], mem)
    assert (core >= 0).all() and (mem >= 0).all()


@pytest.mark.parametrize("N", [SELECT_SPAN, SELECT_SPAN + 1, 400_000])
def test_large_cluster(N):
    """Above 151 552 nodes a k_select warp folds several 128-node chunks into its top-32 lists."""
    eg = _egs()
    w = eg.workloads.config(4, n_nodes=N, n_pods=20000)
    pre = w.prefix(1500)
    o = oc.OracleC(w.policy)
    for n in range(N):
        o.add_node(100 * w.gpus, w.mem_total * w.gpus)
        o.set_rows(n, w.core[n], w.mem[n])
    ref = o.schedule_batch(pre.c_off, pre.units64(), threads=4)
    shapes = eg.workloads.shapes_of(pre)
    assert o.cache_dump(list(shapes[0]))[0][SELECT_SPAN - 128:].any(), "the last chunks must hold candidates"
    for mode in (2, 1):
        e = eg.Egs(w.policy, N)
        e.state_load_bulk(0, w.gpus, w.mem_total, w.core, w.mem)
        got = e.schedule_batch(pre.c_off, pre.units, mode=mode)
        _assert_outputs(ref, got, f"N={N} mode {mode}")
        _assert_rows(e, o, f"N={N} mode {mode}")
        _assert_caches(e, o, shapes, f"N={N} mode {mode}")
        e.close()
    outs = []
    for mode in (1, 2):
        e = eg.Egs(w.policy, N)
        e.state_load_bulk(0, w.gpus, w.mem_total, w.core, w.mem)
        outs.append(e.schedule_batch(w.c_off, w.units, mode=mode))
        if mode == 2:
            _conservation(w, outs[-1], e)
        e.close()
    _assert_outputs(outs[0], outs[1], f"N={N} 20000 pods rounds vs rescan")


# ------------------------------------------------------------------------------------------------ F: sharded
def _sharded(policy, nodes, batch, world, what):
    """Rounds on `world` in-process shards (one thread per rank) against the oracle; every shard's rows against the
    unsharded rounds engine."""
    eg = _egs()
    cap = eg.capi
    N = len(nodes)
    o = _oracle(policy, nodes)
    ref = o.schedule_batch(batch.c_off, batch.units.astype(np.int64), uids=batch.uids)
    e0 = _gpu(policy, nodes)
    _assert_outputs(ref, e0.schedule_batch(batch.c_off, batch.units, uids=batch.uids, mode=2), f"{what} unsharded")
    ref_core, ref_mem, _, _ = e0.state_dump()
    e0.close()
    hs = []
    for r in range(world):
        e = eg.Egs(policy, N)
        e.shard_set(r, world)
        hs.append(e)
    cap.comm_init_local(hs)
    for e in hs:
        _load(e, nodes)
    outs, errs = [None] * world, []

    def run(r):
        try:
            outs[r] = hs[r].schedule_batch(batch.c_off, batch.units, uids=batch.uids, mode=cap.EGS_MODE_ROUNDS)
        except Exception as ex:   # pragma: no cover
            errs.append(repr(ex))
    th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=600)
    assert not errs, errs
    for r in range(world):
        _assert_outputs(ref, outs[r], f"{what} world {world} rank {r}")
        lo, hi = cap.shard_range(N, r, world)
        core, mem, _, _ = hs[r].state_dump(lo, hi - lo)
        assert np.array_equal(core, ref_core[lo:hi]) and np.array_equal(mem, ref_mem[lo:hi]), f"{what}: rows of shard {r}"
    for e in hs:
        e.close()


@pytest.mark.parametrize("world", [2, 8])
def test_sharded_edges(world):
    for D in (97, 200):
        for phased in (False, True):
            nodes, _, batch = _case_a(D, 0, phased)
            _sharded(0, nodes, batch, world, f"D={D} phased={phased}")
    nodes, batch = _case_c()
    _sharded(0, nodes, batch, world, "guard")
