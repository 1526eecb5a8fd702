"""The device kernels at every resource count D = 1..8 and under non-default node-sort weights.

Every hot kernel is a template instance per D (yk_sweep_kernel<D,..>, yk_lattice_kernel<D>, the uniform-run kernels), and the
lattice window halves at D >= 5, so each D is its own code.  Every device result is compared bit for bit with the CPU oracle:
bindings in commit order, ask states, final availability.  Weights are drawn from a non-dyadic set so that share * w is
inexact and a contracted (fused multiply-add) score would change keys; the CPU-side checks below show that the chosen inputs
have that power."""
import copy
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import py_oracle
from yunikorn_k8shim_b200 import Engine, YkError, synth

DIMS = (1, 2, 3, 4, 5, 6, 7, 8)
W_SET = (0.3, 3.0, 0.0, 1.3, 0.7, 0.1, 7.0, 1e-3)
YK_ERR_RANGE = -5
ST_PENDING = 0


def _weights(D, rot=0):
    w = [W_SET[(k + rot) % len(W_SET)] for k in range(D)]
    if not any(w):
        w[0] = 0.3
    return np.array(w, dtype=np.float64)


def _generic(s, D, seed=0):
    """synth.redim to D dimensions, with non-default weights.  redim fills a new dimension of the nodes' totals, of their
    availability and of the requests from independently chosen columns; here each new dimension becomes a resource of its
    own instead (a few thousand units per node, a per-application request), so that every dimension can bind."""
    t = synth.redim(s, D, seed)
    rng = np.random.default_rng(seed + 101)
    N, P = t.n_nodes, t.n_apps
    valid = s.ask_req.any(axis=1)                       # asks that request nothing stay invalid
    for k in range(s.D, D):
        tot = rng.integers(4, 33, N) * 1000
        t.node_total[:, k] = tot
        t.node_avail[:, k] = tot - (rng.random(N) < 0.3) * rng.integers(0, 4, N) * 1000
        per_app = rng.integers(0, 4, P) * 250 * (rng.random(P) < 0.7)
        t.ask_req[:, k] = per_app[t.ask_app] * valid   # per application: gang members and runs keep one request vector
    t.weights = _weights(D, seed % 3)
    t.name = f"{t.name}-w"
    return t


def _run(s, want, commit, **kw):
    with Engine.for_snapshot(s, commit=commit, **kw) as e:
        ask, node, _ = e.cycle(s.n_asks)
        states = e.ask_states(np.arange(s.n_asks))
        avail = e.nodes_available(np.arange(s.n_nodes))
        st = e.stats()
    tag = (s.name, commit, kw)
    assert np.array_equal(ask, want["ask"]), ("ask order differs", tag)
    assert np.array_equal(node, want["node"]), ("node choice differs", tag)
    assert np.array_equal(states, want["state"]), ("ask states differ", tag)
    assert np.array_equal(avail, want["avail"]), ("availability differs", tag)
    return st


# ---- A. the node score: device against two independent float64 restatements ---------------------------------------------

# weight vectors for the three quotient paths of yk_node_score: tw == 1, tw == 2 and the general divide, with zero weights
# between weighted dimensions
SCORE_WEIGHTS = ((1.0,), (0.25, 0.0, 0.75), (0.5, 0.5), (1.0, 1.0), (0.5, 0.0, 1.5), (0.3,), (0.3, 3.0), (0.3, 3.0, 0.0, 1.3),
                 (0.7, 0.0, 0.1, 7.0, 1e-3), (1.3, 0.3, 0.7, 3.0, 0.1, 7.0, 1e-3, 0.3), (0.1, 0.1, 0.1))


def _score_inputs(D, n, seed):
    """n nodes of D dimensions: ordinary values, totals and availabilities up to 2^62 (int64 -> double rounds), available
    above total, negative available, and zero totals with available above, below and at 0 (the infinite and the skipped
    NaN shares).  Two infinite shares of opposite sign would make the score NaN: such rows are excluded."""
    rng = np.random.default_rng(seed)
    tot = np.zeros((n, D), dtype=np.int64)
    av = np.zeros((n, D), dtype=np.int64)
    kind = rng.integers(0, 8, (n, D))
    for i in range(n):
        for k in range(D):
            c = kind[i, k]
            if c <= 2:                                  # ordinary
                t = int(rng.integers(1, 1 << 40))
                a = int(rng.integers(0, t + 1))
            elif c == 3:                                # near 2^62: the conversions round
                t = (1 << 62) - int(rng.integers(0, 1 << 40))
                a = int(rng.integers(1 << 52, t))
            elif c == 4:                                # available above total
                t = int(rng.integers(1, 1 << 30))
                a = t + int(rng.integers(1, 1 << 31))
            elif c == 5:                                # over-committed
                t = int(rng.integers(1, 1 << 50))
                a = -int(rng.integers(1, 1 << 50))
            else:                                       # zero total, available above / below / at zero
                t = 0
                a = int(rng.choice([0, 0, 7, -7, 1 << 61, -(1 << 61)]))
            tot[i, k], av[i, k] = t, a
    return tot, av


def _score_cases(D, policy):
    out = []
    for wi, w in enumerate(SCORE_WEIGHTS):
        w = list(w[:D]) + [0.0] * (D - len(w))
        if not any(w):
            continue
        tot, av = _score_inputs(D, 300, seed=D * 100 + wi * 7 + policy)
        keep = [i for i in range(len(tot)) if not math.isnan(py_oracle.node_score(policy, w, tot[i], av[i]))]
        out.append((np.array(w), tot[keep], av[keep]))
    return out


def _fused_score(policy, w, total, avail):
    """py_oracle.node_score with `usage += share * w` computed as one fused multiply-add (exact product and sum, one
    rounding): what a build that contracts the score would produce"""
    usage, tw = 0.0, 0.0
    for k in range(len(w)):
        if w[k] == 0.0:
            continue
        t, v = float(total[k]), float(avail[k])
        if t == 0.0:
            if v == 0.0:
                continue
            share = 1.0 - math.copysign(math.inf, v)
        else:
            share = 1.0 - v / t
        if math.isnan(share):
            continue
        if math.isinf(share) or math.isinf(usage):
            usage += share * w[k]
        else:
            usage = float(Fraction(share) * Fraction(w[k]) + Fraction(usage))
        tw += w[k]
    a = 0.0 if tw == 0.0 else usage / tw
    return ((1.0 - a) if policy == 1 else a) + 0.0


def test_score_inputs_have_teeth():
    """a device score that fused the multiply-add would differ from the unfused one on several hundred of the inputs the
    GPU test below checks, and the inputs reach every special case"""
    differ = 0
    special = {"inf": 0, "nan_share": 0, "big": 0, "above": 0, "negative": 0}
    for D in DIMS:
        for policy in (synth.POLICY_FAIR, synth.POLICY_BINPACKING):
            for w, tot, av in _score_cases(D, policy):
                for i in range(len(tot)):
                    plain = py_oracle.node_score(policy, w, tot[i], av[i])
                    differ += plain != _fused_score(policy, w, tot[i], av[i])
                    for k in range(D):
                        if w[k] == 0.0:
                            continue
                        special["inf"] += tot[i, k] == 0 and av[i, k] != 0
                        special["nan_share"] += tot[i, k] == 0 and av[i, k] == 0
                        special["big"] += tot[i, k] > 1 << 53
                        special["above"] += av[i, k] > tot[i, k] > 0
                        special["negative"] += av[i, k] < 0 < tot[i, k]
    assert differ >= 500, differ
    assert min(special.values()) > 50, special


@pytest.mark.gpu
@pytest.mark.parametrize("policy", [synth.POLICY_FAIR, synth.POLICY_BINPACKING])
@pytest.mark.parametrize("D", DIMS)
def test_device_node_score_bit_exact(oracle, D, policy):
    for w, tot, av in _score_cases(D, policy):
        n = len(tot)
        with Engine(D=D, policy=policy, weights=w, max_nodes=n, max_asks=1, max_apps=1, max_queues=2) as e:
            e.nodes_upsert(np.arange(n), tot, av, name_rank=np.arange(n))
            got = e.node_scores(np.arange(n))
        for i in range(n):
            py = py_oracle.node_score(policy, w, tot[i], av[i])
            cc = oracle.node_score(policy, w, tot[i], av[i])
            assert py.hex() == cc.hex(), (D, w, tot[i], av[i])
            assert float(got[i]).hex() == py.hex(), (D, policy, w.tolist(), tot[i].tolist(), av[i].tolist())


# ---- B. whole cycles at every D --------------------------------------------------------------------------------------------

DEEP_MID, DEEP_END = 60, 61         # label bits (unused by synth.perf) carried only by nodes deep in the initial order


def _deep_perf(D, seed):
    """config-3 shape (1 500 nodes, masks) where every 8th ask can only go to a node beyond 300 positions into the initial
    order (past the lattice window at D >= 5) and every 16th only to one of the last 150 (past it at every D)"""
    s = _generic(synth.perf(1500, 20, 50, masks=True, seed=seed), D, seed)
    rank = s.node_rank()
    score = np.array([py_oracle.node_score(s.policy, s.weights, s.node_total[n], s.node_avail[n]) for n in range(s.n_nodes)])
    pos = np.empty(s.n_nodes, dtype=np.int64)
    pos[np.lexsort((rank, score))] = np.arange(s.n_nodes)
    one = np.uint64(1)
    s.node_label |= np.where((pos >= 300) & (pos < 480), one << np.uint64(DEEP_MID), np.uint64(0)).astype(np.uint64)
    s.node_label |= np.where(pos >= s.n_nodes - 150, one << np.uint64(DEEP_END), np.uint64(0)).astype(np.uint64)
    for a, bit in ((np.arange(0, s.n_asks, 8), DEEP_MID), (np.arange(4, s.n_asks, 16), DEEP_END)):
        s.ask_tol[a] = np.uint64(0xFFFF)
        s.ask_need[a] = one << np.uint64(bit)
        s.ask_deny[a] = np.uint64(0)
    return s


def _big_first_gang(D):
    """synth.gangs, but asks 100..139 form one gang whose members each need nearly all of a 40-CPU node: its first member
    fits, yet the cluster has fewer such nodes than members, so the gang is rolled back.  The twenty gangs before it are
    placed on the device first."""
    s = _generic(synth.gangs(300, 60, 5, seed=D, fill=1.3), D, D)
    big = np.arange(100, 140)
    s.ask_app[big] = s.ask_app[100]
    s.ask_gang[big] = s.ask_gang[100]
    s.ask_req[big] = s.ask_req[100]
    s.ask_req[big, 0] = 39_500
    return s


def _cycle_snapshots(D):
    """(snapshot, batch, role): fair-policy shapes for the device commit's stats, plus fuzz seeds (either policy)"""
    out = [(_deep_perf(D, 2), 512, "deep"),
           (_generic(synth.hier(400, 3, 3, 2, 40, priorities=True, seed=D), D, D), 128, "hier"),
           (_generic(synth.gangs(300, 60, 5, seed=D, fill=1.3), D, D), 64, "gangs"),
           (_big_first_gang(D), 64, "gangs")]
    for seed in range(6):
        s = _generic(synth.fuzz(seed + 10 * D), D, seed)
        for batch in (7, 64, 1024):
            if (s.ask_gang >= 0).any() and np.bincount(s.ask_gang[s.ask_gang >= 0]).max() > batch:
                continue
            out.append((s, batch, "fuzz"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_cycles_at_every_dimension_count(oracle, D):
    """both commits on every snapshot; per D the device commit must have taken a whole cycle, run a full-order scan and
    handed a gang roll-back over to the host commit, and the host commit must have swept"""
    whole = fullscan = handoff = 0
    wants = {}
    for s, batch, role in _cycle_snapshots(D):
        want = wants.setdefault(id(s), oracle.run(s))
        host = _run(s, want, "host", batch=batch)
        assert host["sweep_launches"] > 0 and host["lattice_launches"] == 0, (s.name, batch)
        dev = _run(s, want, "device", batch=batch)
        if role == "fuzz":
            continue
        assert dev["lattice_asks"] > 0, (s.name, dev)     # fair policy, weights >= 0: the device commit must run
        whole += dev["lattice_asks"] == s.n_asks and dev["sweep_launches"] == 0
        fullscan += dev["lattice_fullscans"] > 0
        handoff += dev["lattice_handoffs"] > 0
    assert whole and fullscan and handoff, (D, whole, fullscan, handoff)


# ---- C. uniform runs at every D ----------------------------------------------------------------------------------------------

def _crowded_reference(D, n_nodes=200, apps=20, tasks=125):
    """the reference benchmark's shape with nine nodes in ten nearly full: the empty ones take far more than the mean share
    of each run, so the first cut depth is too shallow and the run is retried deeper"""
    s = _generic(synth.reference_shape(n_nodes, apps, tasks), D, D)
    busy = np.arange(n_nodes) % 10 != 0
    s.node_avail[busy, 0] = s.node_total[busy, 0] // 10
    if D > 1:
        s.node_avail[busy, 1] = s.node_total[busy, 1] // 10
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_uniform_runs_at_every_dimension_count(oracle, monkeypatch, D):
    monkeypatch.setenv("YK_UNIFORM_MIN", "6")
    retries = 0
    for s, batch in ((synth.runny(_generic(synth.perf(1500, 20, 100), D, D), D), 4096),
                     (synth.runny(_generic(synth.perf(600, 10, 60, masks=True), D, D + 1), D), 1024),
                     (_crowded_reference(D), 4096)):
        want = oracle.run(s)
        dev = _run(s, want, "device", batch=batch)
        assert dev["uniform_asks"] > 0, (s.name, dev)
        retries += dev["uniform_retries"]
        _run(s, want, "host", batch=batch)
    assert retries > 0, D


@pytest.mark.gpu
def test_two_uniform_cycles_then_release_at_d8(oracle, monkeypatch):
    monkeypatch.setenv("YK_UNIFORM_MIN", "6")
    s = _crowded_reference(8)
    full = oracle.run(s)
    k = len(full["ask"]) // 3
    with Engine.for_snapshot(s, batch=4096, commit="device") as e:
        ask, node, _ = e.cycle(k)
        ask2, node2, _ = e.cycle(s.n_asks)
        st = e.stats()
        assert np.array_equal(np.concatenate([ask, ask2]), full["ask"])
        assert np.array_equal(np.concatenate([node, node2]), full["node"])
        assert np.array_equal(e.ask_states(np.arange(s.n_asks)), full["state"])
        assert np.array_equal(e.nodes_available(np.arange(s.n_nodes)), full["avail"])
        assert st["lattice_cycles"] == 2 and st["uniform_asks"] > 0 and st["sweep_launches"] == 0, st
        e.release(np.concatenate([ask, ask2]))
        assert np.array_equal(e.nodes_available(np.arange(s.n_nodes)), s.node_avail)


# ---- D. the sweep's first fit at chosen sorted positions -------------------------------------------------------------------

SWEEP_N = (1, 31, 32, 33, 511, 512, 513, 1023, 1024, 1025, 1537)
SWEEP_ROWS = (1, 31, 32, 33, 127, 128, 129, 257)
SWEEP_TARGETS = (0, 31, 32, 255, 256, 511, 512, 513)
BIG = 1 << 20


def _positional(D, N, rows, kind, seed=0):
    """N nodes identical on the weighted dimensions (every key ties, so the sorted order is NodeID rank), named by a shuffled
    permutation.  The node at sorted position p holds (p+1, BIG-p-1) on the last two dimensions, which are unweighted, and an
    ask aimed at p requests exactly that: only that node fits, and taking it moves no key.  Asks cycle through the targets
    (plus N-1 and one at or beyond N: NOFIT).  kind: "plain" (no masks), "masks" (taints / selectors every node passes, a
    distinct toleration set per ask), "name" (pod.Spec.NodeName = the target node).  -> snapshot, expected bindings"""
    rng = np.random.default_rng(seed + N)
    perm = rng.permutation(N)                              # node i has NodeID rank perm[i]
    at = np.argsort(perm)                                  # node index at sorted position p
    targets = sorted({t for t in SWEEP_TARGETS if t < N} | {N - 1}) + [N + 3]
    tot = np.zeros((N, D), dtype=np.int64)
    tot[:, 0] = 32_000
    if D > 1:
        tot[:, 1] = 256 * synth.GI
    for k in range(2, D - 2):
        tot[:, k] = 1 << 30
    tot[:, D - 2] = perm + 1
    tot[:, D - 1] = BIG - perm - 1
    ids = [f"node-{p:05d}" for p in perm]
    tgt = np.array([targets[(i + rows) % len(targets)] for i in range(rows)], dtype=np.int64)
    req = np.zeros((rows, D), dtype=np.int64)
    req[:, 2:D - 2] = 1
    req[:, D - 2] = tgt + 1
    req[:, D - 1] = BIG - tgt - 1
    z = np.zeros(rows, dtype=np.uint64)
    tol, need, deny = z.copy(), z.copy(), z.copy()
    taint = np.zeros(N, dtype=np.uint64)
    label = np.zeros(N, dtype=np.uint64)
    ask_node = None
    if kind == "masks":
        taint[:] = np.uint64(1 << 5)
        label[:] = np.uint64(1 << 3)
        tol = (np.uint64(1 << 5) | (np.arange(rows, dtype=np.uint64) << np.uint64(8))).astype(np.uint64)
        need[:] = np.uint64(1 << 3)
        deny[:] = np.uint64(1 << 9)
    elif kind == "name":
        ask_node = np.where(tgt < N, at[np.minimum(tgt, N - 1)], at[0]).astype(np.int32)
    s = synth._finish(f"positional-{kind}-N{N}-r{rows}-D{D}", D, synth.POLICY_FAIR, tot, tot.copy(), taint, label, ids,
                      synth._single_queue(D), np.ones(1, dtype=np.int32), np.zeros(rows, dtype=np.int32), req, tol, need,
                      deny, ask_node=ask_node)
    s.weights = np.zeros(D)
    s.weights[:min(D, 2)] = (0.3, 3.0)[:min(D, 2)]
    expect, taken = [], set()
    for i, p in enumerate(tgt.tolist()):
        if p < N and p not in taken:
            taken.add(p)
            expect.append((i, int(at[p])))
    return s, expect


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["plain", "masks", "name"])
@pytest.mark.parametrize("D", [4, 8])
def test_sweep_first_fit_at_exact_positions(oracle, monkeypatch, D, kind):
    """each ask has exactly one feasible node, at a chosen sorted position: across 32-bit words, warps, the 512-position
    node tile, 128-ask sub-chunks, 32-row groups and the padding past the last node"""
    for N in SWEEP_N:
        for rows in SWEEP_ROWS:
            s, expect = _positional(D, N, rows, kind)
            want = oracle.run(s)
            assert list(zip(want["ask"].tolist(), want["node"].tolist())) == expect, s.name
            for share in (True, False):
                for epoch_rows in (True, False):
                    if epoch_rows:
                        monkeypatch.delenv("YK_NO_EPOCH_ROWS", raising=False)
                    else:
                        monkeypatch.setenv("YK_NO_EPOCH_ROWS", "1")
                    st = _run(s, want, "host", batch=rows, share_rows=share)
                    assert st["sweep_launches"] > 0
            monkeypatch.delenv("YK_NO_EPOCH_ROWS", raising=False)
            dev = _run(s, want, "device", batch=rows)
            assert dev["lattice_asks"] > 0


# ---- E. preemption search and predicates at every D ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_preemption_and_predicates_at_every_dimension_count(oracle, D):
    s = _generic(synth.perf(64, 4, 40, masks=True, seed=31), D, D)
    s.node_avail[:, 0] //= 50                                # nearly full nodes: victims are needed
    for k in {min(1, D - 1), D - 1}:                         # over-committed on some dimension: the clamp matters
        s.node_avail[::5, k] = -(s.node_total[::5, k] // 7) - 1
    s.node_avail[::3, 0] = 0
    s.node_flags[7] = 0
    s.ask_node[5] = 3
    rng = np.random.default_rng(D)
    Q = 400
    asks = rng.integers(0, s.n_asks, Q)
    nodes = rng.integers(0, s.n_nodes, Q)
    scale = np.maximum(s.ask_req.max(axis=0) // 6, 1)
    victims, starts = [], []
    for q in range(Q):
        nv = int(rng.integers(0, 101))                       # crosses the 32- and 64-victim warp steps
        v = (rng.random((nv, D)) * scale).astype(np.int64)
        victims.append(v)
        starts.append(int(rng.integers(0, nv + 4)))          # also beyond the victim count
    want = [oracle.preemption_index(s, int(a), int(n), v, st) for a, n, v, st in zip(asks, nodes, victims, starts)]
    assert any(w >= 32 for w in want) and any(w < 0 for w in want) and any(0 <= w < 32 for w in want), want
    with Engine.for_snapshot(s) as e:
        got = e.preemption_search(asks, nodes, victims, starts)
        assert got.tolist() == want
        for a in range(0, s.n_asks, 3):
            for n in range(0, s.n_nodes, 5):
                g, x = e.evaluate(a, n), oracle.predicate(s, a, n)
                assert (g == 0) == (x == 0) and (g == x or {g, x} <= {4, 8}), (a, n, g, x)
                assert e.evaluate_reserve(a, n) == oracle.predicate_reserve(s, a, n), (a, n)


# ---- F. a NaN node score is an error that leaves the engine usable ---------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("commit", ["host", "device"])
def test_nan_node_score_is_an_error_and_the_engine_recovers(oracle, commit):
    """a node whose score is NaN makes the cycle fail with YK_ERR_RANGE on both commits, nothing is bound, and once the node
    is repaired the next cycle equals the oracle's.  Found a bug: the device commit reported the NaN only after its first
    batch had run on the sorted order, and the end of the cycle still exported the node records that batch had changed, so
    the engine kept allocations it never returned (every node's availability dropped while all asks stayed pending)."""
    s = _generic(synth.perf(40, 4, 30, seed=7), 4, 0)
    bad = copy.deepcopy(s)
    bad.node_total[3, :2] = 0
    bad.node_avail[3, :2] = (1, -1)                          # shares -Inf and +Inf on two weighted dimensions: NaN
    assert math.isnan(py_oracle.node_score(bad.policy, bad.weights, bad.node_total[3], bad.node_avail[3]))
    with pytest.raises(RuntimeError):
        oracle.run(bad)
    want = oracle.run(s)
    rank = s.node_rank()
    with Engine.for_snapshot(bad, batch=64, commit=commit) as e:
        with pytest.raises(YkError) as ei:
            e.cycle(s.n_asks)
        assert ei.value.code == YK_ERR_RANGE
        assert set(e.ask_states(np.arange(s.n_asks)).tolist()) == {ST_PENDING}
        assert np.array_equal(e.nodes_available(np.arange(s.n_nodes)), bad.node_avail)
        e.nodes_upsert([3], s.node_total[3:4], s.node_avail[3:4], s.node_taint[3:4], s.node_label[3:4], rank[3:4], s.node_flags[3:4])
        ask, node, _ = e.cycle(s.n_asks)
        assert np.array_equal(ask, want["ask"]) and np.array_equal(node, want["node"])
        assert np.array_equal(e.ask_states(np.arange(s.n_asks)), want["state"])
        assert np.array_equal(e.nodes_available(np.arange(s.n_nodes)), want["avail"])
        if commit == "device":
            assert e.stats()["lattice_asks"] > 0
