"""The three pass kernels (speculative, sequencer, lock-step) at the shapes and edges the ABI accepts, each run
compared bit for bit with the array-form oracle (oracle/fast.c), and each case PROVING which kernel it reached:

- engine 0 (auto) picks a kernel per state pass (k_pick_mode); BLANCE_NO_SEQ / BLANCE_NO_SPEC, read on every plan
  call, take the sequencer / speculative kernel out of that choice;
- engine 2 asks for the sequencer, engine 1 for the lock-step kernel;
- sticky_steps is raised only by the sequencer and the speculative kernel (0 means lock-step everywhere);
- BLANCE_SPEC_STATS=1 prints the speculative counters of instances 0-3 on stderr; every speculative pass starts
  with one list rebuild, so rebuilds > 0 means the speculative kernel ran for that instance.

Also the move-list entry points at large node-id spaces and partial state visits.  Needs a B200; run with -m gpu."""
import copy
import ctypes
import os
import re

import numpy as np
import pytest

from oracle_loader import fast_lib_path, literal

from blance_b200 import _host, tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAST = ctypes.CDLL(fast_lib_path())
FAST.oracle_fast_plan_next_map.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
FAST.oracle_fast_calc_partition_moves.argtypes = [ctypes.c_int32] * 3 + [ctypes.c_void_p] * 3 + [ctypes.c_int32] * 2 + [ctypes.c_void_p] * 4
FAST.oracle_fast_moves_available.argtypes = [ctypes.c_int32] * 2 + [ctypes.c_void_p] * 7

STATS = re.compile(r"\[blance\] inst (\d+): steps (\d+) accepted (\d+) \| resolved by the leader (\d+) \(stale results (\d+)\) "
                   r"movers (\d+) team (\d+) rebuilds (\d+) waits (\d+)")
FIELDS = ("steps", "accepted", "resolved", "stale", "movers", "team", "rebuilds", "waits")
# name -> (engine, environment switch)
ENGINES = {"auto": (0, None), "auto_no_seq": (0, "BLANCE_NO_SEQ"), "auto_no_spec": (0, "BLANCE_NO_SPEC"),
           "sequencer": (2, None), "lockstep": (1, None)}
DEFAULT_ENGINES = ("auto", "auto_no_seq", "sequencer", "lockstep")


def spec_define(name):
    src = open(os.path.join(ROOT, "blance_b200", "csrc", "assign_pass_spec.cuh")).read()
    return int(re.search(r"#define %s (\d+)" % name, src).group(1))


@pytest.fixture(scope="module")
def ctx():
    c = tables.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def oracle_tables(t):
    r = tables.PlanResult(t)
    s = t.struct()
    assert FAST.oracle_fast_plan_next_map(ctypes.byref(s), ctypes.byref(r.out)) == 0
    return r


def same(got, ref):
    return (np.array_equal(got.next_rows, ref.next_rows) and np.array_equal(got.next_shape, ref.next_shape) and
            np.array_equal(got.warn, ref.warn) and
            (got.iters_run, got.converged, got.steps) == (ref.iters_run, ref.converged, ref.steps))


def parse_stats(err):
    return {int(m.group(1)): dict(zip(FIELDS, map(int, m.groups()[1:]))) for m in STATS.finditer(err)}


def set_engine_env(monkeypatch, name):
    monkeypatch.setenv("BLANCE_SPEC_STATS", "1")
    for var in ("BLANCE_NO_SEQ", "BLANCE_NO_SPEC"):
        monkeypatch.delenv(var, raising=False)
    if ENGINES[name][1]:
        monkeypatch.setenv(ENGINES[name][1], "1")


def run_engines(ctx, ts, monkeypatch, capfd, engines=DEFAULT_ENGINES):
    """Runs the batch `ts` (one instance: the single-plan entry point) under every engine; every instance must equal
    the oracle.  Returns the oracle results and, per engine, (results, speculative counters of instances 0-3)."""
    refs = [oracle_tables(t) for t in ts]
    runs, bad = {}, []
    for name in engines:
        set_engine_env(monkeypatch, name)
        for t in ts:
            t.engine = ENGINES[name][0]
        capfd.readouterr()
        got = ctx.plan_next_map_batch(ts) if len(ts) > 1 else [ctx.plan_next_map(ts[0])]
        stats = parse_stats(capfd.readouterr().err)
        assert len(stats) == min(4, len(ts)), name
        bad += [(name, i, list(ts[i].state_constraints), ts[i].n_nodes) for i, (g, r) in enumerate(zip(got, refs)) if not same(g, r)]
        runs[name] = (got, stats)
    assert not bad, "differs from the oracle (engine, instance, k, N): %s" % bad
    return refs, runs


def ran_spec(runs, i, name="auto"):
    return runs[name][1][i]["rebuilds"] > 0


def ran_sequencer(runs, i):
    got, stats = runs["sequencer"]
    return got[i].sticky_steps > 0 and stats[i]["rebuilds"] == 0


def ran_lockstep_only(runs, i, name="lockstep"):
    got, stats = runs[name]
    return got[i].sticky_steps == 0 and (i not in stats or stats[i]["rebuilds"] == 0)


# ---- generators ------------------------------------------------------------------------------------------------

def flat_tables(seed, ks, P, N, prio=None, node_w=True, booster=None, part_w=True, partial=0.05, churn=True,
                max_iters=None, NU=None):
    """A rebalance of a full previous map: every row holds distinct nodes of nodesAll, a `partial` share of the
    state lists is short, some nodes are removed / added, node weights may be <= 0, partition weights and
    stickiness are optional."""
    rng = np.random.default_rng(seed)
    S = len(ks)
    t = tables.PlanTables(N, S, P, list(range(S)) if prio is None else prio, ks, n_node_ids=NU or N)
    SL = t.n_slots
    rows = rng.random((P, N)).argsort(axis=1)[:, :SL].astype(np.int32)
    for s in range(S):
        lo, hi = int(t.state_slot_off[s]), int(t.state_slot_off[s + 1])
        short = rng.random(P) < partial
        cnt = np.where(short, rng.integers(0, hi - lo + 1, P), hi - lo)
        rows[:, lo:hi][np.arange(hi - lo)[None, :] >= cnt[:, None]] = -1
    t.prev_rows[:] = rows
    t.cur_rows[:] = rows
    t.prev_shape[:] = 2
    t.cur_shape[:] = 2
    t.part_in_prev[:] = 1
    if churn:
        t.node_removed[rng.permutation(N)[:int(rng.integers(1, max(2, N // 10)))]] = 1
        t.node_added[rng.permutation(N)[:int(rng.integers(0, N // 4 + 1))]] = 1
    if node_w:
        t.has_node_weights = 1
        t.node_has_weight[:] = (rng.random(N) < 0.8).astype(np.uint8)
        t.node_weight[:] = rng.integers(-3, 7, N)
        t.booster_kind = int(rng.random() < 0.5) if booster is None else booster
    if part_w:
        t.has_part_weights = 1
        t.part_has_weight[:] = (rng.random(P) < 0.5).astype(np.uint8)
        t.part_weight[:] = rng.integers(1, 9, P)
        t.state_has_stickiness[:] = (rng.random(S) < 0.7).astype(np.uint8)
        t.state_stickiness[:] = rng.integers(0, 5, S)
    t.max_iters = int(rng.integers(2, 6)) if max_iters is None else max_iters
    return t


def narrow_batch(seed, n):
    """n mixed instances (K 1-4, N 24..768): instance 0 at N = 768 and instance 3 at N = 769, one past the
    speculative kernel's node limit in the narrow configuration."""
    rng = np.random.default_rng(seed)
    ts = []
    for i in range(n):
        ks = [[1], [2], [3], [4], [1, 2], [2, 2], [1, 3]][int(rng.integers(0, 7))]
        N = {0: 768, 3: 769}.get(i, int(rng.integers(24, 769)))
        P = int(rng.integers(200, 400)) if i < 4 else int(rng.integers(64, 200))
        ts.append(flat_tables(seed * 1000 + i, ks, P, N, booster=i % 2, max_iters=int(rng.integers(1, 4))))
    return ts


# ---- 1. k = 4 and 8-slot rows -------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(2))
def test_k4_and_eight_slot_rows(ctx, monkeypatch, capfd, seed):
    rng = np.random.default_rng(100 + seed)
    models = [[4], [4, 4], [1, 3, 4], [2, 2, 4]]
    ts = [flat_tables(100 + 10 * seed + i, ks, int(rng.integers(500, 5001)), int(rng.integers(16, 401)))
          for i, ks in enumerate(models)]
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in range(4):
        assert ran_spec(runs, i) and ran_spec(runs, i, "auto_no_seq"), i
        assert ran_sequencer(runs, i), i
        assert ran_lockstep_only(runs, i), i
    assert ts[1].n_slots == 8 and ts[3].n_slots == 8


# ---- 2. equal state priorities -----------------------------------------------------------------------------------

def test_equal_state_priorities(ctx, monkeypatch, capfd):
    # instance 0: the first state has k = 5, which no fast kernel takes, so the speculative rebuilds come from the
    # later states of equal priority (the top state is the first one in state order)
    ts = [flat_tables(200, [5, 2, 1], 1500, 64, prio=[0, 0, 0]),
          flat_tables(201, [2, 2], 1200, 48, prio=[3, 3]),
          flat_tables(202, [1, 2, 1], 900, 40, prio=[1, 1, 0])]
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in range(3):
        assert ran_spec(runs, i) and ran_sequencer(runs, i) and ran_lockstep_only(runs, i), i


# ---- 3 / 4. the narrow configuration, and its ring generations wrapping ---------------------------------------------

def test_narrow_configuration_batch(ctx, monkeypatch, capfd, sm_count):
    ts = narrow_batch(300, sm_count // 2 + 1)
    assert 2 * len(ts) > sm_count
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in (0, 1, 2):
        assert ran_spec(runs, i) and ran_spec(runs, i, "auto_no_seq"), i
    assert not ran_spec(runs, 3) and not ran_spec(runs, 3, "auto_no_seq")      # N = 769
    for i in range(4):
        assert ran_lockstep_only(runs, i), i


def test_narrow_ring_generation_wrap(ctx, monkeypatch, capfd, sm_count):
    # the narrow configuration has 3 scout warps of SP_D ring chunks of 32 steps; the generation tag cycles after
    # SP_GEN_MOD rounds of them, so one pass longer than that reuses every ring slot with a wrapped tag
    wrap = spec_define("SP_GEN_MOD") * spec_define("SP_D") * 3 * 32
    P, N = wrap + 3600, 96
    rng = np.random.default_rng(400)
    big = tables.PlanTables(N, 1, P, [0], [2])
    a = rng.integers(0, N, P)
    rows = np.stack([a, (a + rng.integers(1, N, P)) % N], axis=1).astype(np.int32)
    big.prev_rows[:] = rows
    big.cur_rows[:] = rows
    big.prev_shape[:] = 2
    big.cur_shape[:] = 2
    big.part_in_prev[:] = 1
    big.node_removed[[5, 17]] = 1
    big.node_added[[90, 91]] = 1
    big.has_node_weights = 1
    big.node_has_weight[:] = 1
    big.node_weight[:] = rng.integers(-2, 5, N)
    big.booster_kind = 1
    big.max_iters = 1
    ts = [big] + narrow_batch(401, sm_count // 2 + 1)[1:]
    assert 2 * len(ts) > sm_count and big.n_parts > wrap
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd, engines=("auto", "sequencer"))
    assert ran_spec(runs, 0) and runs["auto"][1][0]["steps"] == P
    assert ran_sequencer(runs, 0)


# ---- 5. the node-count limits of the kernel choice ---------------------------------------------------------------------

@pytest.mark.parametrize("N", [2048, 2049, 4096, 4097])
def test_single_plan_selection_limits(ctx, monkeypatch, capfd, N):
    t = flat_tables(500 + N, [2], 640, N, booster=1, max_iters=2)
    assert (t.node_weight[t.node_has_weight > 0] < 0).any()
    refs, runs = run_engines(ctx, [t], monkeypatch, capfd)
    assert ran_spec(runs, 0) == (N <= 2048)
    assert ran_sequencer(runs, 0) == (N <= 4096)
    if N == 2049:
        assert ran_sequencer(runs, 0) and runs["auto"][0][0].sticky_steps > 0      # auto falls back to the sequencer
    if N == 4097:
        assert ran_lockstep_only(runs, 0, "sequencer") and ran_lockstep_only(runs, 0, "auto")
    assert ran_lockstep_only(runs, 0)


# ---- 6. prevMap counts under state names outside the model ----------------------------------------------------------------

@pytest.mark.parametrize("seed", range(3))
def test_prev_counts_outside_the_model(ctx, monkeypatch, capfd, seed):
    rng = np.random.default_rng(600 + seed)
    ts = []
    for i, (ks, N) in enumerate((([2], 40), ([1, 2], 64), ([3], 30), ([4], 120))):
        t = flat_tables(600 + 10 * seed + i, ks, int(rng.integers(600, 2000)), N, max_iters=int(rng.integers(3, 6)))
        t.extra_tot_first[:] = rng.integers(0, 80, N)
        t.extra_tot_rest[:] = (t.extra_tot_first * rng.random(N)).astype(np.int32)
        t.part_in_prev[rng.random(t.n_parts) < 0.01] = 3
        t.part_in_prev[0] = 3
        ts.append(t)
    assert all((t.extra_tot_first != t.extra_tot_rest).any() for t in ts)
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in range(4):
        assert refs[i].iters_run >= 2
        assert ran_spec(runs, i) and ran_sequencer(runs, i), i


# ---- 7. the string API at mid size -------------------------------------------------------------------------------------

def midsize_instance(seed):
    """A randgen-like instance large enough for the fast kernels: full clean lists (a few short), nodes removed and
    added, weights and stickiness, and "dead" state lists in prevMap - on entries being assigned (the first
    iteration then cannot converge) and on entries that are not."""
    rnd = np.random.default_rng(seed)
    N = int(rnd.integers(20, 201))
    nodes = ["n%03d" % i for i in range(N)]
    states = ["primary", "replica", "standby"][:int(rnd.integers(1, 4))]
    ks = [int(rnd.integers(1, 3)) for _ in states]
    model = {s: (i, k) for i, (s, k) in enumerate(zip(states, ks))}
    P = int(rnd.integers(200, 2001))
    names = [str(i) for i in range(P)]
    prev, assign = {}, {}
    for p, n in enumerate(names):
        perm = rnd.permutation(N)
        row, o = {}, 0
        for s, k in zip(states, ks):
            c = k if rnd.random() > 0.03 else int(rnd.integers(0, k + 1))
            row[s] = [nodes[x] for x in perm[o:o + c]]
            o += k
        prev[n] = row
        if p % 7:
            assign[n] = copy.deepcopy(row)
            if rnd.random() < 0.02:
                prev[n]["dead"] = [nodes[int(rnd.integers(0, N))]]
        elif rnd.random() < 0.5:
            prev[n]["dead"] = [nodes[int(x)] for x in rnd.permutation(N)[:2]]
    kw = dict(prev_map=prev, partitions_to_assign=assign, nodes_all=nodes,
              nodes_to_remove=[nodes[int(x)] for x in rnd.permutation(N)[:int(rnd.integers(0, N // 10 + 1))]],
              nodes_to_add=[nodes[int(x)] for x in rnd.permutation(N)[:int(rnd.integers(0, N // 5 + 1))]], model=model)
    if rnd.random() < 0.7:
        kw["node_weights"] = {n: int(rnd.choice([-3, -1, 0, 1, 2, 5])) for n in nodes if rnd.random() < 0.7}
        kw["booster"] = int(rnd.random() < 0.5)
    if rnd.random() < 0.7:
        kw["partition_weights"] = {n: int(rnd.integers(0, 9)) for n in names if rnd.random() < 0.5}
        kw["state_stickiness"] = {s: int(rnd.integers(0, 5)) for s in states if rnd.random() < 0.7}
    return kw


def test_string_api_midsize_vs_oracles(monkeypatch, capfd):
    L = literal()
    monkeypatch.setenv("BLANCE_SPEC_STATS", "1")
    for seed in range(20):
        kw = midsize_instance(700 + seed)
        ip = _host.intern_plan(**copy.deepcopy(kw))
        ref = _host.plan_out(ip)
        assert FAST.oracle_fast_plan_next_map(ip.in_ptr, ref.out_ptr) == 0
        got = _host.plan_out(ip)
        capfd.readouterr()
        _host.run_plan_cuda(ip, got)
        stats = parse_stats(capfd.readouterr().err)
        assert stats[0]["rebuilds"] > 0, seed
        assert np.array_equal(got.next_rows, ref.next_rows), seed
        assert np.array_equal(got.next_shape, ref.next_shape) and np.array_equal(got.warn, ref.warn), seed
        assert (got.iters_run, got.converged, got.steps) == (ref.iters_run, ref.converged, ref.steps), seed
        if seed % 10 == 0:
            lit = L.plan_next_map_ex(**copy.deepcopy(kw))
            nm, w = _host.unintern_plan(ip, got)
            assert nm == lit["next_map"] and w == lit["warnings"] and got.iters_run == lit["iterations"], seed


# ---- 8. partition weights of 0, negative and large -----------------------------------------------------------------------

@pytest.mark.parametrize("sticky", ["absent", "zero"])
def test_partition_weights_zero_negative_large(ctx, monkeypatch, capfd, sticky):
    rng = np.random.default_rng(800)
    ts = []
    for i, (ks, N) in enumerate((([1, 1], 24), ([2], 60))):
        t = flat_tables(800 + i, ks, 900, N, max_iters=4)
        w = rng.integers(-9, 10, t.n_parts)
        w[rng.random(t.n_parts) < 0.1] = 0
        w[3], w[7], w[11] = 999_999_999, -40_000_000, 25_000_000
        t.part_weight[:] = w
        t.part_has_weight[:] = 1
        t.part_has_weight[rng.random(t.n_parts) < 0.2] = 0
        t.part_has_weight[[3, 7, 11]] = 1
        assert int(np.abs(w[t.part_has_weight > 0]).astype(np.int64).sum() + (t.part_has_weight == 0).sum()) * t.n_slots < 2 ** 31
        t.state_has_stickiness[:] = 0 if sticky == "absent" else 1
        t.state_stickiness[:] = 0
        ts.append(t)
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in range(2):
        assert ran_spec(runs, i) and runs["auto"][1][i]["movers"] > 0, i
        assert ran_sequencer(runs, i) and ran_lockstep_only(runs, i), i


# ---- 9. exact score ties -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [32, 96])
def test_exact_score_ties(ctx, monkeypatch, capfd, N):
    """No weights, a balanced round-robin map over N - 2 nodes, two nodes removed and two empty ones added: every
    arg-min is decided by the position order.  N <= 64 gives the speculative kernel a complete list, N > 64 needs
    its upper-bound proof."""
    L_ = N - 2
    P = 12 * L_
    t = tables.PlanTables(N, 2, P, [0, 1], [1, 1])
    p = np.arange(P)
    rows = np.stack([p % L_, (p + 1 + (p // L_) % (L_ - 1)) % L_], axis=1).astype(np.int32)
    t.prev_rows[:] = rows
    t.cur_rows[:] = rows
    t.prev_shape[:] = 2
    t.cur_shape[:] = 2
    t.part_in_prev[:] = 1
    t.node_removed[[3, L_ // 2]] = 1
    t.node_added[[N - 2, N - 1]] = 1
    refs, runs = run_engines(ctx, [t], monkeypatch, capfd)
    st = runs["auto"][1][0]
    assert st["movers"] > 0 and st["rebuilds"] > 1
    assert ran_sequencer(runs, 0) and ran_lockstep_only(runs, 0)


# ---- 10. team paths inside a speculative pass --------------------------------------------------------------------------

def test_team_paths_in_a_speculative_pass(ctx, monkeypatch, capfd):
    ts = []
    for i, (ks, N) in enumerate((([1, 2], 50), ([2], 40), ([2, 1], 70))):
        t = flat_tables(1000 + i, ks, 1280, N, NU=N + 3, partial=0.02, max_iters=3)
        rng = np.random.default_rng(1000 + i)
        full = np.nonzero((t.cur_rows >= 0).all(axis=1))[0]
        bad = rng.permutation(full)[:t.n_parts // 64 - 1]                # at most 1/64 of the rows unclean
        for j, p in enumerate(bad):
            row = t.cur_rows[p]
            if j % 2 == 0:
                row[t.n_slots - 1] = N + j % 3                           # a node id outside nodesAll
            elif t.n_states > 1:
                row[t.state_slot_off[1]] = row[0]                        # one node listed under two states
            else:
                row[0] = N + 2
            t.prev_rows[p] = row
        ts.append(t)
    refs, runs = run_engines(ctx, ts, monkeypatch, capfd)
    for i in range(3):
        assert ran_spec(runs, i) and runs["auto"][1][i]["team"] > 0, i
        assert ran_lockstep_only(runs, i), i


# ---- 11. the lock-step kernel at the ABI limits ------------------------------------------------------------------------------

def limit_kwargs(kind, seed):
    rnd = np.random.default_rng(seed)
    if kind == "k16":
        states, ks, N = ["primary"], [16], 40
    elif kind == "eight_states_32_slots":
        states, ks, N = ["s%d" % i for i in range(8)], [4] * 8, 48
    elif kind == "picks32":
        states, ks, N = ["primary", "replica"], [2, 16], 64
    else:                                                                  # hier4096
        states, ks, N = ["primary", "replica"], [1, 2], 4000
    nodes = ["n%04d" % i for i in range(N)]
    model = {s: (i if i < 4 else 3, k) for i, (s, k) in enumerate(zip(states, ks))}   # states 3..7 share a priority
    P = 300 if kind != "hier4096" else 400
    names = [str(i) for i in range(P)]
    prev = {}
    for n in names:
        perm = rnd.permutation(N)
        row, o = {}, 0
        for s, k in zip(states, ks):
            c = k if rnd.random() > 0.1 else int(rnd.integers(0, k + 1))
            row[s] = [nodes[x] for x in perm[o:o + c]]
            o += k
        prev[n] = row
    kw = dict(prev_map=prev, partitions_to_assign=None, nodes_all=nodes,
              nodes_to_remove=[nodes[int(x)] for x in rnd.permutation(N)[:max(1, N // 20)]],
              nodes_to_add=[nodes[int(x)] for x in rnd.permutation(N)[:N // 8]], model=model,
              node_weights={n: int(rnd.choice([-2, 0, 1, 3])) for n in nodes if rnd.random() < 0.6}, booster=1,
              partition_weights={n: int(rnd.integers(0, 6)) for n in names if rnd.random() < 0.5},
              state_stickiness={states[0]: 2})
    if kind in ("picks32", "hier4096"):
        # racks of 8 nodes under zones of 4 racks; leaves outside nodesAll sit in the racks too
        n_spare = 96 if kind == "hier4096" else 8
        leaves = nodes + ["spare%03d" % i for i in range(n_spare)]
        parents = {x: "rack%d" % (j % (len(leaves) // 8)) for j, x in enumerate(leaves)}
        for r in range(len(leaves) // 8):
            parents["rack%d" % r] = "zone%d" % (r % (len(leaves) // 32 or 1))
        kw["node_hierarchy"] = parents
        if kind == "picks32":
            kw["hierarchy_rules"] = {"primary": [(2, 0)] * 8 + [(1, 0)] * 8, "replica": [(2, 1), (1, 0)]}
        else:
            kw["hierarchy_rules"] = {"primary": [(2, 1)], "replica": [(1, 0), (2, 1)]}
    return kw


@pytest.mark.parametrize("kind", ["k16", "eight_states_32_slots", "picks32", "hier4096"])
def test_lockstep_at_abi_limits_string_api(monkeypatch, capfd, kind):
    kw = limit_kwargs(kind, 1100)
    ip = _host.intern_plan(**copy.deepcopy(kw))
    if kind == "hier4096":
        assert ip.n_hier_bits == 4096 and ip.n_nodes == 4000
    if kind == "eight_states_32_slots":
        assert ip.n_states == 8 and ip.n_slots == 32
    ref = _host.plan_out(ip)
    assert FAST.oracle_fast_plan_next_map(ip.in_ptr, ref.out_ptr) == 0
    for name in DEFAULT_ENGINES:
        set_engine_env(monkeypatch, name)
        ip.set_engine(ENGINES[name][0])
        got = _host.plan_out(ip)
        capfd.readouterr()
        _host.run_plan_cuda(ip, got)
        st = parse_stats(capfd.readouterr().err)[0]
        assert st["accepted"] == 0 and st["rebuilds"] == 0, name           # no sticky step: lock-step only
        assert np.array_equal(got.next_rows, ref.next_rows), name
        assert np.array_equal(got.next_shape, ref.next_shape) and np.array_equal(got.warn, ref.warn), name
        assert (got.iters_run, got.converged, got.steps) == (ref.iters_run, ref.converged, ref.steps), name


# ---- 12. 8192 nodes, alone and in a batch with small instances --------------------------------------------------------------

def test_8192_nodes_with_small_instances(ctx, monkeypatch, capfd):
    """The largest N sets 16 nodes per thread for every instance of the batch: the sequencer cannot run at that
    width, so the lock-step kernel takes every pass unless the speculative kernel does."""
    big = flat_tables(1200, [2, 1], 320, 8192, booster=1, max_iters=2)
    small = [flat_tables(1201 + i, ks, 150 + 40 * i, N) for i, (ks, N) in enumerate((([1], 16), ([2, 1], 40), ([3], 100)))]
    for ts in ([big], [big] + small):
        refs, runs = run_engines(ctx, ts, monkeypatch, capfd, engines=("auto", "auto_no_spec", "sequencer", "lockstep"))
        for i in range(len(ts)):
            assert ran_lockstep_only(runs, i, "lockstep") and ran_lockstep_only(runs, i, "sequencer"), i
            assert ran_lockstep_only(runs, i, "auto_no_spec"), i
        assert ran_lockstep_only(runs, 0, "auto")


# ---- move lists at large node-id spaces and partial state visits ----------------------------------------------------------

@pytest.mark.parametrize("P,NN", [(0, 1 << 20), (1, 1 << 20), (3, 1 << 20), (64, 1 << 22)])
def test_moves_at_node_id_limits(ctx, P, NN):
    rng = np.random.default_rng(P + NN)
    caps = (1, 2, 1)
    S = len(caps)
    slot_off = np.concatenate([[0], np.cumsum(caps)]).astype(np.int32)
    SL, max_ops = int(slot_off[-1]), 2 * int(slot_off[-1])
    pool = np.unique(np.concatenate([[NN - 1, NN - 2, 0, 1], rng.integers(0, NN, 6)])).astype(np.int32)

    def rows():
        r = np.full((P, SL), -1, np.int32)
        for p in range(P):
            perm = rng.permutation(pool)[:SL]
            for s in range(S):
                n = rng.integers(0, caps[s] + 1) if p else caps[s]
                r[p, slot_off[s]:slot_off[s] + n] = perm[slot_off[s]:slot_off[s] + n]
        return r
    beg, end = rows(), rows()
    for nv in range(S + 1):
        for favor in (0, 1):
            on = np.zeros((P, max_ops), np.int32); os_ = np.zeros((P, max_ops), np.uint8)
            ok = np.zeros((P, max_ops), np.uint8); oc = np.zeros(P, np.int32)
            assert FAST.oracle_fast_calc_partition_moves(P, S, nv, slot_off.ctypes.data, beg.ctypes.data, end.ctypes.data, favor,
                                                         max_ops, on.ctypes.data, os_.ctypes.data, ok.ctypes.data, oc.ctypes.data) == 0
            got = ctx.calc_partition_moves(slot_off, beg, end, favor, n_visit_states=nv)
            m = np.arange(max_ops)[None, :] < oc[:, None]
            assert np.array_equal(got[3], oc), (nv, favor)
            assert np.array_equal(got[0][m], on[m]) and np.array_equal(got[1][m], os_[m]) and np.array_equal(got[2][m], ok[m])
            h, total = ctx.moves_create(slot_off, beg, end, favor, NN, n_visit_states=nv)
            try:
                off, node, state, kind = ctx.moves_fetch(h, total)
                ref_off = np.concatenate([[0], np.cumsum(oc)]).astype(np.int64)
                assert total == int(oc.sum()) and np.array_equal(off, ref_off), (nv, favor)
                assert np.array_equal(node, on[m]) and np.array_equal(state, os_[m]) and np.array_equal(kind, ok[m])
                for rnd in range(2):
                    nxt = rng.integers(0, max_ops + 1, P).astype(np.int32) if rnd else np.zeros(P, np.int32)
                    node_off, node_parts, best = ctx.moves_available(h, nxt)
                    r_off = np.zeros(NN + 1, np.int32); r_parts = np.zeros(max(1, P), np.int32); r_best = np.zeros(NN, np.int32)
                    assert FAST.oracle_fast_moves_available(P, NN, ref_off.ctypes.data, node.ctypes.data, kind.ctypes.data,
                                                            nxt.ctypes.data, r_off.ctypes.data, r_parts.ctypes.data,
                                                            r_best.ctypes.data) == 0
                    assert np.array_equal(node_off, r_off) and np.array_equal(best, r_best), (nv, favor, rnd)
                    assert np.array_equal(node_parts, r_parts[:r_off[-1]]), (nv, favor, rnd)
            finally:
                ctx.moves_free(h)
