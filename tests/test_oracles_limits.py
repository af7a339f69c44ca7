"""Literal oracle (oracle/literal.cpp) vs array-form oracle (oracle/fast.c through the interning layer) at the
limits the C ABI advertises: k up to 16 in one state, 8 states and 32 slots, equal state priorities,
rules x constraints = 32 picks, deep hierarchies with leaves outside nodesAll, and prevMap entries under state
names outside the model.  The GPU tests at these shapes (test_gpu_kernel_limits.py) use the fast oracle as their
checker; this pins it to the literal one there.  P stays small so the literal oracle is quick.  CPU only."""
import copy
import random

import pytest

from oracle_loader import literal
from test_fast_oracle import FAST, _host

L = literal()


def limit_instance(seed):
    """k in {0..16}, up to 8 states sharing at most 32 slots, weights from -3 to 9, the booster, stickiness,
    hierarchies up to 5 levels over nodes plus spare leaves outside nodesAll, and up to 32 picks per state.
    "dead" state keys sit only on prevMap entries that are not being assigned: the reference panics when an
    assigned partition holds a state outside the model."""
    rnd = random.Random(seed)
    N = rnd.randint(8, 48)
    nodes = ["n%02d" % i for i in range(N)]
    S = rnd.randint(3, 8)
    states = ["st%d" % i for i in range(S)]
    full = rnd.random() < 0.3                      # spend the whole 32-slot budget
    budget = 32
    ks = []
    for i in range(S):
        k = rnd.choice([0, 1, 2, 4, 5, 8, 16]) if budget > 0 else 0
        k = min(k, budget, 16)
        budget -= k
        ks.append(k)
    if full and budget > 0:
        for i in range(S):
            add = min(16 - ks[i], budget)
            ks[i] += add
            budget -= add
    equal = rnd.random() < 0.3
    model = {s: (0 if equal else (rnd.choice([i, 0]) if rnd.random() < 0.3 else i), ks[i]) for i, s in enumerate(states)}
    P = rnd.randint(1, 10)
    names = [str(i) for i in range(P)]

    def row():
        avail = nodes[:]
        rnd.shuffle(avail)
        d = {}
        for s in states:
            if rnd.random() < 0.2:
                continue
            c = rnd.randint(0, min(model[s][1] + 1, len(avail)))
            d[s] = [avail.pop() for _ in range(c)]
        return d

    prev = {n: row() for n in names}
    assigned = [n for n in names if rnd.random() < 0.8] or names[:1]
    assign = {n: copy.deepcopy(prev[n]) if rnd.random() < 0.8 else row() for n in assigned}
    for n in names:
        if n not in assign and rnd.random() < 0.7:
            prev[n]["dead"] = rnd.sample(nodes, rnd.randint(0, 2))
    prev["zz_dead"] = {"dead": [rnd.choice(nodes)], states[0]: [rnd.choice(nodes)]}
    remove = rnd.sample(nodes, rnd.randint(0, N // 4))
    if any(n not in prev for n in assign):
        remove = []
    kw = dict(prev_map=prev, partitions_to_assign=assign, nodes_all=nodes, nodes_to_remove=remove,
              nodes_to_add=rnd.sample(nodes, rnd.randint(0, N)), model=model)
    if rnd.random() < 0.6:
        kw["node_weights"] = {n: rnd.choice([-3, -2, 0, 1, 2, 3, 9]) for n in nodes if rnd.random() < 0.7}
        kw["booster"] = int(rnd.random() < 0.5)
    if rnd.random() < 0.6:
        kw["partition_weights"] = {n: rnd.randint(-3, 9) for n in names if rnd.random() < 0.6}
        kw["state_stickiness"] = {s: rnd.randint(0, 4) for s in states if rnd.random() < 0.6}
    if rnd.random() < 0.7:
        parents = {}
        cur = nodes[:] + ["spare%d" % i for i in range(rnd.randint(1, 4))]
        for lv in range(rnd.randint(1, 5)):
            g = max(1, len(cur) // rnd.randint(2, 4))
            nxt = ["g%d_%d" % (lv, j) for j in range(g)]
            for i, c in enumerate(cur):
                parents[c] = nxt[i % g]
            cur = nxt
        kw["node_hierarchy"] = parents
        rules = {}
        for s in states:
            k = model[s][1]
            if k and rnd.random() < 0.7:
                nr = 32 // k if rnd.random() < 0.5 else rnd.randint(1, 32 // k)   # often exactly 32 picks
                rules[s] = [(rnd.randint(0, 5), rnd.randint(0, 5)) for _ in range(nr)]
        kw["hierarchy_rules"] = rules
    return kw


def test_generator_reaches_the_limits():
    ks, slots, states, picks, equal, outside, dead = set(), set(), set(), set(), False, False, False
    for seed in range(300):
        kw = limit_instance(seed)
        m = kw["model"]
        ks |= {k for _, k in m.values()}
        slots.add(sum(k for _, k in m.values()))
        states.add(len(m))
        equal |= len({p for p, _ in m.values()}) < len(m)
        for s, rs in kw.get("hierarchy_rules", {}).items():
            picks.add(len(rs) * m[s][1])
        outside |= any(c.startswith("spare") for c in kw.get("node_hierarchy", {}))
        dead |= any("dead" in v for v in kw["prev_map"].values())
    assert 16 in ks and 32 in slots and 8 in states and 32 in picks and equal and outside and dead


@pytest.mark.parametrize("chunk", range(6))
def test_literal_equals_fast_at_abi_limits(chunk):
    for seed in range(chunk * 100, (chunk + 1) * 100):
        kw = limit_instance(seed)
        lit = L.plan_next_map_ex(**copy.deepcopy(kw))
        ip = _host.intern_plan(**copy.deepcopy(kw))
        out = _host.plan_out(ip)
        assert FAST.oracle_fast_plan_next_map(ip.in_ptr, out.out_ptr) == 0, seed
        next_map, warnings = _host.unintern_plan(ip, out)
        assert next_map == lit["next_map"], seed
        assert warnings == lit["warnings"], seed
        assert (out.iters_run, out.steps) == (lit["iterations"], lit["steps"]), seed
