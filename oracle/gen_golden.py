"""Generate tests/golden/*.json by running the REAL reference (build container only).

    python oracle/gen_golden.py            # needs /root/reference

The reference is pure Python over pandas, so it can be imported here but cannot
travel to the GPU box; the vectors it produces are committed instead and pin both
the CPU oracle (tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_*.py).

`vose` (the reference's alias sampler, only used by the sampling algorithms) is not
installed in this image; a stub module is injected so that `import sorobn` works.
Nothing on the exact-inference path touches it.
"""
from __future__ import annotations

import hashlib
import itertools
import json
import os
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")


def import_reference():
    """The reference package, through the same copy (`oracle/_ref`, made by oracle/build_ref.py
    from /root/reference) that the CPU legs of bench.py time."""
    sys.path.insert(0, ROOT)
    from oracle import build_ref

    assert build_ref.build() is not None, "/root/reference is needed to generate the goldens"
    return build_ref.import_reference()


def jsonable(v):
    if isinstance(v, (np.bool_, bool)):
        return bool(v)
    if isinstance(v, (np.integer,)):
        return int(v)
    if isinstance(v, (np.floating,)):
        return float(v)
    return v


def run_case(bn, query, event):
    ans = bn.query(*query, event=event, algorithm="exact")
    idx = [list(map(jsonable, k)) if isinstance(k, tuple) else [jsonable(k)] for k in ans.index.tolist()]
    return {
        "query": list(query),
        "event": [[k, jsonable(v)] for k, v in event.items()],
        "names": list(ans.index.names),
        "index": idx,
        "values": [float(x) for x in ans.to_numpy()],
    }


def run_case_ordered(ref, bn, query, event, order):
    """The reference's operators driven in a given elimination order (oracle/ref_driver.py)."""
    from oracle import ref_driver

    ans = ref_driver.ordered_query(ref, bn, query, event, order)
    idx = [list(map(jsonable, k)) if isinstance(k, tuple) else [jsonable(k)] for k in ans.index.tolist()]
    return {
        "query": list(query),
        "event": [[k, jsonable(v)] for k, v in event.items()],
        "names": list(ans.index.names),
        "index": idx,
        "values": [float(x) for x in ans.to_numpy()],
    }


def impute_cases(ref_bn, our_spec, n_cases, seed):
    """`BayesNet.impute` (bayes_net.py:877-908) on random partial samples: 2-3 missing variables,
    the others observed at states drawn from the network itself (positive probability).
    With ONE missing variable the reference fails: `posterior.idxmax()` is then a scalar and
    `zip(names, scalar)` raises TypeError (bool / int states) or walks the characters of a string
    state (bayes_net.py:905); sorobn_b200 fills the single value, so there is nothing to pin."""
    rng = np.random.default_rng(seed)
    nodes = list(our_spec)
    cases = []
    for _ in range(n_cases):
        full = ref_bn.sample()
        k = int(rng.integers(2, min(3, len(nodes) - 1) + 1))
        missing = set(rng.choice(nodes, size=k, replace=False).tolist())
        sample = {n: (None if n in missing else jsonable(full[n])) for n in nodes}
        filled = ref_bn.impute(dict(sample))
        cases.append({"sample": [[n, sample[n]] for n in nodes],
                      "filled": [[n, jsonable(filled[n])] for n in nodes]})
    return cases


def gibbs_conditionals(ref, ref_bn):
    """The per-variable conditionals P(var | Markov boundary) that `_gibbs_sampling` precomputes
    (bayes_net.py:699-712, restated line by line with the reference's own `pointwise_mul`): they
    are deterministic, unlike the chain itself, so they pin the device sampler's on-the-fly
    conditional exactly."""
    pm = ref.bayes_net.pointwise_mul
    out = {}
    for node in sorted(ref_bn.nodes):
        post = pm(ref_bn.P[n] for n in [node, *ref_bn.children.get(node, [])])
        boundary = ref_bn.markov_boundary(node)
        if boundary:
            post = post.groupby(boundary, group_keys=False).apply(lambda g: g / g.sum())
            post = post.reorder_levels([*boundary, node])
        post = post.sort_index()
        rows = [(list(map(jsonable, k)) if isinstance(k, tuple) else [jsonable(k)]) for k in post.index.tolist()]
        out[node] = {"boundary": list(boundary), "index": rows, "values": [float(x) for x in post.to_numpy()]}
    return out


def example_cases(ref_bn, our_spec):
    """Every single-variable query against every assignment of 0, 1 or 2 evidence
    variables, plus a few two-variable queries."""
    nodes = list(our_spec)
    states = {n: list(our_spec[n][1]) for n in nodes}
    cases = []
    for q in nodes:
        others = [n for n in nodes if n != q]
        for k in (0, 1, 2):
            for evs in itertools.combinations(others, k):
                for vals in itertools.product(*[states[e] for e in evs]):
                    cases.append(((q,), dict(zip(evs, vals))))
    for q2 in list(itertools.combinations(nodes, 2))[:6]:
        others = [n for n in nodes if n not in q2]
        cases.append((q2, {}))
        cases.append((q2, {others[0]: states[others[0]][0]}))
        if len(others) > 1:
            cases.append((q2, {others[0]: states[others[0]][-1], others[-1]: states[others[-1]][0]}))
    return [run_case(ref_bn, q, e) for q, e in cases]


def spec_digest(spec):
    h = hashlib.sha256()
    for n in spec.nodes:
        h.update(n.encode())
        h.update(np.ascontiguousarray(spec.cpt[n], dtype=np.float64).tobytes())
    return h.hexdigest()


def synthetic_cases(ref, synthetic, spec, n_cases, n_ev_range, seed, n_query=(1, 2)):
    bn = synthetic.load(spec, ref.BayesNet)
    rng = np.random.default_rng(seed)
    cases = []
    for c in range(n_cases):
        nq = int(rng.integers(n_query[0], n_query[1] + 1))
        ne = int(rng.integers(n_ev_range[0], n_ev_range[1] + 1))
        perm = rng.permutation(len(spec.nodes))
        query = [spec.nodes[i] for i in perm[:nq]]
        evs = [spec.nodes[i] for i in perm[nq:nq + ne]]
        row = synthetic.random_events(spec, evs, 1, seed=seed * 1000 + c)
        event = {v: int(row[v].iloc[0]) for v in evs}
        cases.append(run_case(bn, query, event))
    return cases


def ordered_golden(ref):
    """The reference's operators driven in the device program's min-fill order (oracle/ref_driver.py,
    what the CPU legs of bench.py time) on a small grid: three seeded evidence rows."""
    from sorobn_b200 import BayesNet, planner, synthetic

    kwargs = dict(rows=4, cols=4, n_states=3, seed=11)
    spec = synthetic.grid(**kwargs)
    net = synthetic.load(spec, BayesNet)._compiled
    query, evs = ("g0303",), ("g0001", "g0102", "g0203", "g0300")
    plan = planner.build_plan(net, [net.index[q] for q in query], [net.index[e] for e in evs])
    order = [net.names[v] for v in plan.order]
    bn = synthetic.load(spec, ref.BayesNet)
    events = synthetic.random_events(spec, evs, 3, seed=5)
    cases = [run_case_ordered(ref, bn, query, {v: int(events[v].iloc[b]) for v in evs}, order)
             for b in range(len(events))]
    return {"network": "grid4x4s3", "kind": "ordered", "generator": "grid", "kwargs": kwargs,
            "digest": spec_digest(spec), "order": order, "cases": cases}


def main():
    ref = import_reference()
    sys.path.insert(0, ROOT)
    from sorobn_b200 import examples, synthetic

    os.makedirs(OUT, exist_ok=True)
    only_workload = "--workload-only" in sys.argv
    with open(os.path.join(OUT, "ordered_grid4x4s3.json"), "w") as f:
        json.dump(ordered_golden(ref), f)

    # ---- the reference's own example networks -------------------------------------
    for name, spec in ({} if only_workload else examples.NETWORKS).items():
        ref_bn = examples.build(spec, cls=ref.BayesNet)
        # sanity: our data-driven spec reproduces the reference's own example network
        theirs = getattr(ref.examples, name)()
        for node in theirs.P:
            a = theirs.P[node].sort_index()
            b = ref_bn.P[node].sort_index()
            assert list(a.index.names) == list(b.index.names), (name, node)
            assert np.allclose(a.to_numpy(), b.reindex(a.index).to_numpy()), (name, node)
        assert theirs.nodes == ref_bn.nodes
        t = time.time()
        cases = example_cases(ref_bn, spec)
        with open(os.path.join(OUT, f"{name}.json"), "w") as f:
            json.dump({"network": name, "kind": "example", "nodes": ref_bn.nodes, "cases": cases}, f)
        print(f"{name}: {len(cases)} cases in {time.time() - t:.1f}s")

    # ---- predict_proba (bayes_net.py:934-962) on the example networks ----------------
    import pandas as pd

    for name, spec in ({} if only_workload else examples.NETWORKS).items():
        ref_bn = examples.build(spec, cls=ref.BayesNet)
        fjd = ref_bn.full_joint_dist()
        nodes = list(fjd.index.names)
        cases = []
        # every row of the joint (all variables observed)
        full = pd.DataFrame(fjd.index.tolist(), columns=nodes)
        cases.append({"columns": nodes, "rows": [[jsonable(v) for v in r] for r in full.to_numpy().tolist()],
                      "prob": [float(x) for x in ref_bn.predict_proba(full).to_numpy()]})
        # marginals over subsets of 2 and 3 columns (one column hits a reference quirk: it
        # returns the whole marginal instead of per-row values)
        for k in (2, 3):
            for cols in list(itertools.combinations(nodes, k))[:8]:
                sub = full[list(cols)].drop_duplicates().reset_index(drop=True)
                prob = ref_bn.predict_proba(sub)
                cases.append({"columns": list(cols), "rows": [[jsonable(v) for v in r] for r in sub.to_numpy().tolist()],
                              "prob": [float(x) for x in prob.to_numpy()]})
        with open(os.path.join(OUT, f"predict_proba_{name}.json"), "w") as f:
            json.dump({"network": name, "kind": "predict_proba", "cases": cases}, f)
        print(f"predict_proba {name}: {len(cases)} cases, {sum(len(c['rows']) for c in cases)} rows")

    # ---- impute (bayes_net.py:877-908) and the Gibbs conditionals (bayes_net.py:699-712) ------
    for name, spec in ({} if only_workload else examples.NETWORKS).items():
        ref_bn = examples.build(spec, cls=ref.BayesNet, seed=7)
        cases = impute_cases(ref_bn, spec, 25, seed=3)
        with open(os.path.join(OUT, f"impute_{name}.json"), "w") as f:
            json.dump({"network": name, "kind": "impute", "cases": cases}, f)
        cond = gibbs_conditionals(ref, ref_bn)
        with open(os.path.join(OUT, f"gibbs_conditionals_{name}.json"), "w") as f:
            json.dump({"network": name, "kind": "gibbs_conditionals", "nodes": cond}, f)
        print(f"impute {name}: {len(cases)} cases; gibbs conditionals: {sum(len(c['values']) for c in cond.values())} entries")

    # ---- synthetic networks ----------------------------------------------------------
    jobs = [
        ("grid4x4s3", ("grid", dict(rows=4, cols=4, n_states=3, seed=11)), 40, (0, 8)),
        ("dag12p3s3", ("random_dag", dict(n_nodes=12, max_parents=3, n_states=3, seed=5)), 40, (0, 8)),
        ("chain9s4", ("chain", dict(n_nodes=9, n_states=4, seed=3)), 20, (0, 5)),
        ("dag20p4s4", ("random_dag", dict(n_nodes=20, max_parents=4, n_states=4, seed=8, window=6)), 20, (4, 12)),
    ]
    for name, (kind, kwargs), n_cases, ev_range in ([] if only_workload else jobs):
        spec = getattr(synthetic, kind)(**kwargs)
        t = time.time()
        cases = synthetic_cases(ref, synthetic, spec, n_cases, ev_range, seed=17)
        with open(os.path.join(OUT, f"{name}.json"), "w") as f:
            json.dump({"network": name, "kind": "synthetic", "generator": kind, "kwargs": kwargs,
                       "digest": spec_digest(spec), "cases": cases}, f)
        print(f"{name}: {len(cases)} cases in {time.time() - t:.1f}s")

    # ---- the benchmark grid (BASELINE.json configs[2]): a few rows of the real workload
    from sorobn_b200 import workloads

    from sorobn_b200 import BayesNet, planner

    wl = workloads.grid10x10()
    bn = synthetic.load(wl.spec, ref.BayesNet)
    ours = wl.build(BayesNet)
    net = ours._compiled
    plan = planner.build_plan(net, [net.index[q] for q in wl.query], [net.index[e] for e in wl.evidence])
    order = [net.names[v] for v in plan.order]  # min-fill, the order the device program uses
    events = wl.events(4, seed=123, bn=ours)
    cases, times = [], []
    for b in range(len(events)):
        event = {v: int(events[v].iloc[b]) for v in wl.evidence}
        t = time.perf_counter()
        cases.append(run_case_ordered(ref, bn, wl.query, event, order))
        times.append(time.perf_counter() - t)
        print(f"  grid row {b}: {times[-1]:.2f}s")
    with open(os.path.join(OUT, "grid10x10s5_bench.json"), "w") as f:
        json.dump({"network": "grid10x10s5", "kind": "workload", "workload": "grid10x10",
                   "digest": spec_digest(wl.spec), "order": order, "reference_seconds_per_query": times,
                   "note": "reference operators driven in min-fill order (the reference's own set-order "
                           "elimination is OOM-killed on this network)", "cases": cases}, f)
    print(f"grid10x10 workload: reference takes {np.mean(times):.2f}s per query here ({os.cpu_count()} cores)")


if __name__ == "__main__":
    main()
