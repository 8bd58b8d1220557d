"""Host-side mirror of `sorobn.BayesNet` for the exact-inference path.

Same surface as the reference (/root/reference/sorobn/bayes_net.py:259-1075) for
everything on the hot path: the constructor's structure grammar, the `P` dict of
pandas Series, `prepare()`, `query(..., algorithm="exact")` and `impute()`, plus the
cheap structural helpers.  What differs is where the arithmetic runs: `prepare()`
additionally compiles the CPTs into dense fp32 tables, and `query()` hands a flat
variable-elimination program to the CUDA engine (`sorobn_b200.engine`, a ctypes
shim over `libsorobn_b200.so`).  There is no CPU fallback: without the CUDA library
or a GPU `query()` raises.

`query_many()` is the batched form of `query()` (one posterior per evidence row of a
DataFrame); it is what the multi-GPU sharding and the benchmark drive.

`predict_proba` / `predict_log_proba` / `full_joint_dist` (bayes_net.py:398-465, :934-973) run
on the same kernels: the probability of a row is the normaliser of an elimination with the
row as evidence.

The approximate algorithms run on the device too (csrc/sbn_gibbs.cuh): `algorithm="gibbs"`
(bayes_net.py:665-737) one chain per evidence row, `"likelihood"` (:621-663) and `"rejection"`
(:577-619) n_iterations forward samples per row.  `fit` / `partial_fit` / `sample`
(:467-575) stay on the host (pandas / numpy), as in the reference.
"""
from __future__ import annotations

import graphlib
import random
import threading
import typing
from collections import OrderedDict, defaultdict

import numpy as np
import pandas as pd

from . import planner as _planner

__all__ = ["BayesNet"]


def _as_list(obj):
    return obj if isinstance(obj, list) else [obj]


class BayesNet:
    """Bayesian network with CUDA exact inference.

    Parameters mirror bayes_net.py:286: `structure` items are either bare nodes or
    (parent(s), child(ren)) tuples whose members may be lists.
    """

    def __init__(self, *structure, prior_count: int = None, seed: int = None, device: int | None = None):
        self.prior_count = prior_count
        self.seed = seed
        self._rng = random.Random(seed)  # seeds the device samplers (bayes_net.py:289)
        self.device = device

        parents = defaultdict(set)
        children = defaultdict(set)
        lone = set()
        for item in structure:
            if isinstance(item, tuple):
                srcs, dsts = item
                for s in _as_list(srcs):
                    for d in _as_list(dsts):
                        parents[d].add(s)
                        children[s].add(d)
            else:
                lone.add(item)

        # bayes_net.py:312-315: plain dicts of sorted lists
        self.parents = {n: sorted(ps) for n, ps in parents.items()}
        self.children = {n: sorted(cs) for n, cs in children.items()}

        # bayes_net.py:317-322: topological order, lexicographic within a level.
        # graphlib raises CycleError for a cyclic structure, as the reference does.
        sorter = graphlib.TopologicalSorter()
        for n in sorted({*self.parents, *self.children, *lone}):
            sorter.add(n, *self.parents.get(n, []))
        self.nodes = list(sorter.static_order())

        self.P = {}
        self._P_sizes = {}
        self._compiled = None
        # compiled device programs, one per (query vars, evidence vars, mode); least recently
        # used ones are dropped (their streams, graph and scratch are freed with them)
        self._engine_cache = OrderedDict()
        self._cache_lock = threading.RLock()  # query_many(devices=...) looks programs up from worker threads
        self.max_cached_programs = 128

    def __getstate__(self):
        """Copies and pickles carry the network, not the device objects (programs hold CUDA
        handles that must have exactly one owner); they are rebuilt on first use."""
        state = self.__dict__.copy()
        state["_engine_cache"] = OrderedDict()
        state.pop("_cache_lock", None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._cache_lock = threading.RLock()

    # ------------------------------------------------------------------ structure
    def ancestors(self, node):
        """bayes_net.py:373-378."""
        found = set()
        frontier = list(self.parents.get(node, ()))
        while frontier:
            p = frontier.pop()
            if p not in found:
                found.add(p)
                frontier.extend(self.parents.get(p, ()))
        return found

    @property
    def roots(self):
        return [n for n in self.nodes if n not in self.parents]

    @property
    def leaves(self):
        return [n for n in self.nodes if n not in self.children]

    @property
    def is_tree(self):
        return all(len(ps) <= 1 for ps in self.parents.values())

    def markov_boundary(self, node):
        """Parents, children and the children's other parents (bayes_net.py:1002-1039)."""
        kids = self.children.get(node, [])
        blanket = set(self.parents.get(node, [])) | set(kids)
        for k in kids:
            blanket |= set(self.parents[k])
        blanket.discard(node)
        return sorted(blanket)

    def impute_many(self, samples: pd.DataFrame, **query_params) -> pd.DataFrame:
        """Batched `impute` (bayes_net.py:877-908): every missing cell (None / NaN) of `samples`
        is replaced by the most probable joint value of that row's missing variables given its
        observed ones.  Rows are grouped by which columns they lack; each group is one
        `query_many` call, i.e. one device program run over all its rows."""
        out = samples.copy()
        missing = samples.isna()
        patterns = missing.apply(lambda r: tuple(c for c in samples.columns if r[c]), axis=1)
        for pattern, rows in samples.groupby(patterns, sort=False).groups.items():
            if not pattern:
                continue
            observed = [c for c in samples.columns if c not in pattern]
            if not observed:
                raise ValueError("a row with every variable missing cannot be imputed")
            post = self.query_many(*pattern, events=samples.loc[rows, observed], **query_params)
            values = post.to_numpy()
            impossible = np.isnan(values).all(axis=1)
            if impossible.any():
                # `impute` raises here too (idxmax of the reference's empty posterior, bayes_net.py:902)
                raise ValueError(f"{int(impossible.sum())} row(s) have evidence of probability zero "
                                 f"(first: {post.index[impossible][0]!r}); they cannot be imputed")
            best = values.argmax(axis=1)
            labels = post.columns  # joint states, variables sorted by name
            names = list(labels.names)
            for k, name in enumerate(names):
                values = labels.get_level_values(k) if len(names) > 1 else labels
                out.loc[rows, name] = np.asarray(values, dtype=object)[best]
        return out.infer_objects()

    def graphviz(self):
        """The structure as a `graphviz.Digraph` (bayes_net.py:910-929); the module is imported
        here, so it is only needed when this is called."""
        import graphviz

        g = graphviz.Digraph()
        for node in self.nodes:
            g.node(str(node))
        for parent, kids in self.children.items():
            for kid in kids:
                g.edge(str(parent), str(kid))
        return g

    def _repr_svg_(self):
        return self.graphviz()

    def iter_dfs(self):
        """Depth-first walk from each root (bayes_net.py:1041-1075)."""
        seen = set()

        def walk(n):
            yield n
            seen.add(n)
            for c in self.children.get(n, []):
                if c not in seen:
                    yield from walk(c)

        for r in self.roots:
            yield from walk(r)

    # -------------------------------------------------------------------- prepare
    def prepare(self) -> "BayesNet":
        """House-keeping (bayes_net.py:327-371) + compile the tables for the device.

        The pandas side ends in the same state as the reference's: each `P[node]` is
        a Series named "P(node | parents)" whose index levels are
        [*parents, node], sorted.  Then every CPT is densified into an fp32 table
        (domain order == the sorted level values) ready to be shipped.
        """
        for node in list(self.P):
            table = self.P[node]
            node_parents = self.parents.get(node, [])

            if isinstance(table, pd.DataFrame):
                # bayes_net.py:339-358
                if "p" not in table.columns:
                    raise ValueError(
                        f"DataFrame for '{node}' must have a 'p' column containing probabilities"
                    )
                given = [c for c in table.columns if c != "p"]
                wanted = set(node_parents) | {node}
                if set(given) != wanted:
                    raise ValueError(
                        f"DataFrame for '{node}' has columns {given}, but expected {sorted(wanted)} (plus 'p')"
                    )
                table = table.set_index([*node_parents, node])["p"]
                self.P[node] = table

            if node not in self.parents:
                table.index.name = node
            elif set(table.index.names) == {*node_parents, node}:
                table = table.reorder_levels([*node_parents, node])
            else:
                table.index.names = [*node_parents, node]
            # reorder_levels returns a new object: sort it and store it back so that
            # P[node] always carries [*parents, node] levels, sorted
            table = table.sort_index()
            table.name = (
                f"P({node} | {', '.join(map(str, node_parents))})" if node in self.parents else f"P({node})"
            )
            self.P[node] = table

        self._compile()
        return self

    def _compile(self):
        missing = [n for n in self.nodes if n not in self.P]
        if missing:
            # The reference tolerates a partially specified network until a query
            # touches the hole; keep that: compile lazily once everything is there.
            self._compiled = None
            self._engine_cache = OrderedDict()
            return
        seen = {n: set() for n in self.nodes}
        for node, series in self.P.items():
            idx = series.index
            if isinstance(idx, pd.MultiIndex):
                for lvl, name in enumerate(idx.names):
                    seen[name].update(idx.get_level_values(lvl).unique().tolist())
            else:
                seen[node].update(idx.unique().tolist())
        domains = {n: sorted(v) for n, v in seen.items()}
        vid = {n: i for i, n in enumerate(self.nodes)}
        cpts = []
        for node in self.nodes:
            scope = [*self.parents.get(node, []), node]
            series = self.P[node]
            shape = [len(domains[v]) for v in scope]
            dense = np.zeros(shape, dtype=np.float64)
            idx = series.index
            if isinstance(idx, pd.MultiIndex):
                codes = [pd.Index(domains[v]).get_indexer(idx.get_level_values(l)) for l, v in enumerate(scope)]
            else:
                codes = [pd.Index(domains[node]).get_indexer(idx)]
            dense[tuple(codes)] = series.to_numpy(dtype=np.float64)
            cpts.append(dense)
        self._compiled = _planner.CompiledNet(
            names=list(self.nodes),
            domains=[domains[n] for n in self.nodes],
            parents=[[vid[p] for p in self.parents.get(n, [])] for n in self.nodes],
            cpt=cpts,
        )
        self._engine_cache = OrderedDict()

    # ------------------------------------------------------------- learning / sampling
    def partial_fit(self, X: pd.DataFrame) -> "BayesNet":
        """Update every CPT from a batch of rows (host side, pandas; bayes_net.py:467-510).

        Counts are kept per node (`_P_sizes` holds the number of rows behind every parent
        configuration), so feeding the data in chunks gives the same tables as one `fit`.
        With `prior_count`, every combination of the values seen in the first batch gets one
        pseudo-observation, as in the reference."""
        for child, parents in self.parents.items():
            scope = [*parents, child]
            seen = X.groupby(scope).size()
            if child in self.P:
                counts = (self.P[child] * self._P_sizes[child]).add(seen, fill_value=0)
            else:
                counts = seen
                if self.prior_count:
                    grid = pd.MultiIndex.from_product([X[v].unique() for v in scope], names=scope)
                    counts = counts.add(pd.Series(1, index=grid), fill_value=0)
            totals = counts.groupby(parents).sum()
            self._P_sizes[child] = totals
            self.P[child] = counts / totals
        for root in self.roots:
            if root in self.P:
                counts = (self.P[root] * self._P_sizes[root]).add(X[root].value_counts(), fill_value=0)
                self._P_sizes[root] += len(X)
                self.P[root] = counts / self._P_sizes[root]
            else:
                self._P_sizes[root] = len(X)
                self.P[root] = X[root].value_counts(normalize=True)
        self.prepare()
        return self

    def fit(self, X: pd.DataFrame) -> "BayesNet":
        """Estimate every CPT from `X` (bayes_net.py:512-516)."""
        self.P = {}
        self._P_sizes = {}
        return self.partial_fit(X)

    def sample(self, n=1, init: dict | None = None, method="forward"):
        """Forward (ancestral) samples (bayes_net.py:550-575): a Series for n == 1, otherwise a
        DataFrame with the columns sorted.  Variables named in `init` keep the given value.
        Vectorised over the n samples on the host; the stream comes from `seed`."""
        if method != "forward":
            raise ValueError("Unknown method, must be one of: forward")
        if self._compiled is None:
            self._compile()
            if self._compiled is None:
                raise ValueError("every node needs a CPT in P before sampling; call prepare()")
        net = self._compiled
        init = init or {}
        rng = np.random.default_rng(self._rng.getrandbits(63))
        n = int(n)
        codes = np.zeros((len(net.names), n), dtype=np.int64)
        for v, name in enumerate(net.names):
            if name in init:
                codes[v] = net.domains[v].index(init[name])
                continue
            table = net.cpt[v]
            probs = table[tuple(codes[p] for p in net.parents[v])] if net.parents[v] else np.broadcast_to(table, (n, table.shape[-1]))
            cdf = np.cumsum(probs, axis=-1)
            u = rng.random((n, 1)) * cdf[:, -1:]
            codes[v] = np.minimum((u > cdf).sum(axis=-1), table.shape[-1] - 1)
        frame = pd.DataFrame({name: np.asarray(net.domains[v], dtype=object)[codes[v]] for v, name in enumerate(net.names)})
        frame = frame.infer_objects().sort_index(axis="columns")
        return frame if n > 1 else frame.iloc[0]

    # ---------------------------------------------------------------------- query
    def _plan(self, query, evidence_vars, mode, robust=False, device=None, slot=0):
        """(plan, program) for the pair on `device`, cached.  A program is not thread-safe: callers
        that run several at once on the same device ask for distinct `slot`s."""
        with self._cache_lock:
            return self._plan_locked(query, evidence_vars, mode, robust, device, slot)

    def _plan_locked(self, query, evidence_vars, mode, robust, device, slot):
        if self._compiled is None:
            self._compile()
            if self._compiled is None:
                raise ValueError("every node needs a CPT in P before querying; call prepare()")
        net = self._compiled
        device = self.device if device is None else device
        key = (tuple(query), tuple(evidence_vars), mode, robust, device, slot)
        hit = self._engine_cache.get(key)
        if hit is None:
            for name in (*query, *evidence_vars):
                if name not in net.index:
                    raise KeyError(name)
            twin = next((v for k, v in self._engine_cache.items() if isinstance(v, tuple) and k[:4] == key[:4]), None)
            plan = twin[0] if twin else _planner.build_plan(
                net, [net.index[q] for q in query], [net.index[e] for e in evidence_vars],
                mode=mode, allow_empty_query=True)  # the same plan serves every device
            from . import engine  # raises if libsorobn_b200.so cannot be loaded

            # single-event programs run in float64 (latency-bound anyway); batches in float32,
            # except the robust re-run of flagged rows (mode key "batched64")
            hit = (plan, engine.Program(plan, device=device, f64=(mode == _planner.MODE_FLAT or robust)))
            self._engine_cache[key] = hit
            self._evict()
        else:
            self._engine_cache.move_to_end(key)
        return hit

    def _evict(self):
        """Drop the least recently used device objects (programs and samplers) beyond the cap."""
        while len(self._engine_cache) > self.max_cached_programs:
            _, old = self._engine_cache.popitem(last=False)
            (old[1] if isinstance(old, tuple) else old).close()

    def _encode_events(self, evidence_vars, columns):
        """State values -> uint8 codes [n_ev, B].  Unknown values get code 255 and the
        row is reported as impossible evidence (the reference's boolean filter at
        bayes_net.py:772-774 leaves an empty factor, hence an empty answer)."""
        net = self._compiled
        n = len(columns[0]) if columns else 0
        codes = np.empty((len(evidence_vars), n), dtype=np.uint8)
        bad = np.zeros(n, dtype=bool)
        for i, (name, col) in enumerate(zip(evidence_vars, columns)):
            dom = pd.Index(net.domains[net.index[name]])
            c = dom.get_indexer(pd.Index(col))
            bad |= c < 0
            codes[i] = np.where(c < 0, 0, c).astype(np.uint8)
        return codes, bad

    def _answer_index(self, plan):
        net = self._compiled
        names = [net.names[v] for v in plan.query]
        doms = [net.domains[v] for v in plan.query]
        if len(names) == 1:
            return pd.Index(doms[0], name=names[0])
        return pd.MultiIndex.from_product(doms, names=names)

    def query(self, *query, event: dict, algorithm="exact", n_iterations=100) -> pd.Series:
        """Answer P(query | event) (bayes_net.py:796-875), exact inference on the GPU.

        The answer is a Series named "P(q1, q2)" indexed by the query variables
        (levels sorted by name, rows sorted by state); states with zero posterior
        are left out, as the reference's zero-filtering join does
        (bayes_net.py:253-256).
        """
        if not query:
            raise ValueError("At least one query variable has to be specified")
        for q in query:
            if q in event:
                raise ValueError("A query variable cannot be part of the event")
        if algorithm in ("gibbs", "likelihood", "rejection"):
            freq = self._sample_query(algorithm, query, tuple(event), [[event[v]] for v in event], 1, n_iterations)
            values = freq[0][:, 0].astype(np.float64)
            name = f"P({', '.join(map(str, query))})"
            if np.isnan(values).any():  # rejection sampling kept no sample: the reference's answer is empty
                return pd.Series([], index=freq[1][:0], name=name, dtype=np.float64)
            answer = pd.Series(values, index=freq[1], name=name)
            return answer[answer > 0]  # the reference only lists the states that were sampled
        if algorithm != "exact":
            raise ValueError("Unknown algorithm, must be one of: exact, gibbs, likelihood, rejection")

        ev_vars = tuple(event)
        plan, program = self._plan(query, ev_vars, _planner.MODE_FLAT)
        # One event is launch-latency bound on the device (~20 us): the host side must not cost ten
        # times that.  State codes come from per-variable dicts, the answer's index is cached on the plan.
        net = self._compiled
        codes = np.empty((len(ev_vars), 1), dtype=np.uint8)
        bad = False
        for i, v in enumerate(ev_vars):
            code = self._code_of(net.index[v]).get(event[v], -1)
            bad |= code < 0
            codes[i, 0] = max(code, 0)
        index = getattr(plan, "_answer_index_cache", None)
        if index is None:
            index = plan._answer_index_cache = self._answer_index(plan)
        name = f"P({', '.join(map(str, query))})"
        if bad:  # a value outside the variable's domain: the reference's filter leaves nothing
            return pd.Series([], index=index[:0], name=name, dtype=np.float64)
        post = program.run(codes, 1)[:, 0].astype(np.float64)
        if np.isnan(post).any():  # impossible evidence: P(event) == 0
            return pd.Series([], index=index[:0], name=name, dtype=np.float64)
        keep = post > 0
        if keep.all():
            return pd.Series(post, index=index, name=name)
        return pd.Series(post[keep], index=index[keep], name=name)

    def _code_of(self, v):
        """state value -> uint8 code of variable id `v` (position in its sorted domain)."""
        cache = self.__dict__.setdefault("_code_cache", {})
        table = cache.get(v)
        if table is None or cache.get("net") is not self._compiled:
            if cache.get("net") is not self._compiled:
                cache.clear()
                cache["net"] = self._compiled
            table = cache[v] = {value: k for k, value in enumerate(self._compiled.domains[v])}
        return table

    def _sample_query(self, algorithm, query, ev_vars, columns, n_rows, n_iterations):
        """The approximate algorithms on the device, per evidence row: one Gibbs chain
        (bayes_net.py:665-737), or n_iterations forward samples for likelihood weighting
        (:621-663) / rejection sampling (:577-619).  Returns (estimates [Q, n_rows], index)."""
        if self._compiled is None:
            self._compile()
            if self._compiled is None:
                raise ValueError("every node needs a CPT in P before querying; call prepare()")
        net = self._compiled
        for name in (*query, *ev_vars):
            if name not in net.index:
                raise KeyError(name)
        key = ("sampler", tuple(query), tuple(ev_vars))
        sampler = self._engine_cache.get(key)
        q_sorted = sorted(query)  # same key as the exact path (planner: sorted by name) and bayes_net.py:873
        if sampler is None:
            from . import engine

            nonevents = sorted(set(self.nodes) - set(ev_vars))  # bayes_net.py:697, the Gibbs cycle order
            sampler = engine.GibbsSampler(net, [net.index[q] for q in q_sorted], [net.index[e] for e in ev_vars],
                                          [net.index[v] for v in nonevents], device=self.device)
            self._engine_cache[key] = sampler
            self._evict()
        codes, bad = self._encode_events(ev_vars, columns)
        if bad.any():
            raise ValueError("an event value is not a state of its variable")
        freq = sampler.run(codes, n_rows, n_iterations, self._rng.getrandbits(63), algorithm=algorithm)
        doms = [net.domains[net.index[q]] for q in q_sorted]
        index = pd.Index(doms[0], name=q_sorted[0]) if len(q_sorted) == 1 else pd.MultiIndex.from_product(doms, names=q_sorted)
        return freq, index

    def query_many(self, *query, events: pd.DataFrame, algorithm="exact", n_iterations=100,
                   devices: typing.Sequence[int] | None = None) -> pd.DataFrame:
        """Batched `query`: one posterior per row of `events` (columns = evidence
        variables).  Returns a DataFrame with one row per evidence row and one column
        per joint state of the query variables (same order as `query`'s index);
        impossible rows are NaN.  Zero-probability states stay (as 0.0).

        devices: CUDA device ids to shard the rows over (exact algorithm).  Rows are independent,
        so each device answers a contiguous slice with its own program (one host thread per
        device; the C ABI call releases the GIL) and the slices land in one host array: there is
        no collective.  One process per GPU under torchrun is `sorobn_b200.sharding.query_many_sharded`."""
        if not query:
            raise ValueError("At least one query variable has to be specified")
        ev_vars = tuple(events.columns)
        for q in query:
            if q in ev_vars:
                raise ValueError("A query variable cannot be part of the event")
        if algorithm in ("gibbs", "likelihood", "rejection"):
            freq, index = self._sample_query(algorithm, query, ev_vars, [events[v].to_numpy() for v in ev_vars],
                                             len(events.index), n_iterations)
            return pd.DataFrame(freq.T.astype(np.float64), index=events.index, columns=index)
        if algorithm != "exact":
            raise ValueError("Unknown algorithm, must be one of: exact, gibbs, likelihood, rejection")
        plan, _ = self._plan(query, ev_vars, _planner.MODE_BATCHED, device=None if devices is None else devices[0])
        n = len(events.index)
        if n == 0:
            return pd.DataFrame(np.zeros((0, plan.Q)), index=events.index, columns=self._answer_index(plan))
        codes, bad = self._encode_events(ev_vars, [events[v].to_numpy() for v in ev_vars])
        if not ev_vars:
            bad = np.zeros(n, dtype=bool)
        if devices is None or len(devices) <= 1:
            post = self._posterior_codes(query, ev_vars, codes, bad, device=None if devices is None else devices[0])
        else:
            post = self._posterior_codes_multi(query, ev_vars, codes, bad, list(devices))
        out = pd.DataFrame(post.T, index=events.index, columns=self._answer_index(plan))
        if bad.any():
            out.loc[events.index[bad]] = np.nan
        return out

    def _posterior_codes(self, query, ev_vars, codes, bad, device=None, slot=0):
        """Posterior float64 [Q, n] for uint8 evidence codes [n_ev, n] on one device.  Rows the
        float32 program flags (NaN: impossible evidence, or an entry below the float32 range)
        are settled in float64 -- a few one by one with the single-event program, many as one
        batch with the batched float64 program; a row that is still NaN there is impossible."""
        n = codes.shape[1] if len(ev_vars) else len(bad)
        _, program = self._plan(query, ev_vars, _planner.MODE_BATCHED, device=device, slot=slot)
        post = self._run_evicting(program, codes, n).astype(np.float64)  # [Q, n]
        suspect = np.isnan(post).any(axis=0) & ~bad
        rows = np.nonzero(suspect)[0]
        if len(rows) > 8:
            _, robust = self._plan(query, ev_vars, _planner.MODE_BATCHED, robust=True, device=device, slot=slot)
            post[:, rows] = robust.run(np.ascontiguousarray(codes[:, rows]), len(rows))
        elif len(rows):
            _, flat = self._plan(query, ev_vars, _planner.MODE_FLAT, device=device, slot=slot)
            for b in rows:
                post[:, b] = flat.run(np.ascontiguousarray(codes[:, b:b + 1]), 1)[:, 0]
        return post

    def _run_evicting(self, program, codes, n):
        """`program.run`, retried once after closing every OTHER cached device object when the device
        is out of memory: each program owns a scratch arena sized for its largest batch (3.9 GB for
        100k rows of the benchmark grid), and a BayesNet caches up to `max_cached_programs` of them --
        many evidence patterns at large batches would otherwise exhaust the GPU long before the LRU
        cap evicts anything (VERDICT r1)."""
        from . import engine

        try:
            return program.run(codes, n)
        except engine.EngineError as exc:
            if exc.code != engine.SBN_E_NOMEM:
                raise
        with self._cache_lock:
            for key in [k for k, v in self._engine_cache.items() if (v[1] if isinstance(v, tuple) else v) is not program]:
                old = self._engine_cache.pop(key)
                (old[1] if isinstance(old, tuple) else old).close()
        return program.run(codes, n)

    def _posterior_codes_multi(self, query, ev_vars, codes, bad, devices):
        """Row-shard `_posterior_codes` over several GPUs of this process: contiguous balanced
        slices (sharding.row_shard), one thread per device."""
        import threading

        from .sharding import row_shard

        n = len(bad)
        world = len(devices)
        # a device listed k times runs k shards at once: each needs a program of its own
        slots = [devices[:r].count(d) for r, d in enumerate(devices)]
        # programs are created up front, on this thread (the cache is not thread-safe)
        for d, s in zip(devices, slots):
            self._plan(query, ev_vars, _planner.MODE_BATCHED, device=d, slot=s)
        plan, _ = self._plan(query, ev_vars, _planner.MODE_BATCHED, device=devices[0])
        post = np.empty((plan.Q, n), dtype=np.float64)
        errors = []

        def work(r):
            sl = row_shard(n, r, world)
            if sl.stop == sl.start:
                return
            try:
                post[:, sl] = self._posterior_codes(query, ev_vars, np.ascontiguousarray(codes[:, sl]), bad[sl],
                                                    device=devices[r], slot=slots[r])
            except Exception as exc:  # surfaced on the calling thread
                errors.append(exc)

        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return post

    # ------------------------------------------------------- joint / likelihood of rows
    def full_joint_dist(self, event: dict = None, keep_zeros=False) -> pd.Series:
        """The normalised product of every CPT (bayes_net.py:398-465), computed on the GPU
        as one exact query over all the variables with no evidence.  Like the reference the
        levels are sorted by name and combinations of probability zero are left out unless
        `keep_zeros`.  Practical for small networks only (the joint has prod(card) rows)."""
        names = sorted(self.nodes)
        plan, program = self._plan(tuple(names), (), _planner.MODE_FLAT)
        post = program.run(np.zeros((0, 1), dtype=np.uint8), 1)[:, 0].astype(np.float64)
        fjd = pd.Series(post, index=self._answer_index(plan), name=f"P({', '.join(map(str, names))})")
        return fjd if keep_zeros else fjd[post > 0]

    def predict_proba(self, X: typing.Union[dict, pd.DataFrame]):
        """Probability of each row of `X` (bayes_net.py:934-962).

        The reference builds the full joint, sums out the columns `X` lacks and looks the
        rows up.  Here P(row) is the normaliser of a variable elimination with the row as
        evidence and no query variable: same number, no joint, any network size.  Rows of
        probability zero give 0.0 (the reference's joint has no such row and raises
        KeyError).  With a single column the reference returns the whole marginal instead
        of per-row values; this returns per-row values in every case."""
        if isinstance(X, dict):
            return self.predict_proba(pd.DataFrame([X])).iloc[0]
        ev_vars = tuple(sorted(X.columns))
        n = len(X.index)
        name = f"P({', '.join(map(str, ev_vars))})"
        if len(ev_vars) == 1:
            index = pd.Index(X[ev_vars[0]], name=ev_vars[0])
        else:
            index = pd.MultiIndex.from_frame(X[list(ev_vars)])
        if n == 0:
            return pd.Series([], index=index, name=name, dtype=np.float64)
        plan, program = self._plan((), ev_vars, _planner.MODE_BATCHED)
        codes, bad = self._encode_events(ev_vars, [X[v].to_numpy() for v in ev_vars])
        prob = program.evidence(codes, n).astype(np.float64)
        rows = np.nonzero(np.isnan(prob) & ~bad)[0]
        if len(rows) > 8:  # below the float32 range (or exactly zero): settle in float64
            _, robust = self._plan((), ev_vars, _planner.MODE_BATCHED, robust=True)
            prob[rows] = robust.evidence(np.ascontiguousarray(codes[:, rows]), len(rows))
        elif len(rows):
            _, flat = self._plan((), ev_vars, _planner.MODE_FLAT)
            for b in rows:
                prob[b] = flat.evidence(np.ascontiguousarray(codes[:, b:b + 1]), 1)[0]
        prob[np.isnan(prob) | bad] = 0.0
        return pd.Series(prob, index=index, name=name)

    def predict_log_proba(self, X: typing.Union[dict, pd.DataFrame]):
        """Log-likelihood of each row (bayes_net.py:964-973)."""
        with np.errstate(divide="ignore"):
            return np.log(self.predict_proba(X))

    def impute(self, sample: dict, **query_params) -> pd.Series:
        """Fill the `None` entries of `sample` with their most probable joint value
        (bayes_net.py:877-908)."""
        known = {k: v for k, v in sample.items() if v is not None}
        unknown = [k for k, v in sample.items() if v is None]
        posterior = self.query(*unknown, event=known, **query_params)
        best = posterior.idxmax()
        if not isinstance(best, tuple):
            best = (best,)
        for k, v in zip(posterior.index.names, best):
            known[k] = v
        return pd.Series(known)
