"""Pin the CPU oracle (oracle/ve_oracle.py) against the reference.

The golden vectors were produced by the real reference (oracle/gen_golden.py); the
hand-written values below are the reference's own doctest outputs
(/root/reference/sorobn/bayes_net.py and examples.py)."""
import numpy as np
import pytest

from conftest import build_network, case_event, dense_answer, golden_names, load_golden
from oracle import ve_oracle


def oracle_net(bn):
    return ve_oracle.dense_from_pandas(bn.P, bn.parents, bn.nodes)


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference_goldens(name):
    golden = load_golden(name)
    bn = build_network(golden)
    net = oracle_net(bn)
    worst = 0.0
    for case in golden["cases"]:
        vars_, values, support = ve_oracle.query(net, *case["query"], event=case_event(case))
        assert list(vars_) == case["names"]
        want = dense_answer(case, net.domains)
        # same support: the reference drops exactly the zero-posterior rows
        assert np.array_equal(support, want > 0), case
        err = np.max(np.abs(values - want) / np.maximum(want, 1e-300) * (want > 0))
        worst = max(worst, err)
    assert worst < 1e-12, worst


def test_aima_figure_14_10_product_and_sum_out():
    # doctest of pointwise_mul_two / sum_out, bayes_net.py:62-97 and :114-140
    a = ve_oracle.Factor(("A", "B"), np.array([[0.1, 0.9], [0.7, 0.3]]))  # states sorted F, T
    b = ve_oracle.Factor(("B", "C"), np.array([[0.4, 0.6], [0.8, 0.2]]))
    ab = ve_oracle.pointwise_mul_two(a, b)
    assert ab.vars == ("A", "B", "C")
    # (A=T, B=T, C=T) = .3 * .2
    assert np.isclose(ab.values[1, 1, 1], 0.06)
    assert np.isclose(ab.values[1, 0, 0], 0.28)
    assert np.isclose(ab.values[0, 1, 0], 0.72)
    s = ve_oracle.sum_out(ab, "B")
    assert s.vars == ("A", "C")
    assert np.allclose(s.values, [[0.76, 0.24], [0.52, 0.48]])


def test_disjoint_product_is_outer():
    # bayes_net.py:145-179
    a = ve_oracle.Factor(("A",), np.array([0.7, 0.3]))
    b = ve_oracle.Factor(("B",), np.array([0.8, 0.2]))
    ab = ve_oracle.pointwise_mul_two(a, b)
    assert np.allclose(ab.values, np.outer([0.7, 0.3], [0.8, 0.2]))


def test_reference_doctest_values():
    from sorobn_b200 import examples

    # bayes_net.py:751-755
    net = oracle_net(examples.sprinkler())
    _, v, _ = ve_oracle.query(net, "Rain", event={"Sprinkler": True})
    assert np.allclose(v, [0.7, 0.3])
    # bayes_net.py:829-836
    net = oracle_net(examples.asia())
    vars_, v, _ = ve_oracle.query(net, "Lung cancer", "Tuberculosis", event={"Visit to Asia": True, "Smoker": True})
    assert vars_ == ("Lung cancer", "Tuberculosis")
    assert np.allclose(v, [[0.855, 0.045], [0.095, 0.005]])
    # examples.py:21-27
    net = oracle_net(examples.alarm())
    _, v, _ = ve_oracle.query(net, "John calls", "Mary calls", event={"Burglary": True, "Earthquake": False})
    assert np.allclose(v, [[0.08463, 0.06637], [0.25677, 0.59223]])
    # examples.py:268-274
    net = oracle_net(examples.grades())
    _, v, _ = ve_oracle.query(net, "Letter", "SAT", event={"Intelligence": "Smart"})
    assert np.allclose(v, [[0.153544, 0.614176], [0.046456, 0.185824]], atol=1e-6)


def test_elimination_order_does_not_matter():
    from sorobn_b200 import examples

    net = oracle_net(examples.asia())
    hidden_orders = [
        ["Tuberculosis", "Lung cancer", "Bronchitis", "TB or cancer", "Smoker"],
        ["Smoker", "TB or cancer", "Bronchitis", "Lung cancer", "Tuberculosis"],
    ]
    ev = {"Visit to Asia": True, "Positive X-ray": True}
    base = ve_oracle.query(net, "Dispnea", event=ev)[1]
    for order in hidden_orders:
        assert np.allclose(ve_oracle.query(net, "Dispnea", event=ev, order=order)[1], base, rtol=1e-13)
    # and equals brute force over the full joint (bayes_net.py:398-465)
    _, bf = ve_oracle.brute_force_query(net, ("Dispnea",), ev)
    assert np.allclose(bf, base, rtol=1e-12)


def test_query_argument_errors():
    from sorobn_b200 import examples

    net = oracle_net(examples.alarm())
    with pytest.raises(ValueError):
        ve_oracle.query(net, event={})
    with pytest.raises(ValueError):
        ve_oracle.query(net, "Alarm", event={"Alarm": True})


@pytest.mark.parametrize("name", golden_names(kinds=("predict_proba",)))
def test_evidence_probability_matches_reference_predict_proba(name):
    """`predict_proba` of the REAL reference (bayes_net.py:934-962: full joint, marginalised and
    looked up) against the oracle's P(event) and against a brute-force sum over the joint."""
    from sorobn_b200 import examples

    golden = load_golden(name)
    bn = examples.build(examples.NETWORKS[golden["network"]])
    net = oracle_net(bn)
    joint = ve_oracle.full_joint(net)
    for case in golden["cases"]:
        cols = case["columns"]
        for row, want in zip(case["rows"], case["prob"]):
            ev = dict(zip(cols, row))
            got = ve_oracle.evidence_probability(net, ev)
            assert abs(got - want) <= 1e-12 * max(want, 1e-300), (ev, got, want)
            idx = tuple(net.domains[v].index(ev[v]) if v in ev else slice(None) for v in joint.vars)
            assert abs(joint.values[idx].sum() - want) <= 1e-12


def _example(name):
    from sorobn_b200 import examples

    return examples.build(examples.NETWORKS[name])


@pytest.mark.parametrize("name", golden_names(("impute",)))
def test_oracle_impute_matches_reference(name):
    """`impute` (bayes_net.py:877-908) on 25 partial samples per example network (2-3 missing
    variables; with one the reference itself fails, see oracle/gen_golden.py)."""
    golden = load_golden(name)
    net = oracle_net(_example(golden["network"]))
    for case in golden["cases"]:
        sample = {k: v for k, v in case["sample"]}
        want = {k: v for k, v in case["filled"]}
        assert ve_oracle.impute(net, sample) == want, case


@pytest.mark.parametrize("name", golden_names(("gibbs_conditionals",)))
def test_oracle_gibbs_conditionals_match_reference(name):
    """The deterministic half of `_gibbs_sampling`: P(var | Markov boundary) for every variable
    (bayes_net.py:699-712), entry by entry, including which configurations the reference drops."""
    golden = load_golden(name)
    net = oracle_net(_example(golden["network"]))
    for node, g in golden["nodes"].items():
        boundary, table = ve_oracle.gibbs_conditional(net, node)
        assert boundary == g["boundary"], (node, boundary, g["boundary"])
        pos = [{v: i for i, v in enumerate(net.domains[u])} for u in [*boundary, node]]
        seen = np.zeros(table.shape, dtype=bool)
        for key, want in zip(g["index"], g["values"]):
            idx = tuple(pos[i][k] for i, k in enumerate(key))
            seen[idx] = True
            assert abs(table[idx] - want) <= 1e-12 * max(want, 1e-300), (node, key, table[idx], want)
        # what the reference leaves out is exactly what is zero (or undefined: 0/0) here
        rest = table[~seen]
        assert np.all((rest == 0) | np.isnan(rest)), (node, rest)


def test_reference_copy_driven_in_min_fill_order_matches_the_oracle():
    """The reference's own operators driven through oracle/ref_driver.ordered_query in min-fill
    order -- what bench.py's CPU legs time -- give the oracle's posterior.  Their answers are
    stored in tests/golden/ordered_grid4x4s3.json (oracle/gen_golden.py); where `oracle/_ref`
    (the reference itself, copied by oracle/build_ref.py) is present, the live run must still
    reproduce them."""
    import warnings

    from conftest import spec_digest
    from oracle import build_ref, ref_driver
    from sorobn_b200 import BayesNet, synthetic

    golden = load_golden("ordered_grid4x4s3")
    spec = synthetic.grid(**golden["kwargs"])
    assert spec_digest(spec) == golden["digest"], "synthetic generator drifted: regenerate tests/golden"
    dn = oracle_net(synthetic.load(spec, BayesNet))
    for case in golden["cases"]:
        query, event = case["query"], case_event(case)
        want = ve_oracle.query(dn, *query, event=event)[1]
        assert np.allclose(dense_answer(case, dn.domains), want, rtol=1e-12, atol=0), case
    if build_ref.available():
        ref = build_ref.import_reference()
        theirs = synthetic.load(spec, ref.BayesNet)
        for case in golden["cases"]:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                got = ref_driver.ordered_query(ref, theirs, case["query"], case_event(case), golden["order"])
            assert np.allclose(got.to_numpy(), case["values"], rtol=1e-12, atol=0), case
