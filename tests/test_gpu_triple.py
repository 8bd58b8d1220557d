"""The two bodies of the fused expanding product + contraction (csrc/sbn_pair.cu) on the benchmark grid:
`sbn_triple_kernel` (default: 32-row blocks staged in shared memory, two rows per thread, packed FFMA2) against
`sbn_triple_kernel_l1` (SOROBN_B200_TRIPLE_KERNEL=0, one row per thread, operands re-read through L1) and against
one launch per step.  The staged body sums in the order of the L1 body, so the two agree bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-6


@pytest.fixture(scope="module")
def grid():
    from sorobn_b200 import planner, workloads

    wl = workloads.grid10x10()
    bn = wl.build()
    net = bn._compiled
    plan = planner.build_plan(net, [net.index[q] for q in wl.query], [net.index[e] for e in wl.evidence])
    return wl, bn, net, plan


def program(plan):
    from sorobn_b200 import engine

    prog = engine.Program(plan)
    prog.set_graph(False)  # plain launches: the body is chosen at every launch
    roles = prog.step_roles()
    assert (roles == 4).sum() == (roles == 5).sum() == 1
    return prog


def run_body(prog, codes, rows, monkeypatch, body):
    if body == "l1":
        monkeypatch.setenv("SOROBN_B200_TRIPLE_KERNEL", "0")
    else:
        monkeypatch.delenv("SOROBN_B200_TRIPLE_KERNEL", raising=False)
    try:
        return prog.run(codes, rows).copy()
    finally:
        monkeypatch.delenv("SOROBN_B200_TRIPLE_KERNEL", raising=False)


# 7: fewer rows than one 32-row block (and an odd last row pair); 257, 5003: ragged last blocks; 100,000: the benchmark
@pytest.mark.parametrize("rows", [7, 257, 5003, 100_000])
def test_staged_body_matches_the_l1_body_and_one_launch_per_step(grid, rows, monkeypatch):
    wl, bn, _, plan = grid
    codes = wl.codes(bn, rows, seed=37)
    prog = program(plan)
    staged = run_body(prog, codes, rows, monkeypatch, "staged")
    assert np.array_equal(staged, run_body(prog, codes, rows, monkeypatch, "staged"))  # deterministic
    l1 = run_body(prog, codes, rows, monkeypatch, "l1")
    assert np.isfinite(staged).all()
    assert np.array_equal(staged, l1)
    prog.set_tiled(10)
    single = prog.run(codes, rows).copy()
    prog.set_tiled(11)
    assert np.isfinite(single).all()
    assert np.allclose(staged, single, rtol=3e-6, atol=1e-30)
    prog.set_graph(True)
    for _ in range(2):  # capture, then replay
        assert np.array_equal(prog.run(codes, rows), staged)


def test_staged_body_matches_the_oracle(grid, monkeypatch):
    from oracle import ve_oracle

    wl, bn, net, plan = grid
    rows = 5003
    codes = wl.codes(bn, rows, seed=41)
    staged = run_body(program(plan), codes, rows, monkeypatch, "staged")
    dn = ve_oracle.dense_from_pandas(bn.P, bn.parents, bn.nodes)
    order = [net.names[v] for v in plan.order]
    for b in (0, 31, 32, rows // 2, rows - 1):  # both ends of a row block, and the ragged last one
        ev = {v: net.domains[net.index[v]][codes[i, b]] for i, v in enumerate(wl.evidence)}
        want = ve_oracle.query(dn, *wl.query, event=ev, order=order)[1].reshape(-1).astype(np.float64)
        got = staged[:, b].astype(np.float64)
        assert np.max(np.abs(got - want) / want) < RTOL, (b, got, want)


def test_the_switch_selects_the_body_that_runs(grid, monkeypatch):
    """Kernel names as the CUDA profiler sees them: the default launches the staged body, the switch the L1 body."""
    import torch

    wl, bn, _, plan = grid
    rows = 257
    codes = wl.codes(bn, rows, seed=43)
    prog = program(plan)
    for body, want, other in (("staged", "sbn_triple_kernel(", "sbn_triple_kernel_l1"),
                              ("l1", "sbn_triple_kernel_l1", "sbn_triple_kernel(")):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            run_body(prog, codes, rows, monkeypatch, body)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages()]
        assert any(want in n for n in names), (body, names)
        assert not any(other in n for n in names), (body, names)
