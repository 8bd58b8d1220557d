"""A/B of the two bodies of the fused expanding product + contraction (csrc/sbn_pair.cu: `sbn_triple_kernel`, staged
in shared memory, against `sbn_triple_kernel_l1`, selected with SOROBN_B200_TRIPLE_KERNEL=0) on ONE program: the
triple launch's CUDA-event time from the per-step profile of whole runs (plain launches), the two bodies alternating,
a 256 MB write (L2 flush) before every run.  Prints per body the median / min / max launch time, the achieved rate on
the launch's algorithmic bytes (A, B, C read once, the output written once), and the largest relative difference of
the posteriors between the bodies.
   python tools/triple_ab.py [workload] [rows] [runs]          (default: grid10x10 100000 30)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sorobn_b200 import engine, planner, workloads  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "grid10x10"
rows = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
runs = int(sys.argv[3]) if len(sys.argv) > 3 else 30
wl = workloads.WORKLOADS[name]()
bn = wl.build()
net = bn._compiled
plan = planner.build_plan(net, [net.index[q] for q in wl.query], [net.index[e] for e in wl.evidence])
prog = engine.Program(plan)
prog.set_graph(False)
prog.reserve(rows)
roles = prog.step_roles()
firsts = np.flatnonzero(roles == 4)
if len(firsts) != 1:
    sys.exit(f"{name}: {len(firsts)} fused expanding products, this script times exactly one")
i1 = int(firsts[0])
i2 = int(np.flatnonzero(roles == 5)[0])


def entries(f):
    return int(np.prod([net.card[v] for v in f.vars], dtype=np.int64))


s1, s2 = plan.steps[i1], plan.steps[i2]
bytes_per_row = 4 * (sum(entries(f) for f, _, _ in s1.inputs if f.batched)
                     + sum(entries(f) for f, _, _ in s2.inputs if f.batched and f.buf != s1.out_slot)
                     + int(np.prod(s2.cards, dtype=np.int64)))

codes = wl.codes(bn, rows, seed=1000)
d_ev = torch.from_numpy(np.ascontiguousarray(codes)).cuda()
d_out = torch.empty((prog.Q, rows), dtype=torch.float32, device="cuda")
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
stream = torch.cuda.current_stream().cuda_stream
bodies = (("staged", "1"), ("l1", "0"))


def run(value):
    os.environ["SOROBN_B200_TRIPLE_KERNEL"] = value
    flush.fill_(1)
    torch.cuda.synchronize()
    ms = prog.profile(d_ev.data_ptr(), rows, rows, d_out.data_ptr(), rows, stream)
    return float(ms[i1]) * 1e3  # us


for _ in range(3):
    for _, value in bodies:
        run(value)
times = {label: [] for label, _ in bodies}
out = {}
for _ in range(runs):
    for label, value in bodies:
        times[label].append(run(value))
for label, value in bodies:
    run(value)
    out[label] = d_out.cpu().numpy().copy()

print(f"{name} rows={rows} runs={runs} triple = steps {i1} + {i2}, {bytes_per_row} B/row algorithmic, "
      f"stages={os.environ.get('SOROBN_B200_TRIPLE_STAGES', 'default')}")
for label, _ in bodies:
    t = np.array(times[label])
    med = float(np.median(t))
    print(f"  {label:7s} median {med:7.1f} us  min {t.min():7.1f}  max {t.max():7.1f}  "
          f"{bytes_per_row * rows / (med * 1e-6) / 1e9:7.0f} GB/s")
a, b = out["staged"], out["l1"]
rel = np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b.astype(np.float64)), 1e-30)
print(f"  posteriors: max rel diff staged vs l1 {float(np.nanmax(rel)):.3g}, "
      f"bitwise equal {bool(np.array_equal(a, b, equal_nan=True))}, "
      f"finite {bool(np.isfinite(a).all())}")
