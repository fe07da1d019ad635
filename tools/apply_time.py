"""Exact-mode nhood step at configs[1] (1M spots, 30 clusters, P permutations) for several replay variants: per-kernel-class
CUDA-event times.  usage: python tools/apply_time.py [P] [algo:threads:r[:key=value...]] ..."""
import sys

import numpy as np

sys.path.insert(0, ".")
import squidpy_b200 as sq  # noqa: E402
from squidpy_b200._rng import spawn_states  # noqa: E402
from squidpy_b200.gr import NhoodPlan  # noqa: E402
from tools import synth  # noqa: E402

P = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
variants = sys.argv[2:] or ["-1:1024:2", "7:1024:4"]
ctx = sq.default_context(0)
g = synth.hex_graph(1000, 1000)
base = synth.categorical_labels(g.shape[0], 30, seed=0).cat.codes.to_numpy().astype(np.uint32)
ref = None
for v in variants:
    parts = v.split(":")
    plan = NhoodPlan(g.indptr, g.indices, 30, ctx)
    plan.set_option("shuffle_algo", int(parts[0]))
    if int(parts[0]) >= 0:
        plan.set_option("shuffle_threads", int(parts[1]))
        plan.set_option("shuffle_r", int(parts[2]))
    for kv in parts[3:]:
        k, x = kv.split("=")
        plan.set_option(k, int(x))
    plan.set_base(base)
    plan.upload(spawn_states(0, P))
    plan.run_async()
    ctx.sync()
    ctx.profile(True)
    ctx.profile_reset()
    plan.run_async()
    ctx.sync()
    kms = {k: round(ctx.profile_get(k)[0], 3) for k in ("fill", "misc", "shuffle", "transpose", "count")}
    ctx.profile(False)
    got = plan.download()
    if ref is None:
        ref = got
    print(v, P, kms, "total %.3f ms" % sum(kms.values()), "equal" if np.array_equal(ref, got) else "DIFFERENT", flush=True)
    plan.close()
