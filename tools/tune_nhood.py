"""GPU tuning sweep for the nhood permutation pipeline (1M spots, 30 clusters, P permutations): per-kernel-class CUDA
event times for shuffle variants, plus a host-side breakdown of the public API call.  Output: gpurun_out/tune_nhood.json"""
from __future__ import annotations

import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import squidpy_b200 as sq  # noqa: E402
from squidpy_b200._rng import spawn_states  # noqa: E402
from squidpy_b200.gr import NhoodPlan  # noqa: E402
from tools import synth  # noqa: E402


def main():
    P = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
    ctx = sq.default_context(0)
    g = synth.hex_graph(1000, 1000)
    labels = synth.categorical_labels(g.shape[0], 30, seed=0)
    base = labels.cat.codes.to_numpy().astype(np.uint32)
    plan = NhoodPlan(g.indptr, g.indices, 30, ctx)
    plan.set_base(base)
    st = spawn_states(0, P)
    plan.upload(st)
    plan.run_async()
    ctx.sync()
    ref_counts = plan.download()
    results = []
    ctx.profile(True)
    variants = []
    base = dict(shuffle_algo=1, shuffle_threads=512, shuffle_r=4, shuffle_ctas=0, shuffle_wfactor_x100=400, shuffle_q=4, shuffle_low=0, shuffle_stagger_us=0)
    # the default (auto) next to every replay variant at its best measured shape (edit this list for a focused sweep;
    # profiles/r01_tune_nhood.json holds the last run)
    variants.append({**base, "shuffle_algo": -1})
    a7 = {**base, "shuffle_algo": 7, "shuffle_threads": 1024, "shuffle_r": 2, "shuffle_low": 98304}
    for low in (0, 65536):
        variants.append({**a7, "shuffle_low": low})
    variants.append({**a7, "shuffle_low": 65536, "shuffle_q": 8})
    variants.append({**a7, "shuffle_low": 65536, "shuffle_q": 2})
    variants.append({**a7, "shuffle_r": 4, "shuffle_low": 0})
    variants.append({**base, "shuffle_algo": 2})
    variants.append({**base, "shuffle_algo": 1, "shuffle_threads": 1024, "shuffle_ctas": 148})
    variants.append({**base, "shuffle_algo": -1, "count_sym": 0})
    for v in variants:
        for k, val in v.items():
            plan.set_option(k, val)
        best = None
        for rep in range(2):
            ctx.profile_reset()
            plan.run_async()
            ctx.sync()
            kms = {k: ctx.profile_get(k)[0] for k in ("fill", "shuffle", "transpose", "count", "misc")}
            if best is None or kms["shuffle"] < best["shuffle"]:
                best = kms
        ok = bool((plan.download() == ref_counts).all())
        results.append({**v, **best, "ok": ok})
        print(json.dumps(results[-1]), flush=True)
    ctx.profile(False)
    plan.close()

    # host-side breakdown of the public API (one call = what a user pays)
    ad = synth.make_adata(np.zeros((g.shape[0], 2)), g, labels)
    from squidpy_b200.gr import _nhood as nh
    from squidpy_b200.gr._utils import category_codes

    tb = {}
    t = time.perf_counter(); codes, n_cls = category_codes(ad.obs["cluster"], dtype=np.uint32); tb["category_codes"] = time.perf_counter() - t
    t = time.perf_counter(); plan = NhoodPlan(g.indptr, g.indices, 30, ctx); tb["plan_create(H2D CSR)"] = time.perf_counter() - t
    t = time.perf_counter(); plan.count(codes); tb["count"] = time.perf_counter() - t
    t = time.perf_counter(); plan.set_base(codes); tb["set_base"] = time.perf_counter() - t
    t = time.perf_counter(); st = spawn_states(0, P); tb["spawn_states"] = time.perf_counter() - t
    t = time.perf_counter(); plan.upload(st); tb["upload(+alloc)"] = time.perf_counter() - t
    t = time.perf_counter(); plan.run_async(); ctx.sync(); tb["run"] = time.perf_counter() - t
    t = time.perf_counter(); perms = plan.download(); tb["download"] = time.perf_counter() - t
    t = time.perf_counter(); pf = perms.astype(np.float64); z = (ref_counts[0] - pf.mean(axis=0)) / pf.std(axis=0); tb["zscore_host"] = time.perf_counter() - t
    t = time.perf_counter(); plan.close(); tb["close(free)"] = time.perf_counter() - t
    t = time.perf_counter(); sq.gr.nhood_enrichment(ad, "cluster", n_perms=P, seed=0, copy=True); tb["api_total"] = time.perf_counter() - t
    print(json.dumps({"api_breakdown_s": tb}), flush=True)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump({"variants": results, "api_breakdown_s": tb}, open(os.path.join(ROOT, "gpurun_out", "tune_nhood.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
