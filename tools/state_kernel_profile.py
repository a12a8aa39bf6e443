"""Per-launch durations of the fused NUTS state kernel (`nuts_state_kernel`) over one timed step of a GLM workload,
in tick order, labelled by what each tick closes.

    python tools/state_kernel_profile.py [--workload c4] [--warmup 3] [--out profiles/state_kernel_ticks.json]

The setup is bench.py's (same model, chains in the typical set, adapted step sizes, same seed and iteration offsets);
the step is then run once under torch.profiler with CUDA activities.  Launch order of the fused loop (one
b2m_nuts_run call): tick 0 is one launch (tick + pack), tick t > 0 one launch (finish + tick + pack), except every
8th tick, which is two (finish alone, then tick + pack).  Tick t >= 1 completes leaf t - 1, so with the tree depth of
every transition known, the tick that completes the last leaf of a doubling is a "doubling" tick, the one that
completes the last leaf of a transition a "transition" tick, the rest "plain"; ticks after the last leaf are "idle".
The labels follow the most common depth of each transition: exact when every chain has that depth (reported as
`lockstep_fraction`), approximate otherwise.
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402

KCHECK = 8   # ticks between the drains of the fused loop (glm_nuts_run_fused)


def leaf_types(modal_depths):
    """what completing each leaf of the call closes: 'plain', 'doubling' or 'transition'"""
    out = []
    for d in modal_depths:
        for j in range(d):
            out += ["plain"] * ((1 << j) - 1) + ["transition" if j == d - 1 else "doubling"]
    return out


def label_launches(n_launches, types):
    labels, tick = [], 0
    while len(labels) < n_launches:
        if tick == 0:
            labels.append((0, "tick", "start"))
        else:
            if tick % KCHECK == 0:
                labels.append((tick, "finish", "finish"))
            labels.append((tick, "tick", types[tick - 1] if tick - 1 < len(types) else "idle"))
        tick += 1
    return labels[:n_launches]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4", choices=[k for k, w in bench.WORKLOADS.items() if w["kind"] == "glm"])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "state_kernel_ticks.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    import mlx_mcmc_b200 as B
    from mlx_mcmc_b200 import _cabi
    from mlx_mcmc_b200.engine import launch_nuts

    wl = bench.WORKLOADS[args.workload]
    C, MD, ITERS, seed = wl["chains"], wl["max_tree_depth"], wl["iters"], 1234
    _, _, model, st, _ = bench.glm_setup(torch, B, wl, C, 0, seed)
    draws = torch.empty((ITERS, C, wl["d"]), dtype=torch.float32, device="cuda")
    depths = torch.empty((ITERS, C), dtype=torch.int32, device="cuda")
    it0 = [wl["adapt_iters"]]

    def one_step():
        launch_nuts(st, ITERS, MD, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, seed, it0[0], draws=draws, depths=depths)
        it0[0] += ITERS

    for _ in range(max(args.warmup, 1)):
        one_step()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        one_step()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kern = sorted((e for e in events if e.get("cat") == "kernel" and "nuts_state_kernel" in e.get("name", "")),
                  key=lambda e: e["ts"])
    dep = depths.cpu().numpy()
    modal = [int(np.bincount(row).argmax()) for row in dep]
    lockstep = float((dep == np.asarray(modal)[:, None]).all(0).mean())
    labels = label_launches(len(kern), leaf_types(modal))
    launches = [{"tick": t, "kind": k, "type": ty, "us": float(e["dur"])} for (t, k, ty), e in zip(labels, kern)]
    summary = {}
    for ty in ("start", "plain", "doubling", "transition", "finish", "idle"):
        us = [x["us"] for x in launches if x["type"] == ty]
        if us:
            summary[ty] = {"launches": len(us), "mean_us": float(np.mean(us)), "median_us": float(np.median(us)),
                           "max_us": float(np.max(us)), "total_ms": float(np.sum(us)) / 1e3}
    props = torch.cuda.get_device_properties(0)
    out = {"workload": args.workload, "device": props.name, "chains": C, "transitions": ITERS,
           "modal_depths": modal, "lockstep_fraction": lockstep, "launches_total": len(kern),
           "state_kernel_ms_total": float(sum(x["us"] for x in launches)) / 1e3, "by_type": summary, "launches": launches}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "launches"}))


if __name__ == "__main__":
    main()
