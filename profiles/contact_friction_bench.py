"""Cost of per-world contact friction on the fused step: human36_contact_262144 stepped with the friction
coefficient of all 8 contacts bound (the model's own 0.6 in every world), next to the same batch with
nothing bound.

Both runs start from the same states (bench.py's seeded initial states) and step the same number of
times.  The configurations alternate, `--repeats` times each; step time = CUDA events around
`--steps` steps after `--warmup` unmeasured ones.  Each is run with the default sort_period 2 (worlds
re-sorted by their contact state every other step, so mu is gathered through the permutation) and
with sort_period 0 (identity assignment).  The bound values are the model's, so the bound and unbound
states must agree bit for bit; the result records whether they do.

    python profiles/contact_friction_bench.py [--worlds 262144] [--steps 100] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "arboris-python_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

DT = 1e-3


def gpu_info(index):
    import torch
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in out.stdout.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(clk))
    except Exception as e:     # the timing stands without it, but says so
        info["power_limit_w"] = "unavailable (%s)" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=262144)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out")
    a = ap.parse_args()
    import numpy as np
    import torch
    from arboris_b200 import scenarios
    from arboris_b200.batch import BatchedWorld
    from arboris_b200.flatten import flatten

    scen = "human36_contact"
    model = flatten(scenarios.BUILDERS[scen]())
    W = a.worlds
    gp, gv = scenarios.initial_states(model, scen, 0, W)
    bws = {0: BatchedWorld(model, W, device="cuda:0"), 2: BatchedWorld(model, W, device="cuda:0")}
    bws[0].set_option("sort_period", 0)
    bws[2].set_option("sort_period", 2)
    dev = bws[2].device
    gpos0, gvel0 = torch.as_tensor(gp, device=dev), torch.as_tensor(gv, device=dev)
    cons = bws[2].contact_indices()
    mu0 = [float(model.cons_dbl[c][36]) for c in cons]
    mu = torch.as_tensor(np.repeat(np.array(mu0)[:, None], W, 1), device=dev).contiguous()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run(sort, bound):
        bw = bws[sort]
        bw.set_contact_friction(mu, cons) if bound else bw.set_contact_friction(False)
        bw.gpos.copy_(gpos0)
        bw.gvel.copy_(gvel0)
        bw.cforce.zero_()
        bw.step(DT, a.warmup)
        e0.record()
        bw.step(DT, a.steps)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)/a.steps

    names = {(2, False): "unbound", (2, True): "bound", (0, False): "unbound_sort0", (0, True): "bound_sort0"}
    ms = {v: [] for v in names.values()}
    states = {}
    for _ in range(a.repeats):
        for (sort, bound), name in names.items():
            ms[name].append(run(sort, bound))
            states[name] = [x.cpu().numpy() for x in (bws[sort].gpos, bws[sort].gvel, bws[sort].cforce)]
    best = {k: min(v) for k, v in ms.items()}
    res = {
        "workload": "%s_%d" % (scen, W), "steps": a.steps, "warmup": a.warmup, "repeats": a.repeats,
        "gpu": gpu_info(0),
        "bound": "mu (%d, W) of all contacts, the model's own values %s" % (len(cons), sorted(set(mu0))),
        "ms_per_step": ms,
        "world_steps_per_s": {k: W/(v*1e-3) for k, v in best.items()},
        "bound_over_unbound_best": best["bound"]/best["unbound"],
        "bound_over_unbound_best_sort0": best["bound_sort0"]/best["unbound_sort0"],
        "bits_equal_bound_vs_unbound": all(x.tobytes() == y.tobytes() for x, y in zip(states["bound"], states["unbound"])),
        "bits_equal_bound_vs_unbound_sort0": all(x.tobytes() == y.tobytes()
                                                 for x, y in zip(states["bound_sort0"], states["unbound_sort0"])),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
