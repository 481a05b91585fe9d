"""Cost of per-world applied forces on the fused step: human36_contact_262144 stepped with generalized
forces on every dof and a wrench on every body bound, next to the same batch with nothing bound.

Both runs start from the same states (bench.py's seeded initial states) and step the same number of
times; the bound arrays hold zeros, so that both take the same trajectory and the same contact
branches -- the prepare stage reads the arrays and does the arithmetic of the term whatever their
values.  The two configurations alternate, `--repeats` times each; step time = CUDA events around
`--steps` steps after `--warmup` unmeasured ones.

    python profiles/applied_forces_bench.py [--worlds 262144] [--steps 100] [--out FILE]
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
    bw = BatchedWorld(model, W, device="cuda:0")
    gpos0, gvel0 = torch.as_tensor(gp, device=bw.device), torch.as_tensor(gv, device=bw.device)
    nj = len(model.joint_type)
    tau = torch.zeros((model.ndof, W), dtype=torch.float64, device=bw.device)
    wrench = torch.zeros((nj, 6, W), dtype=torch.float64, device=bw.device)
    bodies = list(range(1, nj + 1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run(bound):
        if bound:
            bw.set_applied_forces(gforce=tau, wrench=wrench, bodies=bodies)
        else:
            bw.set_applied_forces(gforce=False, wrench=False)
        bw.gpos.copy_(gpos0)
        bw.gvel.copy_(gvel0)
        bw.cforce.zero_()
        bw.step(DT, a.warmup)
        e0.record()
        bw.step(DT, a.steps)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)/a.steps

    ms = {"unbound": [], "bound": []}
    states = {}
    for _ in range(a.repeats):
        for name in ("unbound", "bound"):
            ms[name].append(run(name == "bound"))
            states[name] = bw.gvel.cpu().numpy()
    res = {
        "workload": "%s_%d" % (scen, W), "steps": a.steps, "warmup": a.warmup, "repeats": a.repeats,
        "gpu": gpu_info(0),
        "bound": "gforce (%d, W) and wrenches on all %d bodies, zeros" % (model.ndof, nj),
        "applied_bytes_per_world_step": 8*(model.ndof + 6*nj),
        "ms_per_step": ms,
        "world_steps_per_s": {k: W/(min(v)*1e-3) for k, v in ms.items()},
        "bound_over_unbound_best": min(ms["bound"])/min(ms["unbound"]),
        "same_final_state": states["bound"].tobytes() == states["unbound"].tobytes(),     # (bitwise: NaN worlds too)
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
