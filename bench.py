#!/usr/bin/env python
"""Benchmark of the batched Arboris step (BASELINE.json metric: world-steps/s,
human36, fp64, dt = 1 ms).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # ... and the state after the last timed step

A "step" is one pass of the hot path (update_dynamic -> update_controllers ->
update_constraints -> integrate) over the whole batch of worlds.  Prints ONE JSON
line (rank 0).  Under torchrun (N > 1) the worlds are sharded over the ranks with
no data-path collective; NCCL only carries the timing/diagnostics reduction.

Headline (`value`, `e2e`): weak scaling -- every GPU steps the workload's 262 144
worlds.  At N > 1 the same line also carries `"strong"`: BASELINE.json configs[4]
read literally (262 144 worlds IN TOTAL, split over the N GPUs), measured in the
same run with the same protocol.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "arboris-python_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

DT = 1e-3
STATE_BYTES_PER_WORLD_STEP = 1504   # read+write of 94 doubles (SURVEY.md 8(d))
WORKLOADS = {
    # BASELINE.json configs[4] (the configuration the metric's "1/2/4/8 B200" sweep is quoted on)
    "human36_contact_262144": ("human36_contact", 262144),
    # BASELINE.json configs[1]
    "human36_free_4096": ("human36_free", 4096),
    "human36_contact_16384": ("human36_contact", 16384),
}
EPISODE = 250      # steps after which a world is re-initialised (the uncontrolled humanoid
                   # collapses and the reference's own sliding solve diverges after ~0.35 s)
GROUPS = 10        # the batch is split into GROUPS contiguous blocks whose episodes are staggered
PHASE = EPISODE//GROUPS   # by PHASE steps, so that at ANY step the batch holds every age of the
                   # episode (free fall, first contacts, 8 contacts with ~20 % sliding) in equal
                   # shares: the measured rate does not depend on which steps are timed
DUMP_BYTES = 32 << 20      # --dump-outputs: at most this many bytes of arrays (well under 64 MB)


# ---------------------------------------------------------------------------------------
# SURVEY.md section 8(d): algorithmic flops per world-step (1 FMA = 2 flop), the "primary
# (structure-exploiting) count" of the assembled-matrix algorithm, evaluated on the ACTUAL active
# sets of the batch instead of assuming every constraint active.
# ---------------------------------------------------------------------------------------
def flop_free(model):
    """W_free = sum_b(216 k_b + 2900) + sum_b(24 k_b^2 + 222 k_b) + 2 n^3 + 4 n^2."""
    n = int(model.ndof)
    kb = [len(a) for a in model.ancestors_dofs()[1:]]
    return float(sum(216*k + 2900 for k in kb) + sum(24*k*k + 222*k for k in kb) + 2*n**3 + 4*n*n)


def flop_contact_increment(model, active):
    """Contact increment of SURVEY.md 8(d) for an (W, nc) array of active flags:
    Jacobians sum_c(2*72 n + 12 d_c n + d_c n), Delassus 2 L n^2 + 2 L^2 n, rhs 4 n^2 + 2 L n,
    Gauss-Seidel 20 sum_c(30 d_c^3 + 2 d_c^2 + 2 L d_c); zero for a world without active constraint.
    Returns the per-world flop counts (W,)."""
    n = float(model.ndof)
    d = np.array([(1, 3, 4)[int(t)] for t in model.cons_type], dtype=float)      # rows per constraint
    a = np.asarray(active, dtype=float)
    L = a @ d
    jac = a @ (2*72*n + 12*d*n + d*n)
    gs = 20.*(a @ (30*d**3 + 2*d**2) + 2*L*(a @ d))
    inc = jac + 2*L*n*n + 2*L*L*n + 4*n*n + 2*L*n + gs
    return np.where(a.sum(1) > 0, inc, 0.)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="human36_contact_262144", choices=sorted(WORKLOADS))
    ap.add_argument("--worlds", type=int, default=0, help="override the workload's number of worlds")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="which reading is the headline `value`: weak (default) = every GPU steps the "
                         "workload's number of worlds; strong = they are split over the GPUs.  At N > 1 the "
                         "other reading is measured too and printed under its own key")
    ap.add_argument("--no-other-scaling", action="store_true", help="N > 1: headline reading only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-sample", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.)
    ap.add_argument("--e2e-chunks", type=lambda t: t if t == "auto" else ([int(x) for x in t.split(",")] if "," in t else int(t)),
                    default="auto",
                    help="column blocks of the end-to-end pass: 'auto' (by batch size, HostPipeline.auto_chunks), a "
                         "number of equal blocks or their relative sizes (a,b,c,...)")
    ap.add_argument("--e2e-mode", default="serial", choices=["serial", "streams"],
                    help="HostPipeline mode: 'serial' = the kernels of all blocks on --e2e-compute-streams "
                         "streams, block after block, copies on two more streams; 'streams' = one stream per block")
    ap.add_argument("--e2e-compute-streams", type=lambda t: t if t == "priority" else int(t), default="priority",
                    help="serial mode: 'priority' = one compute stream per block, earlier blocks at higher "
                         "priority (default); N = N plain streams")
    ap.add_argument("--opt", action="append", help="arb_batch_set_option switch, name=value (A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the state they leave (gpos, gvel, cforce) of a fixed, "
                         "seeded sample of rank 0's worlds to DIR/<name>.npy (float64, %d MB of arrays at "
                         "most), with the sampled world indices in DIR/world.npy; worlds whose state is not "
                         "finite are left out of the sample and listed in DIR/nonfinite_world.npy"
                         % (DUMP_BYTES >> 20))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def config_of(a, scen, total, per_gpu, world_size, scaling, model=None):
    """The `config` object; the reference arm prints the same keys."""
    return {"workload": a.workload, "scenario": scen, "worlds_total": int(total),
            "worlds_per_gpu": int(per_gpu), "distinct_worlds": int(total), "dt": DT,
            "constraints": int(model.nc) if model is not None else None,
            "initial_states": "every world its own seed: numpy default_rng(20260000 + w); SURVEY.md 8(d) "
                              "config 3 distribution (root lift U(0, 0.05) m, tilt U(-.05, .05)^3 rad, joint "
                              "angles U(-.1, .1) rad, zero velocity)" if scen == "human36_contact" else
                              "every world its own seed: numpy default_rng(20260000 + w); SURVEY.md 8(d) config 2",
            "episode_steps": EPISODE, "episode_groups": GROUPS,
            "episodes": "worlds restart from their seeded state every %d steps; %d blocks of "
                        "the batch are staggered by %d steps so every timed step sees the "
                        "whole episode's mix of contact states" % (EPISODE, GROUPS, PHASE),
            "l2": "state of all worlds (%.0f MB) and per-world scratch exceed L2; no flush needed"
                  % (per_gpu*STATE_BYTES_PER_WORLD_STEP/2/1e6),
            "parallelism": "worlds sharded over %d GPU(s) (%s scaling: %s), no collective on the "
                           "step path" % (world_size, scaling,
                                          "every GPU holds the workload's number of worlds"
                                          if scaling == "weak" else
                                          "the workload's worlds are split over the GPUs")}


# ---------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference on the host cores (multiprocessing)
# ---------------------------------------------------------------------------------------
def _cpu_worker(args):
    scen, wid, seconds = args
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    from arboris_b200 import scenarios
    from arboris_b200.flatten import flatten
    from oracle.arboris_oracle import OracleWorld
    model = flatten(scenarios.BUILDERS[scen]())
    o = OracleWorld(model.to_dict())
    o.gpos[:], o.gvel[:] = scenarios.initial_state(model, scen, wid)
    o.step(DT)                                   # warm-up (imports, caches)
    o.gpos[:], o.gvel[:] = scenarios.initial_state(model, scen, wid)
    o.cforce[:] = 0.
    # one whole episode from the reset state = the age mix the GPU batch holds at any step
    n, t0 = 0, time.perf_counter()
    while n < EPISODE and time.perf_counter() - t0 < seconds:
        o.step(DT)
        n += 1
    return n, time.perf_counter() - t0


def cpu_baseline(scen, seconds):
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(scen, w, seconds) for w in range(cores)])
    steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    nmin = min(r[0] for r in res)
    return {"value": steps/wall, "unit": "world-steps/s", "cores": cores, "kind": "port",
            "sample": "%d worlds (one per core), each one episode of %s from its reset state "
                      "(%d of %d steps done within the %.0f s cap), numpy oracle port of the "
                      "reference, BLAS threads = 1" % (cores, scen, nmin, EPISODE, seconds),
            "per_core": steps/wall/cores}


# ---------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows)
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm)//2], "sm_max_mhz": float(self.rows[0][2]),
                "power_w_max": max(float(r[3]) for r in self.rows), "samples": len(self.rows),
                "reasons": sorted(reasons)}


class Episodes(object):
    """Staggered episodes over GROUPS contiguous blocks of the batch (see EPISODE).
    ``state`` is a triple of (elem, W) tensors (device tensors of the BatchedWorld, or
    pinned host tensors for the end-to-end pass), ``init`` the matching reset values."""

    def __init__(self, W, state, init, step_fn):
        from arboris_b200.shard import shard_range
        self.blocks = [shard_range(W, g, GROUPS) for g in range(GROUPS)]
        self.state, self.init, self.step_fn = state, init, step_fn
        self.t = -(EPISODE - PHASE)
        for g in range(GROUPS):
            self.reset(g)

    def reset(self, g):
        w0, w1 = self.blocks[g]
        if w1 > w0:
            for dst, src in zip(self.state, self.init):
                if src is None:
                    dst[:, w0:w1].zero_()
                else:
                    dst[:, w0:w1].copy_(src[:, w0:w1])

    def advance(self, k):
        while k > 0:
            if self.t % PHASE == 0:
                for g in range(GROUPS):
                    if (self.t + PHASE*g) % EPISODE == 0:
                        self.reset(g)
            c = min(k, PHASE - self.t % PHASE)
            self.step_fn(c)
            self.t += c
            k -= c

    def prime(self):
        """Untimed: bring group g to age PHASE*g."""
        self.advance(-self.t)


def parity_sample(bw, model, scen, nsample=8):
    """Checker leg: `nsample` worlds of the TIMED batch (spread over the episode groups), one more
    step on the device from their current state, against the oracle from the same state."""
    import torch
    from oracle.arboris_oracle import OracleWorld
    W = bw.nworlds
    ids = sorted(set(int(x) for x in np.linspace(0, W - 1, nsample)))
    idx = torch.as_tensor(ids, device=bw.device)
    g0, v0, f0 = (t[:, idx].cpu().numpy() for t in (bw.gpos, bw.gvel, bw.cforce))
    bw.step(DT, 1)
    torch.cuda.synchronize()
    g1, v1 = bw.gpos[:, idx].cpu().numpy(), bw.gvel[:, idx].cpu().numpy()
    act = bw.constraints("active").cpu().numpy()[ids] if model.nc else np.zeros((len(ids), 0), int)
    worst_v, worst_g, flips, nact = 0., 0., 0, 0
    for i in range(len(ids)):
        o = OracleWorld(model.to_dict())
        o.gpos[:], o.gvel[:] = g0[:, i], v0[:, i]
        if model.nrows:
            o.cforce[:] = f0[:int(model.nrows), i]
        o.step(DT)
        worst_v = max(worst_v, float(np.abs(v1[:, i] - o.gvel).max()/max(np.abs(o.gvel).max(), 1e-300)))
        worst_g = max(worst_g, float(np.abs(g1[:, i] - o.gpos).max()))
        if model.nc:
            oa = np.asarray(o.active, dtype=int)
            flips += int((oa != act[i]).sum())
            nact += int(oa.sum())
    return {"worlds": ids, "max_rel_err_gvel": worst_v, "max_abs_err_gpos": worst_g,
            "active_set_flips": flips, "active_constraints_in_sample": nact,
            "how": "after the timed region: one more device step of the whole timed batch; the sampled "
                   "worlds' states before/after are compared with one step of the numpy oracle from the "
                   "same state (checker only, not timed)"}


def dump_sample(W, model):
    """Indices (ascending) of the worlds of a W-world batch whose state --dump-outputs writes: all of
    them when their state fits DUMP_BYTES, otherwise a fixed, seeded sample that does."""
    per_world = 8*(int(model.ngpos) + int(model.ndof) + int(model.nrows) + 1)     # + its index
    n = min(W, DUMP_BYTES//per_world)
    return np.sort(np.random.default_rng(0).choice(W, size=n, replace=False))


def sample_outputs(bw, model, w0):
    """What a caller of the timed step reads back (BatchedWorld.get_state: gpos, gvel, cforce as
    (elem, worlds) float64) for the worlds of dump_sample whose state is finite, and their indices in
    the whole batch.  A world whose state is not finite has no result to compare: the reference's own
    algorithm diverges there (profiles/README.md).  Those worlds of the whole batch are listed by index
    instead ("nonfinite_world", only when there are any)."""
    import torch
    state = {"gpos": bw.gpos, "gvel": bw.gvel}
    if model.nrows:
        state["cforce"] = bw.cforce[:int(model.nrows)]
    finite = torch.ones(bw.nworlds, dtype=torch.bool, device=bw.gpos.device)
    for t in state.values():
        finite &= torch.isfinite(t).all(0)
    finite = finite.cpu().numpy()
    ids = dump_sample(bw.nworlds, model)
    ids = ids[finite[ids]]
    idx = torch.as_tensor(ids, device=bw.gpos.device)
    out = {name: t[:, idx].cpu().numpy() for name, t in state.items()}
    out["world"] = (ids + w0).astype(np.float64)
    if not finite.all():
        out["nonfinite_world"] = (np.flatnonzero(~finite) + w0).astype(np.float64)
    return out


def measure(a, scen, model, w0, w1, rank, world_size, local, full):
    """Time `a.steps` steps of worlds [w0, w1) on this rank's GPU.  Returns a dict of raw numbers
    (before the reduction over ranks).  `full`: also stage times, active-set mix, parity sample."""
    import torch
    import torch.distributed as dist
    from arboris_b200 import scenarios
    from arboris_b200.batch import BatchedWorld, HostPipeline

    W = w1 - w0
    gp, gv = scenarios.initial_states(model, scen, w0, w1)     # every world its own seed
    bw = BatchedWorld(model, W, device="cuda:%d" % local)
    for opt in (a.opt or []):                      # kernel A/B switches: --opt gs_coop=1
        name, val = opt.split("=")
        bw.set_option(name, int(val))
    gpos0 = torch.as_tensor(gp, device=bw.device)
    gvel0 = torch.as_tensor(gv, device=bw.device)
    ep = Episodes(W, (bw.gpos, bw.gvel, bw.cforce), (gpos0, gvel0, None),
                  lambda c: bw.step(DT, c))

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ep.prime()                      # untimed: stagger the episodes
    warm = max(a.warmup, 3)
    sampler = ClockSampler(local)   # samples cover the warm-up and the timed region (same load)
    sampler.start()
    ep.advance(warm)
    barrier()
    l0 = bw.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ep.advance(a.steps)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = bw.launch_count() - l0
    dump = None
    if a.dump_outputs and full and rank == 0:     # before anything below steps the batch further
        dump = sample_outputs(bw, model, w0)
    if not sampler.rows:            # a very short timed region: keep the load up until one sample exists
        t_end = time.time() + 10.
        while not sampler.rows and time.time() < t_end:
            ep.advance(PHASE)
            torch.cuda.synchronize()
    sampler.stop_flag = True
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, v in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), v)
    bad = (~torch.isfinite(bw.gvel)).any(0)
    nonfinite = int(bad.sum())
    out = {"W": W, "ms": ms, "launches": launches, "nonfinite": nonfinite, "warm": warm,
           "clocks": sampler.summary(), "device": bw.device,
           "nonfinite_ids": [int(x) + w0 for x in torch.nonzero(bad)[:8, 0].tolist()]}

    if full:
        # ---- active-set mix of the batch (for the mix-weighted flop count) and parity sample ------
        if model.nc:
            act = bw.constraints("active").cpu().numpy()
            out["flop_sum"] = float(flop_contact_increment(model, act).sum()) + W*flop_free(model)
            out["active_sum"] = float(act.sum())
        else:
            out["flop_sum"] = W*flop_free(model)
            out["active_sum"] = 0.
        if not a.no_parity_sample and rank == 0:
            out["parity_sample"] = parity_sample(bw, model, scen)
            ep.t += 1               # (the sample's extra step belongs to the episodes' clock)
        # ---- per-stage device time (diagnostic pass, CUDA events around every kernel) ----------
        bw.set_option("time_stages", 1)
        ep.advance(PHASE)
        torch.cuda.synchronize()
        out["stage"] = bw.stage_ms()
        bw.set_option("time_stages", 0)

    # ---- end to end through the host-buffer entry point ------------------------------------------
    if not a.no_e2e:
        nrows = max(int(model.nrows), 1)
        hg = torch.empty(gp.shape, dtype=torch.float64).pin_memory()
        hv = torch.empty(gv.shape, dtype=torch.float64).pin_memory()
        hf = torch.zeros((nrows, W), dtype=torch.float64).pin_memory()
        hg.copy_(bw.gpos); hv.copy_(bw.gvel); hf.copy_(bw.cforce)    # continue the same episodes
        hgn, hvn, hfn = hg.numpy(), hv.numpy(), hf.numpy()
        hep = Episodes.__new__(Episodes)
        hep.blocks, hep.t = ep.blocks, ep.t
        hep.state, hep.init = (hg, hv, hf), (torch.as_tensor(gp), torch.as_tensor(gv), None)

        pipe = None
        chunks = HostPipeline.auto_chunks(W) if a.e2e_chunks == "auto" else a.e2e_chunks
        chunks = list(chunks) if isinstance(chunks, (tuple, list)) else chunks
        out["e2e_chunks"] = chunks
        if isinstance(chunks, list) or chunks > 1:
            # the public end-to-end call: column blocks of the host state, so that copies and
            # kernels of different blocks overlap (batch.HostPipeline)
            bw.close()              # its scratch (~10 GB) is not needed any more
            pipe = HostPipeline(model, W, chunks=chunks, device=bw.device, mode=a.e2e_mode,
                                compute_streams=a.e2e_compute_streams)
            for opt in (a.opt or []):
                name, val = opt.split("=")
                pipe.set_option(name, int(val))

        def host_steps(c):
            for _ in range(c):
                if pipe is not None:
                    pipe.step(hgn, hvn, hfn if model.nrows else None, DT, 1)
                else:
                    bw.step_host(hgn, hvn, hfn, DT, 1)    # H2D state, 1 step, D2H state, sync
        hep.step_fn = host_steps
        k_e2e = max(3, min(a.steps, 100))
        hep.advance(max(3, min(a.warmup, 8)))    # the blocks' first sorts happen here
        barrier()
        t0 = time.perf_counter()
        hep.advance(k_e2e)
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
        # constraint forces travel host -> device only when they are state (ball-and-socket rows)
        has_warm = any(int(t) == 1 for t in model.cons_type)
        h2d = hgn.nbytes + hvn.nbytes + (hfn.nbytes if (model.nrows and has_warm) else 0)
        d2h = hgn.nbytes + hvn.nbytes + (hfn.nbytes if model.nrows else 0)
        out["e2e"] = {"s_per_step": t_e2e/k_e2e, "h2d": h2d, "d2h": d2h, "steps": k_e2e}
        if model.nrows and not has_warm:
            # the same pass for a caller that wants the state only (cforce = None: constraint forces stay
            # on the device): 27 % fewer bytes device -> host -- what matters where the host is the limit
            def host_steps_state(c):
                for _ in range(c):
                    if pipe is not None:
                        pipe.step(hgn, hvn, None, DT, 1)
                    else:
                        bw.step_host(hgn, hvn, None, DT, 1)
            hep.step_fn = host_steps_state
            k2 = max(3, k_e2e//2)
            hep.advance(3)
            barrier()
            t0 = time.perf_counter()
            hep.advance(k2)
            torch.cuda.synchronize()
            out["e2e"]["state_only_s_per_step"] = (time.perf_counter() - t0)/k2
            out["e2e"]["state_only_bytes"] = hgn.nbytes + hvn.nbytes
        if pipe is not None and a.e2e_mode == "serial":
            # the same pass with the calls QUEUED (HostPipeline.step(sync=False)): every step still moves
            # its state host -> device and device -> host through the in-place host arrays (a block's
            # copy-in waits for its own copy-out of the step before), but the host waits only when it
            # touches the arrays (the episode restarts, every 25 steps) -- no idle GPU between steps
            def host_steps_queued(c):
                for _ in range(c):
                    pipe.step(hgn, hvn, hfn if model.nrows else None, DT, 1, sync=False)
                pipe.wait()
            hep.step_fn = host_steps_queued
            k3 = max(3, k_e2e//2)
            hep.advance(3)
            barrier()
            t0 = time.perf_counter()
            hep.advance(k3)
            torch.cuda.synchronize()
            out["e2e"]["queued_s_per_step"] = (time.perf_counter() - t0)/k3
        if pipe is not None:
            pipe.close()
        else:
            bw.close()
        del hg, hv, hf
    else:
        bw.close()
    return out


def reduce_measure(m, device):
    """Max over ranks of the timed durations, sums of the counters."""
    from arboris_b200.shard import reduce_report
    e = m.get("e2e")
    maxes = [m["ms"], e["s_per_step"]*1e3 if e else 0., e.get("state_only_s_per_step", 0.)*1e3 if e else 0.,
             e.get("queued_s_per_step", 0.)*1e3 if e else 0.]
    sums = [m["nonfinite"], m["launches"], m["W"], m.get("flop_sum", 0.), m.get("active_sum", 0.),
            e["h2d"] if e else 0., e["d2h"] if e else 0.]
    (ms_all, e2e_ms, e2e_state_ms, e2e_queued_ms), s = reduce_report(maxes, sums, device=device)
    return {"ms": ms_all, "e2e_ms": e2e_ms, "e2e_state_ms": e2e_state_ms, "e2e_queued_ms": e2e_queued_ms, "nonfinite": int(s[0]), "launches": int(s[1]),
            "worlds": int(s[2]), "flop_sum": s[3], "active_sum": s[4], "h2d": int(s[5]), "d2h": int(s[6])}


def bind_cpu(rank, world_size):
    """Give every rank its own slice of the host cores (the end-to-end pass is bound by host memory
    traffic and the Python thread that enqueues the copies; ranks hopping over each other's cores
    cost throughput at N = 8)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores)//world_size
        if world_size > 1 and per >= 1:
            os.sched_setaffinity(0, set(cores[rank*per:(rank + 1)*per]))
            return per
    except Exception:
        pass
    return None


def run_ours(a):
    import torch
    import torch.distributed as dist
    from arboris_b200 import scenarios, _capi
    from arboris_b200.flatten import flatten
    from arboris_b200.shard import env_rank, shard_range

    rank, world_size, local = env_rank()
    torch.cuda.set_device(local)
    # stdout carries exactly ONE line (the JSON, rank 0): anything a library prints there
    # meanwhile (NCCL's version banner at the first collective) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cores_per_rank = bind_cpu(rank, world_size)
    scen, nworlds = WORKLOADS[a.workload]
    if a.worlds:
        nworlds = a.worlds
    model = flatten(scenarios.BUILDERS[scen]())
    device = torch.device("cuda", local)

    def run(scaling, full):
        total = nworlds*world_size if scaling == "weak" else nworlds
        w0, w1 = shard_range(total, rank, world_size)   # contiguous block of worlds per GPU
        m = measure(a, scen, model, w0, w1, rank, world_size, local, full)
        r = reduce_measure(m, device)
        r["total"], r["per_gpu"], r["raw"] = total, w1 - w0, m
        return r

    head = run(a.scaling, True)
    other = None
    if world_size > 1 and not a.no_other_scaling:
        other_name = "strong" if a.scaling == "weak" else "weak"
        other = run(other_name, False)
    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return
    m = head["raw"]
    W = head["per_gpu"]
    total_worlds = head["worlds"]
    value = total_worlds*a.steps/(head["ms"]*1e-3)
    lib = _capi.load()
    peak = C_double()
    lib.arb_measure_fp64_peak(local, peak.ref())
    fp64_peak = peak.value
    flop_mix = head["flop_sum"]/max(total_worlds, 1)         # mix-weighted, SURVEY.md 8(d) formula
    flop_all_active = flop_free(model) + float(flop_contact_increment(
        model, np.ones((1, int(model.nc)))).sum()) if model.nc else flop_free(model)
    achieved = (value/world_size)*flop_mix        # per GPU, flop/s
    peaks, traffic = {}, {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(scen, {})
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.))
    st = m.get("stage", {"prepare": 0., "gs": 0., "finish": 0., "steps": 0})
    nst = max(st["steps"], 1)
    stage = {k: st[k]/nst for k in ("prepare", "gs", "finish")}
    tot_stage = sum(stage.values()) or 1.
    dom = max(stage, key=stage.get)
    gs_unstaged = "gs_stage=0" in (a.opt or []) or model.nc > 32     # (arb_batch_set_option: gs_stage)
    dram_per_world = traffic.get("dram_bytes_per_world_step")
    exec_flop = traffic.get("executed_fp64_flop_per_world_step")
    out = {
        "metric": "world-steps/s (human36, fp64, dt=1ms)", "value": value, "unit": "world-steps/s",
        "n_gpus": world_size, "steps": a.steps, "warmup": m["warm"], "ms_per_step": head["ms"]/a.steps,
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (seeded random initial states, one seed per world, SURVEY.md 8(d))",
        "config": config_of(a, scen, total_worlds, W, world_size, a.scaling, model),
        "gpu_launches": int(head["launches"]),
        "nonfinite_worlds": int(head["nonfinite"]),
        "nonfinite_world_ids": m["nonfinite_ids"],
        "roofline": {"bound": "fp64", "achieved": achieved/1e12, "peak": fp64_peak/1e12,
                     "unit": "TFLOP/s", "frac": achieved/fp64_peak if fp64_peak else None,
                     "frac_algorithmic": achieved/fp64_peak if fp64_peak else None,
                     "frac_all_active": (value/world_size)*flop_all_active/fp64_peak if fp64_peak else None,
                     "frac_executed": ((value/world_size)*exec_flop/fp64_peak
                                       if (exec_flop and fp64_peak) else None),
                     "traffic": dram_per_world*W if dram_per_world else None,
                     "traffic_note": traffic.get("source"),
                     "peak_source": "DFMA micro-benchmark measured in this run (arb_measure_fp64_peak); "
                                    "MEASURED_PEAKS.json has no fp64 entry",
                     "flop_per_world_step": flop_mix,
                     "flop_per_world_step_all_active": flop_all_active,
                     "flop_per_world_step_executed": exec_flop,
                     "flop_note": "frac / frac_algorithmic: SURVEY.md 8(d) primary count evaluated on the ACTIVE "
                                  "SETS of the timed batch (mean %.2f of %d constraints active per world); "
                                  "frac_all_active: the same formula with every constraint active (0.99 Mflop, "
                                  "round 1's numerator); frac_executed: fp64 flops the kernels EXECUTE per "
                                  "world-step (ncu smsp__sass_thread_inst_executed_op_{dfma x2, dmul, dadd}_pred_on "
                                  "summed over the three stage launches, profiles/traffic.json) -- the articulated "
                                  "form does far fewer flops than the assembled-matrix count"
                                  % (head["active_sum"]/max(total_worlds, 1), int(model.nc)),
                     "per_launch": "one (prepare, gs, finish) triple = one step of the %d worlds of a GPU; "
                                   "achieved = worlds x flop_per_world_step / step time" % W,
                     "stage_ms": stage,
                     "dominant_kernel": {"prepare": "k_fused_prepare_lane", "finish": "k_fused_finish",
                                         "gs": "k_fused_gs" if gs_unstaged else "k_fused_gs_staged"}[dom],
                     "dominant_share": stage[dom]/tot_stage,
                     "hbm": {"achieved": value/world_size*STATE_BYTES_PER_WORLD_STEP/1e9,
                             "peak": hbm_peak, "unit": "GB/s",
                             "frac": value/world_size*STATE_BYTES_PER_WORLD_STEP/1e9/hbm_peak,
                             "dram_bytes_per_world_step": dram_per_world,
                             "dram_achieved": (dram_per_world*value/world_size/1e9
                                               if dram_per_world else None),
                             "dram_frac": (dram_per_world*value/world_size/1e9/hbm_peak
                                           if dram_per_world else None)}},
        "clocks": m["clocks"],
    }
    if cores_per_rank:
        out["config"]["host_cores_per_rank"] = cores_per_rank
    if "parity_sample" in m:
        out["parity_sample"] = m["parity_sample"]

    def e2e_obj(r):
        o = {"value": r["worlds"]/(r["e2e_ms"]*1e-3), "unit": "world-steps/s",
             "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
             "steps": r["raw"]["e2e"]["steps"], "chunks": r["raw"].get("e2e_chunks"), "mode": a.e2e_mode}
        if r.get("e2e_state_ms"):
            nb = r["raw"]["e2e"]["state_only_bytes"]*world_size
            o["state_only"] = {"value": r["worlds"]/(r["e2e_state_ms"]*1e-3), "unit": "world-steps/s",
                               "h2d_bytes_per_step": nb, "d2h_bytes_per_step": nb,
                               "how": "the same call with cforce = None: gpos and gvel travel, the constraint "
                                      "forces stay on the device"}
        if r.get("e2e_queued_ms"):
            o["queued"] = {"value": r["worlds"]/(r["e2e_queued_ms"]*1e-3), "unit": "world-steps/s",
                           "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                           "how": "the same copies and steps with HostPipeline.step(sync=False): calls are "
                                  "queued, a block's copy-in waits for its own copy-out of the step before, "
                                  "the host waits (HostPipeline.wait) only before it touches the arrays "
                                  "(episode restarts, every 25 steps)"}
        return o
    if "e2e" in m:
        out["e2e"] = e2e_obj(head)
        ch = m.get("e2e_chunks")
        nblocks = len(ch) if isinstance(ch, list) else ch
        out["e2e"]["how"] = (
            ("HostPipeline.step (%d column blocks of the pinned host state; %s): host -> "
             "device (gpos, gvel; constraint forces only for models whose forces are state), 1 step, "
             "device -> host (gpos, gvel, cforce), all blocks synchronised, every step; same "
             "staggered episodes as the timed region"
             % (nblocks,
                ("kernels of all blocks on %s, block after block, "
                 "arb_state_copy_host_strided copies on two more streams ordered by events"
                 % ("one stream per block, earlier blocks at higher priority"
                    if a.e2e_compute_streams == "priority" else "%d streams" % a.e2e_compute_streams))
                if a.e2e_mode == "serial"
                else "arb_step_host_strided, one stream per block"))
            if nblocks > 1 else
            "arb_step_host: pinned host state -> device, 1 step, device -> host, "
            "synchronised, every step; same staggered episodes as the timed region")
    if other is not None:
        o = {"scaling": other_name, "value": other["worlds"]*a.steps/(other["ms"]*1e-3),
             "unit": "world-steps/s", "ms_per_step": other["ms"]/a.steps,
             "worlds_total": other["worlds"], "worlds_per_gpu": other["per_gpu"],
             "nonfinite_worlds": other["nonfinite"], "gpu_launches": other["launches"],
             "clocks": other["raw"]["clocks"],
             "note": "BASELINE.json configs[4] read literally: the workload's worlds IN TOTAL, split over "
                     "the GPUs; same protocol, same run" if other_name == "strong" else
                     "every GPU steps the workload's number of worlds; same protocol, same run"}
        if "e2e" in other["raw"]:
            o["e2e"] = e2e_obj(other)
        out[other_name] = o
    if not a.no_cpu_baseline and world_size == 1:      # rank 0 at N = 1 only
        out["cpu_baseline"] = cpu_baseline(scen, a.cpu_seconds)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(out), flush=True)
    os.dup2(2, 1)
    if world_size > 1:
        dist.destroy_process_group()


class C_double(object):
    def __init__(self):
        import ctypes
        self._c = ctypes.c_double(0.)
        self._ct = ctypes

    def ref(self):
        return self._ct.byref(self._c)

    value = property(lambda self: self._c.value)


def run_reference(a):
    """Reference arm: the reference's CPU implementation of the path (the numpy oracle
    port -- the Python reference cannot travel to the GPU box) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from arboris_b200 import scenarios
    from arboris_b200.flatten import flatten
    scen, total = WORKLOADS[a.workload]
    if a.worlds:
        total = a.worlds
    n = max(a.gpus, 1)
    per_gpu = total if a.scaling == "weak" else -(-total//n)
    if a.scaling == "weak":
        total *= n
    model = flatten(scenarios.BUILDERS[scen]())
    base = cpu_baseline(scen, a.cpu_seconds)
    v = base["value"]
    out = {
        "impl": "reference", "metric": "world-steps/s (human36, fp64, dt=1ms)", "value": v,
        "unit": "world-steps/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3/v if v else None, "higher_is_better": True, "scaling": a.scaling,
        "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (seeded random initial states, one seed per world, SURVEY.md 8(d))",
        "config": config_of(a, scen, total, per_gpu, n, a.scaling, model),
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "world-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
