"""bench.py's host-side helpers: the SURVEY.md 8(d) flop formulas (pinned to the survey's own
worked numbers), the config object both arms print, and what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from arboris_b200 import scenarios  # noqa: E402
from arboris_b200.flatten import flatten  # noqa: E402


def test_flop_formulas_reproduce_survey_numbers():
    """SURVEY.md 8(d): human36 free step 360 118 flop; with 8 active contacts the increment is
    65 856 + 198 912 + 9 744 + 353 280; snake9 111 080."""
    m = flatten(scenarios.human36_contact_world())
    assert bench.flop_free(m) == 360118.
    act = np.zeros((3, 10))
    act[0, :8] = 1          # the 8 contacts, no knee limit
    act[2, :] = 1           # everything
    inc = bench.flop_contact_increment(m, act)
    assert inc[0] == 65856 + 198912 + 9744 + 353280
    assert inc[1] == 0.     # no active constraint: no contact work
    assert inc[2] > inc[0]
    s = flatten(scenarios.snake_loop_world())
    # (the survey's snake has no constraints and 9 links + free base: k_b = 6..15)
    assert bench.flop_free(s) == 111080.


def test_both_arms_print_the_same_config_keys():
    class A(object):
        workload = "human36_contact_262144"
    m = flatten(scenarios.human36_contact_world())
    ours = bench.config_of(A, "human36_contact", 262144, 262144, 1, "weak", m)
    ref = bench.config_of(A, "human36_contact", 262144, 262144, 1, "weak", m)
    assert set(ours) == set(ref) and ours["distinct_worlds"] == 262144 and ours["constraints"] == 10


def test_auto_chunks_follow_batch_size():
    from arboris_b200.batch import HostPipeline
    assert HostPipeline.auto_chunks(32768) == 1
    assert HostPipeline.auto_chunks(131072) == (1, 2, 1)
    assert HostPipeline.auto_chunks(262144) == (1, 1, 2, 2, 2, 1, 1)


def test_traffic_json_follows_from_the_committed_ncu_summaries():
    """profiles/traffic.json (what bench.py reports as roofline.traffic and frac_executed) can be
    recomputed from the ncu summaries committed beside it (profiles/make_traffic.py)."""
    import importlib.util
    import json
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prof = os.path.join(root, "profiles")
    doc = json.load(open(os.path.join(prof, "traffic.json")))["human36_contact"]
    tag = re.search(r"profiles/(\w+)_ncu_", doc["source"]).group(1)
    spec = importlib.util.spec_from_file_location("make_traffic", os.path.join(prof, "make_traffic.py"))
    mt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mt)
    W = 262144
    tot_b = tot_f = 0.
    for st in ("prepare", "gs", "finish"):
        r = mt.read(os.path.join(prof, "%s_ncu_%s_%d.txt" % (tag, st, W)))
        b = (r["dram__bytes_read.sum"] + r["dram__bytes_write.sum"])/W
        f = (2*r["smsp__sass_thread_inst_executed_op_dfma_pred_on.sum"]
             + r["smsp__sass_thread_inst_executed_op_dmul_pred_on.sum"]
             + r["smsp__sass_thread_inst_executed_op_dadd_pred_on.sum"])/W
        assert abs(doc["per_kernel_bytes_per_world"][r["kernel"]] - b) <= 1e-9*b
        assert abs(doc["per_kernel_executed_fp64_flop_per_world"][r["kernel"]] - f) <= 1e-9*f
        tot_b += b
        tot_f += f
    assert abs(doc["dram_bytes_per_world_step"] - tot_b) <= 1e-9*tot_b
    assert abs(doc["executed_fp64_flop_per_world_step"] - tot_f) <= 1e-9*tot_f


def test_dump_sample_is_fixed_and_bounded():
    """--dump-outputs writes the same worlds every run: a seeded sample below 64 MB at the bench size,
    the whole batch when it fits."""
    m = flatten(scenarios.human36_contact_world())
    ids = bench.dump_sample(262144, m)
    assert np.array_equal(ids, bench.dump_sample(262144, m))
    assert ids[0] >= 0 and ids[-1] < 262144 and (np.diff(ids) > 0).all()
    assert len(ids)*8*(m.ngpos + m.ndof + m.nrows + 1) <= bench.DUMP_BYTES < 64 << 20
    assert np.array_equal(bench.dump_sample(640, m), np.arange(640))


def test_dump_leaves_out_worlds_without_a_finite_state():
    """A world whose state is not finite (the reference's own algorithm diverges there) is not part
    of the dumped sample; every such world of the batch is listed by index instead."""
    import torch
    m = flatten(scenarios.human36_contact_world())
    W, w0 = 300, 1000

    class Batch(object):          # the state tensors of a BatchedWorld, on the host
        nworlds = W
        gpos = torch.rand(m.ngpos, W, dtype=torch.float64)
        gvel = torch.rand(m.ndof, W, dtype=torch.float64)
        cforce = torch.rand(m.nrows, W, dtype=torch.float64)
    Batch.gvel[3, 17] = float("nan")
    Batch.gpos[0, 250] = float("inf")
    Batch.cforce[m.nrows - 1, 5] = float("nan")
    out = bench.sample_outputs(Batch, m, w0)
    keep = [w for w in range(W) if w not in (5, 17, 250)]
    assert np.array_equal(out["world"], np.array(keep) + w0)
    assert np.array_equal(out["nonfinite_world"], [w0 + 5, w0 + 17, w0 + 250])
    for name in ("gpos", "gvel", "cforce"):
        assert np.array_equal(out[name], getattr(Batch, name)[:, keep].numpy())
    assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in out.values())
    Batch.gvel[3, 17] = Batch.gpos[0, 250] = Batch.cforce[m.nrows - 1, 5] = 0.
    assert "nonfinite_world" not in bench.sample_outputs(Batch, m, w0)


@pytest.mark.gpu
def test_dump_outputs_is_the_state_after_the_timed_steps(tmp_path):
    """bench.py --dump-outputs writes the state its last timed step leaves: bit for bit that of the
    same worlds stepped here through the same staggered episodes, warm-up then --steps steps."""
    import torch
    from arboris_b200.batch import BatchedWorld
    W, warm, steps = 640, 4, 7
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--worlds", str(W),
                          "--steps", str(steps), "--warmup", str(warm), "--no-e2e", "--no-cpu-baseline",
                          "--no-parity-sample", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, check=True)
    line = json.loads(run.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warm and line["config"]["worlds_total"] == W
    scen = bench.WORKLOADS[line["config"]["workload"]][0]
    model = flatten(scenarios.BUILDERS[scen]())
    gp, gv = scenarios.initial_states(model, scen, 0, W)
    bw = BatchedWorld(model, W, device="cuda:0")
    ep = bench.Episodes(W, (bw.gpos, bw.gvel, bw.cforce),
                        (torch.as_tensor(gp, device=bw.device), torch.as_tensor(gv, device=bw.device), None),
                        lambda c: bw.step(bench.DT, c))
    ep.prime()
    ep.advance(warm)
    ep.advance(steps)
    g, v, f = bw.get_state()
    got = {name: np.load(str(tmp_path/(name + ".npy"))) for name in ("gpos", "gvel", "cforce", "world")}
    assert all(x.dtype == np.float64 for x in got.values())
    assert np.array_equal(got["world"], np.arange(W))
    assert np.array_equal(got["gpos"], g) and np.array_equal(got["gvel"], v) and np.array_equal(got["cforce"], f)
