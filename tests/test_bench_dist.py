"""CPU: the N>1 plumbing of bench.py (one process per GPU, max-over-ranks timing, rank 0 reports) exercised with the
gloo backend at world_size 2."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    # same reduction bench.py performs on [t_dev, t_e2e]
    t = torch.tensor([0.10 + 0.05 * rank, 0.20 - 0.03 * rank], dtype=torch.float64)
    dist.barrier()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    frames = 100 * world / float(t[0])
    q.put((rank, float(t[0]), float(t[1]), frames))
    dist.destroy_process_group()


def test_max_over_ranks_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, 29631, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in ps:
        p.join(60)
    for rank, tdev, te2e, frames in res:
        assert abs(tdev - 0.15) < 1e-12 and abs(te2e - 0.20) < 1e-12
        assert abs(frames - 200 / 0.15) < 1e-9


def test_reference_arm_nonzero_ranks_exit_quietly():
    import subprocess
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "4", "--warmup", "3"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


_DEADLINE_SCRIPT = r"""
import sys, time, json
sys.path.insert(0, {root!r})
import numpy as np
import bench
import rvio_b200  # noqa: F401
from rvio_b200 import synth
cfg = synth.baseline_config(1)
wl = dict(imus=[np.zeros((10, 8))] * 8, cand2=[np.zeros((5, 2), np.float32)] * 8)
bench._LINE_CTX.update(cfg=cfg, wl=wl, world=2, K=4, W=3, peaks=dict(hbm_gbs=6564.2, _measured=True), workload=dict(workload="test"))
res = dict(t_dev=0.002, t_e2e=0.004, t_e2s=0.005, dev_ms=[0.5] * 4, e2e_ms=[1.0] * 4, launches=80, clocks=dict(sm_mhz=1965.0),
           prof=dict(), dev_wall=0.002, e2e_wall=0.004, e2s_wall=0.005, timeline=None, batch=None, infos=[(1, 1, 9, 9, 0)],
           affinity=None, sharded=None, t_dev_rank=[0.002, 0.0019], t_e2e_rank=[0.004, 0.0038], pref_hits=4, h2d_frame_us=12.0)
bench._arm_legs_deadline(res, int(sys.argv[1]))
time.sleep(30)            # "an extra leg that never returns"
print("not reached")
"""


def test_legs_deadline_prints_the_line_from_completed_legs(tmp_path):
    """bench.py's headline numbers exist before any extra leg starts; if a leg wedges, rank 0 still prints the JSON line from
    the completed legs and every rank exits 0 (a hung collective on one box must not cost the whole measurement)."""
    import json
    import subprocess
    script = tmp_path / "deadline.py"
    script.write_text(_DEADLINE_SCRIPT.format(root=ROOT))
    env = dict(os.environ, RVIO_BENCH_LEGS_DEADLINE_S="1")
    out0 = subprocess.run([sys.executable, str(script), "0"], capture_output=True, text=True, env=env, timeout=120)
    assert out0.returncode == 0, out0.stderr[-800:]
    line = json.loads(out0.stdout.strip().splitlines()[-1])
    assert line["metric"] == "vio_frames_per_sec" and line["n_gpus"] == 2 and line["steps"] == 4
    assert abs(line["value"] - 2 * 4 / 0.002) < 1e-6 and abs(line["e2e"]["value"] - 2 * 4 / 0.004) < 1e-6
    assert abs(line["e2e"]["strict"]["value"] - 2 * 4 / 0.005) < 1e-6
    assert "legs_deadline" in line and line["sharded"] is None and line["roofline"] is None
    out1 = subprocess.run([sys.executable, str(script), "1"], capture_output=True, text=True, env=env, timeout=120)
    assert out1.returncode == 0 and out1.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_repeat_from_run_to_run(tmp_path):
    """--dump-outputs writes the last timed step's pose, filter state and update counters as float64; two runs with the same
    arguments write the same arrays (seeded inputs), and --steps is the number of timed steps."""
    import json
    import subprocess
    env = dict(os.environ, RVIO_BENCH_SETTLE_STEPS="0")
    runs = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "7", "--warmup", "3", "--no-extra-legs",
                              "--no-cpu-baseline", "--batch-streams", "0", "--dump-outputs", str(d)],
                             capture_output=True, text=True, env=env, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 7 and len(line["update_frames"]["rows_kept_flags"]) == 7
        runs.append({n: np.load(d / f"{n}.npy") for n in ("pose", "state_x", "state_P", "update_info")})
    a, b = runs
    for n in a:
        assert a[n].dtype == np.float64 and np.array_equal(a[n], b[n]), n
    n_clones = (len(a["state_x"]) - 26) // 7
    assert a["pose"].shape == (7,) and np.isfinite(a["pose"]).all()
    assert a["state_P"].shape == (24 + 6 * n_clones,) * 2 and a["update_info"].shape == (5,)


def test_no_undefined_names_in_the_python_sources():
    """pyflakes is not in this image; tools/check_names.py catches a name that is used but bound nowhere (a function lost in an edit)."""
    import glob
    import subprocess
    files = [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]
    for d in ("r-vio_b200", "tools", "tests", "oracle"):
        files += sorted(glob.glob(os.path.join(ROOT, d, "*.py")))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "check_names.py")] + files, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout[-2000:]
