"""bench.py's one-line JSON contract and its --dump-outputs files: the reference arm on the CPU, the GPU arm (gpu-marked)
against the library's own proofs of the same seeded inputs."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "groth16_withdraw_proofs_per_sec" and line["unit"] == "proofs/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["steps"] == 1 and line["warmup"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["gpu_launches"] == 0
    proofs, pub = np.load(tmp_path / "proofs.npy"), np.load(tmp_path / "public_inputs.npy")
    assert proofs.dtype == pub.dtype == np.float32 and proofs.shape[1:] == (256,) and pub.shape == (proofs.shape[0], 96)
    assert proofs.shape[0] >= 8 and 0 <= proofs.min() and proofs.max() <= 255 and (proofs == np.round(proofs)).all()


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_launch_list_tool_reads_the_committed_ncu_csv(tmp_path):
    """tools/launch_list_summary.py turns the committed ncu launch list into the table under profiles/: the dominant kernel of
    the bench command must come out on top (this is the evidence the roofline share is checked against)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "ll.md"
    subprocess.run([sys.executable, os.path.join(root, "tools", "launch_list_summary.py"),
                    os.path.join(root, "profiles", "r2_launches_bench_steps2.csv"), str(out), "t"], check=True)
    rows = [l for l in out.read_text().splitlines() if l.startswith("| `")]
    assert rows and rows[0].startswith("| `k_bucket_acc_sm1"), rows[:2]


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(ctx, tmp_path):
    """--dump-outputs of the GPU arm holds the proofs and public inputs the library computes for bench.py's seeded inputs,
    and --steps is the number of timed steps."""
    import bench
    import owshen_b200 as ob
    batch = 4
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", str(batch),
                          "--no-cpu-baseline", "--no-parity", "--sharded-log-n", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["proofs_verify"] and line["config"]["e2e_bytes_equal_device_path"]
    proofs, pub = np.load(tmp_path / "proofs.npy"), np.load(tmp_path / "public_inputs.npy")
    assert proofs.dtype == pub.dtype == np.float32 and proofs.shape == (batch, 256) and pub.shape == (batch, 96)
    pk, _ = ob.setup_withdraw(ctx, bench.DEPTH, *bench.toxic(random.Random(bench.TOXIC_SEED)))
    PK = ob.ProvingKey(ctx, pk)
    nul, sec, rec, sib, bits, rs = bench.synth_inputs(random.Random(bench.INPUT_SEED), batch, bench.DEPTH)
    exp_proofs, exp_pub = ob.prove(PK, nul, sec, rec, sib, bits, rs)
    PK.close()
    assert proofs.astype(np.uint8).tobytes() == exp_proofs and pub.astype(np.uint8).tobytes() == exp_pub
