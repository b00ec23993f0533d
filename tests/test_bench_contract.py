"""The bench contract, checked without a GPU through the reference arm (`bench.py --impl reference`): one JSON line with
the keys a reader of the line relies on, the oracle port timed on the host cores, and no kernel launches claimed.  On a GPU, the
outputs `--dump-outputs` writes are checked against the line's digests and the oracle."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-log-n", "10", "--ref-sc-log-n", "10"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "points/s" and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["sumcheck"]["unit"] == "field-elems/s" and line["sumcheck"]["value"] > 0
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1", "--ref-log-n", "10", "--ref-sc-log-n", "10"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_traffic_comes_from_the_committed_profiles_and_config_is_shared():
    """roofline.traffic is read from the newest ncu summary under profiles/ (not a constant in bench.py); both arms of
    the bench print the same `config` object; the digest file the GPU arm compares itself with is complete."""
    import argparse
    import json

    import bench

    msm, msm_src = bench.profile_traffic("msm")
    sc, sc_src = bench.profile_traffic("sumcheck")
    assert msm_src.startswith("profiles/") and sc_src.startswith("profiles/")
    assert 14.5e9 < msm < 40e9      # algorithmic 14.5 GB; the 64-byte gathers pull 128-byte lines
    assert 6.0e9 < sc < 7.5e9       # algorithmic 6.44 GB: no re-reads
    args = argparse.Namespace(log_n=24, no_precompute=False)
    assert bench.workload_config(args, 1) == bench.workload_config(args, 1, peer_memory=False)  # one GPU: no exchange
    assert bench.workload_config(args, 8)["exchange"] != bench.workload_config(args, 8, peer_memory=False)["exchange"]
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_digests_2_24.json")))
    assert g["log_n"] == 24 and set(g["digests"]) >= {"commitment_xy", "commitment_serialized", "sumcheck_claimed_sum",
                                                      "sumcheck_final_transcript_state", "sumcheck_evaluation",
                                                      "zerocheck_final_transcript_state"}
    assert bench.shard_seed(5, 0) == 5 and bench.shard_seed(5, 1) == (5 + 4 * bench.GOLDEN64) % (1 << 64)


def _limb_bytes(a) -> bytes:
    return a.astype("<u4").tobytes()


def test_dump_outputs_writes_every_byte_of_a_proof_exactly(tmp_path):
    """--dump-outputs: a proof object (dataclasses, lists, tuples, arrays, bytes) becomes one float64 vector of 32-bit
    limbs holding all its bytes in field order, exactly"""
    import numpy as np

    import bench
    import quill_zkvm_b200 as q

    rng = np.random.default_rng(7)
    fr = lambda *shape: rng.integers(0, 256, size=shape + (32,), dtype=np.uint8)  # noqa: E731
    proof = q.SumcheckProof(2, fr(), [fr(4), fr(3)])
    claim = q.EvaluationClaim(fr(2), fr())
    state = bytes(range(32))
    bench.dump_outputs(str(tmp_path / "out"), {"sumcheck": (proof, claim), "state": state})
    assert sorted(os.listdir(tmp_path / "out")) == ["state.npy", "sumcheck.npy"]
    got = np.load(tmp_path / "out" / "sumcheck.npy")
    assert got.dtype == np.float64 and np.all(got == np.floor(got)) and got.max() < 2 ** 32
    want = b"".join(a.tobytes() for a in (proof.claimed_sum, *proof.r_polys, claim.point, claim.evaluation))
    assert _limb_bytes(got) == want
    assert _limb_bytes(np.load(tmp_path / "out" / "state.npy")) == state


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_gpu_path(ctx, tmp_path):
    """bench.py --dump-outputs at a small size with every leg on: the files hold what the line's digests report, and the
    MSM commitment is the oracle's closed form p(tau) * g on the bench's seeded scalars"""
    import numpy as np

    import bench
    from oracle import coracle as co

    log_n, steps = 12, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                          "--log-n", str(log_n), "--mlpcs-log-n", "10", "--hyperplonk-log-rows", "5", "--no-verify",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    d = tmp_path / "out"
    names = {f[:-4] for f in os.listdir(d)}
    assert names == {"msm_commitment", "msm_commitment_host_scalars", "msm_pair_levels_commitment", "sumcheck_proof",
                     "sumcheck_transcript_state", "sumcheck_proof_host_tables", "sumcheck_transcript_state_host_tables",
                     "zerocheck_proof", "zerocheck_transcript_state", "mlpcs_commitment", "mlpcs_opening",
                     "hyperplonk_proof"}
    assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
    got = {n: _limb_bytes(np.load(d / f"{n}.npy")) for n in names}
    dg = line["digests"]
    assert got["msm_commitment"].hex() == dg["commitment_xy"]
    assert got["msm_commitment_host_scalars"] == got["msm_pair_levels_commitment"] == got["msm_commitment"]
    assert got["sumcheck_transcript_state"].hex() == dg["sumcheck_final_transcript_state"]
    assert got["sumcheck_transcript_state_host_tables"] == got["sumcheck_transcript_state"]
    assert got["sumcheck_proof_host_tables"] == got["sumcheck_proof"]
    assert got["sumcheck_proof"][-32:].hex() == dg["sumcheck_evaluation"]
    assert got["zerocheck_transcript_state"].hex() == dg["zerocheck_final_transcript_state"]
    assert got["hyperplonk_proof"][-32:].hex() == line["hyperplonk_prove"]["final_transcript_state"]
    sc = ctx.random_fr(1 << log_n, bench.shard_seed(0x5155494C4C, 0))
    y, _ = co.kzg_open_quotient(sc.download().reshape(-1, 32), co.fr1(bench.TAU))
    sc.free()
    assert bytes(co.g1_mul(co.g1_to_bytes((1, 2)), y)).hex() == dg["commitment_xy"]
