#!/usr/bin/env python
"""bench.py -- the reference's headline metric (BASELINE.json): KZG-commit MSM points/s and sumcheck field-elems/s
at 2^24, on N B200s of one node, with the host-CPU restatement of the reference timed beside it.

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port), host cores
    python bench.py ... --dump-outputs DIR                   # + the outputs of every timed leg's last step, DIR/*.npy

One JSON line on stdout.  Top-level value = MSM points/s (inputs resident in HBM); `sumcheck` holds the second half of
the metric; `e2e` = the same MSM through the public API from pinned HOST buffers (H2D + D2H inside the timed region).
A step = one KZG commit of 2^log_n scalars (MSM loop) / one sumcheck proof over three 2^log_n tables (sumcheck loop);
both loops are timed separately, each bracketed by barrier + synchronize, max over ranks.  N > 1 shards the SAME 2^log_n
problem (strong scaling): MSM by index range, sumcheck tables by the top variables (SURVEY 8e).
Inputs (0.5 GiB scalars + 1 GiB bases; 1.5 GiB tables) are far larger than the 126 MB L2, so no flush is needed.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FR = 21888242871839275222246405745257275088548364400416034343698204186575808495617
TAU = 0x1234567890ABCDEF1234567890ABCDEF
MSM_LIMB_PRODUCTS_PER_POINT = 20480  # SURVEY 8(d): 16 windows x (8M + 2S) x 128 32x32->64 products per Montgomery mult
SC_BYTES_PER_ELEM = 128              # SURVEY 8(d): 4 * 32 B per input table element over the whole proof
SC_ZC_WEIGHT_BYTES_PER_ENTRY = 64    # eq-factored zero-check: the weight tables E_1, E_2, .. (N/2, N/4, .. entries) are
                                     # written once and read once each: 2 * 32 B * N = 64 B per entry of ONE table


def profile_traffic(kind: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, read from the newest committed
    `ncu --set full` summary under profiles/ (tools/summarise_profiles.py writes them), 2^24 on one GPU.
    msm: the single msm_accumulate launch.  sumcheck: the captured launches are round 0 (evaluate only) and round 1
    (fold fused); the later streaming rounds halve, so the proof's traffic is round0 + 2 * round1 (geometric series,
    the 2^-k tail below the streamed sizes neglected).  Returns (bytes, source file) or (None, None)."""
    import glob
    import re
    pat = {"msm": "*_ncu_msm_accumulate.txt", "sumcheck": "*_ncu_sc_round_prod.txt"}[kind]
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pat)))
    if not files:
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    per_launch, cur = [], None
    for line in open(files[-1]):
        if line.startswith("## captured launch"):
            cur = 0.0
            per_launch.append(cur)
        m = re.match(r"dram__bytes_(read|write)\.sum \[(\w+)\] = ([0-9.,]+)", line)
        if m and per_launch:
            per_launch[-1] += float(m.group(3).replace(",", "")) * unit.get(m.group(2), 1.0)
    if not per_launch:
        return None, None
    src = os.path.relpath(files[-1], ROOT)
    if kind == "msm":
        return per_launch[0], src
    if len(per_launch) < 2:
        return None, None
    return per_launch[0] + 2.0 * per_launch[1], src


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


GOLDEN64 = 0x9E3779B97F4A7C15


def shard_seed(seed: int, first_index: int) -> int:
    """qz_dev_random_fr derives element i from seed + GOLDEN64 * (4 i + 1) (mod 2^64), so a shard that starts at global
    index `first_index` continues the SAME sequence when seeded with seed + 4 * first_index * GOLDEN64: every GPU count
    proves the same problem and the digests printed in the line must be equal for N = 1, 2, 4, 8."""
    return (seed + 4 * first_index * GOLDEN64) & 0xFFFFFFFFFFFFFFFF


def workload_config(args, world: int, peer_memory: bool = True) -> dict:
    """The `config` object of the line: the workload both arms are quoted on (the reference arm times a bounded sample
    of it and says so in `cpu_baseline.sample`)."""
    return {"workload": f"KZG commit MSM of 2^{args.log_n} random Fr scalars on a tau-power SRS + linear-time "
                        f"sumcheck over a degree-3 product of three 2^{args.log_n}-entry tables (BN254)",
            "log_n": args.log_n, "msm_precomputed_windows": not args.no_precompute,
            "sharding": f"index ranges / top variables over {world} GPU(s)",
            "exchange": ("peer mailboxes in HBM over NVLink (CUDA IPC), written by the producing kernel" if peer_memory
                         else "NCCL all-gather") if world > 1 else "none",
            "l2": "inputs (>= 1.5 GiB) exceed the 126 MB L2; no flush needed"}


def product_expr(q, k):
    e = q.VirtualPolyExpr.Input(0)
    for i in range(1, k):
        e = e * q.VirtualPolyExpr.Input(i)
    return e


def output_bytes(o) -> list:
    """The byte arrays of one output (a G1 point, a transcript state, or a proof built of dataclasses, lists and tuples
    of them) in field order; integer fields (num_vars) follow from the arguments and are left out."""
    import numpy as np
    if dataclasses.is_dataclass(o):
        return [b for f in dataclasses.fields(o) for b in output_bytes(getattr(o, f.name))]
    if isinstance(o, (list, tuple)):
        return [b for x in o for b in output_bytes(x)]
    if isinstance(o, bytes):
        return [np.frombuffer(o, dtype=np.uint8)]
    if isinstance(o, np.ndarray):
        return [np.ascontiguousarray(o).view(np.uint8).reshape(-1)]
    return []


def dump_outputs(path: str, outputs: dict) -> None:
    """--dump-outputs: each output as PATH/<name>.npy, the float64 vector of its little-endian 32-bit limbs (Montgomery
    form for field elements and points, as the API returns them).  Every limb is below 2^53, so the values are exact and
    two builds can be compared output for output.  The outputs are proofs and commitments: a few hundred KB at most."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, o in outputs.items():
        b = np.concatenate([np.zeros(0, dtype=np.uint8)] + output_bytes(o))
        np.save(os.path.join(path, name + ".npy"), b.view("<u4").astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's CPU algorithm for the path (oracle port; the arkworks binary cannot be built: no Rust toolchain),
    on the box's host cores.  Each step is a bounded sample: KZG::commit (pcs/src/kzg.rs:61-73, including its per-call
    SRS normalisation) on 2^ref_log_n points, and SumcheckProof::prove on three 2^ref_sc_log_n tables."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from oracle import coracle as co
    from oracle import pyref as py
    from tests import util

    cores = os.cpu_count() or 1
    n = 1 << args.ref_log_n
    g = co.g1_to_bytes(py.g1_mul(py.G1_GEN, 7))
    srs = co.srs_generate(g, co.fr1(TAU), n, threads=cores)
    sc = util.rand_fr(n, 1)
    nsc = 1 << args.ref_sc_log_n
    tabs = [util.rand_fr(nsc, 10 + t) for t in range(3)]
    nodes, consts = util.expr_product(3)
    t_msm, t_sc, t_norm = [], [], []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        _, s_norm, s_msm = co.kzg_commit_reference_shape(srs, sc, threads=cores)
        t1 = time.perf_counter()
        co.sumcheck_prove(args.ref_sc_log_n, tabs, nodes, consts, co.fr1(1), co.transcript_new(b"sumcheck_bench"),
                          max_coeffs=8, threads=cores)
        t2 = time.perf_counter()
        if it >= args.warmup:
            t_msm.append(t1 - t0)
            t_sc.append(t2 - t1)
            t_norm.append(s_norm)
    ms = 1e3 * sum(t_msm) / len(t_msm)
    v = n / (ms * 1e-3)
    sc_ms = 1e3 * sum(t_sc) / len(t_sc)
    sc_v = 3 * nsc / (sc_ms * 1e-3)
    sample = (f"KZG::commit of 2^{args.ref_log_n} coefficients (SRS normalisation {1e3 * sum(t_norm) / len(t_norm):.0f} ms "
              f"of the step, single-threaded as in the reference, + Pippenger over {cores} threads); "
              f"sumcheck over three 2^{args.ref_sc_log_n} tables over {cores} threads")
    line = {
        "impl": "reference", "metric": f"KZG MSM points/s (sumcheck field-elems/s in `sumcheck`)", "value": v,
        "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (254-bit modular integer)",
        "data": "synthetic", "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": v, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample,
                         "msm_log_n": args.ref_log_n, "sumcheck_log_n": args.ref_sc_log_n},
        "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "sumcheck": {"value": sc_v, "unit": "field-elems/s", "ms_per_step": sc_ms,
                     "e2e": {"value": sc_v, "unit": "field-elems/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
def cpu_baseline(args):
    """Oracle port timed on the host, rank 0 at N=1 only: 1 thread (faithful: the reference has no rayon / `parallel`)."""
    import numpy as np

    from oracle import coracle as co
    from oracle import pyref as py
    from tests import util

    cores = os.cpu_count() or 1
    n = 1 << args.cpu_log_n
    g = co.g1_to_bytes(py.g1_mul(py.G1_GEN, 7))
    srs = co.srs_generate(g, co.fr1(TAU), n, threads=cores)
    sc = util.rand_fr(n, 1)
    t0 = time.perf_counter()
    _, s_norm, s_msm = co.kzg_commit_reference_shape(srs, sc, threads=1)
    t_commit = time.perf_counter() - t0
    nsc = 1 << args.cpu_sc_log_n
    tabs = [util.rand_fr(nsc, 10 + t) for t in range(3)]
    nodes, consts = util.expr_product(3)
    t0 = time.perf_counter()
    co.sumcheck_prove(args.cpu_sc_log_n, tabs, nodes, consts, co.fr1(1), co.transcript_new(b"sumcheck_bench"),
                      max_coeffs=8, threads=1)
    t_sc = time.perf_counter() - t0
    # BASELINE.json configs[0], literally: KZG commit of a random degree-2^16 polynomial + sumcheck prove over a
    # 2^16-entry degree-3 product, 1 thread
    n1 = 1 << 16
    srs1 = srs[:n1] if srs.shape[0] >= n1 else co.srs_generate(g, co.fr1(TAU), n1, threads=cores)  # kzg.rs:65: <= max degree
    sc1 = util.rand_fr(n1, 2)
    t0 = time.perf_counter()
    co.kzg_commit_reference_shape(srs1, sc1, threads=1)
    t_c1 = time.perf_counter() - t0
    tabs1 = [util.rand_fr(n1, 20 + t) for t in range(3)]
    t0 = time.perf_counter()
    co.sumcheck_prove(16, tabs1, nodes, consts, co.fr1(1), co.transcript_new(b"sumcheck_bench"), max_coeffs=8, threads=1)
    t_s1 = time.perf_counter() - t0
    return {
        "config_1": {"kzg_commit_2_16_s": t_c1, "kzg_commit_points_per_s": n1 / t_c1, "sumcheck_2_16_s": t_s1,
                     "sumcheck_field_elems_per_s": 3 * n1 / t_s1, "cores": 1},
        "value": n / t_commit, "unit": "points/s", "cores": 1, "kind": "port",
        "sample": (f"KZG::commit (kzg.rs:61-73) of 2^{args.cpu_log_n} coefficients, 1 thread: {t_commit:.2f} s "
                   f"({s_norm:.2f} s per-call SRS normalisation + {s_msm:.2f} s Pippenger); sumcheck prove over three "
                   f"2^{args.cpu_sc_log_n} tables, 1 thread: {t_sc:.2f} s"),
        "msm_only_points_per_s": n / s_msm,
        "sumcheck": {"value": 3 * nsc / t_sc, "unit": "field-elems/s", "cores": 1},
        "host_cores_available": cores,
    }


def zc_roofline(rounds_ms, t_loc, hbm_peak, hbm_src, step_ms):
    """Streaming rounds of the eq-factored zero-check (sc_round_zc): the three tables move 128 B per entry over the proof
    as in the sumcheck, the weight tables E_1, E_2, .. (built on the device, then halved by additions in the pass that
    folds the tables) another 64 B per entry of one table."""
    ms = sum(rounds_ms) / len(rounds_ms)
    alg = (SC_BYTES_PER_ELEM * 3 + SC_ZC_WEIGHT_BYTES_PER_ENTRY) * t_loc
    return {"kernel": "sc_round_zc<3> (streaming rounds incl. the weight-table build)", "bound": "hbm",
            "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm_peak,
            "kernel_ms": ms, "kernel_share_of_step": ms / step_ms, "traffic": None, "peak_source": hbm_src,
            "note": "integer-bound like the sumcheck rounds (DESIGN.md section 4): 2 more products per pair for the weight"}


def imad_roofline(stats, imad_peak, step_ms, steps):
    """msm_accumulate over all the MSMs of a multi-MSM step (stats = qz_msm_accumulate_stats over the timed steps):
    executed limb products against the IMAD.WIDE rate measured in this run, and the kernel's share of the step."""
    ms, adds, launches = stats
    if launches == 0 or ms <= 0:
        return None
    return {"kernel": f"msm_accumulate ({launches // steps} launches per step)", "bound": "int32-imad", "unit": "T limb-MAC/s",
            "achieved": adds * 1280 / (ms * 1e-3) / 1e12, "peak": imad_peak / 1e12, "frac": adds * 1280 / (ms * 1e-3) / imad_peak,
            "kernel_ms": ms / steps, "kernel_share_of_step": ms / steps / step_ms, "mixed_additions_per_step": adds / steps,
            "traffic": None, "peak_source": "qz_bench_imad measured in this run"}


def bench_hyperplonk(ctx, q, log_rows, g_bytes, tau_mont, timed_loop, steps, verify=False):
    """BASELINE.json config 5 shape: two traces (Fibonacci, 4 columns; modified Fibonacci, 5 columns padded to 8) of
    2^log_rows rows each, proved with HyperPlonk::prove (zero-check + logup permutation check + MLPCS openings)."""
    import numpy as np

    from quill_zkvm_b200 import hyperplonk as hp

    rows = 1 << log_rows
    In, C = q.VirtualPolyExpr.Input, hp.Const

    def fib():
        c = hp.TransitionCircuit(rows)
        s1, s2 = c.allocate_state_cell(), c.allocate_state_cell()
        c.enforce_boundary_constraint(0, In(s1[0]))
        c.enforce_boundary_constraint(0, hp.Sub(In(s2[0]), C(1)))
        c.enforce_constraint(hp.Sub(In(s2[1]), In(s1[0]) + In(s2[0])))
        c.enforce_constraint(hp.Sub(In(s1[1]), In(s2[0])))
        w = [[0] * rows for _ in range(c.num_cols())]
        a, b = 0, 1
        for r in range(rows):
            w[s1[0]][r], w[s2[0]][r] = a, b
            a, b = b, (a + b) % FR
            w[s1[1]][r], w[s2[1]][r] = a, b
        return c, w

    def modfib():
        c = hp.TransitionCircuit(rows)
        s1, s2 = c.allocate_state_cell(), c.allocate_state_cell()
        t = c.allocate_witness_cell()
        c.enforce_boundary_constraint(0, hp.Sub(In(s1[0]), C(1)))
        c.enforce_boundary_constraint(0, hp.Sub(In(s2[0]), C(1)))
        c.enforce_constraint(hp.Sub(In(t), In(s1[0]) * In(s2[0])))
        c.enforce_constraint(hp.Sub(In(s2[1]), In(s1[0]) + In(t)))
        c.enforce_constraint(hp.Sub(In(s1[1]), In(s2[0])))
        w = [[0] * rows for _ in range(c.num_cols())]
        a, b = 1, 1
        for r in range(rows):
            w[s1[0]][r], w[s2[0]][r] = a, b
            w[t][r] = a * b % FR
            a, b = b, (a + a * b) % FR
            w[s1[1]][r], w[s2[1]][r] = a, b
        return c, w

    def to_table(col):  # canonical bytes via Python, Montgomery conversion on the device; the witness columns the prover
        # receives live in PINNED host memory (as the e2e contract asks of host inputs), so their upload runs at PCIe rate
        raw = np.frombuffer(b"".join(v.to_bytes(32, "little") for v in col), dtype=np.uint8).reshape(-1, 32)
        t = ctx.field_op(0, 4, raw)
        try:
            import torch
            pin = torch.empty(t.size, dtype=torch.uint8, pin_memory=True)
            pins.append(pin)  # keep the allocation alive
            out = pin.numpy().reshape(t.shape)
            out[:] = t
            return out
        except Exception:
            return t

    pins = []

    circuits, witnesses = [], []
    for mk in (fib, modfib):
        c, w = mk()
        circuits.append(c)
        witnesses.append([to_table(col) for col in w])
    max_degree = max(c.num_cols() * c.num_rows() for c in circuits)
    kzg = q.KZG.trusted_setup(ctx, max_degree, g_bytes, tau_mont).precompute()
    prover = hp.HyperPlonk.preprocess(ctx, circuits, kzg)
    out = {}
    out["p"] = prover.prove(kzg, witnesses)  # warm-up proof (untimed)
    ctx.msm_accumulate_stats(1)
    ms, launches = timed_loop(lambda: out.__setitem__("p", prover.prove(kzg, witnesses)), steps, 0)
    acc_stats = ctx.msm_accumulate_stats(-1)
    kzg.srs.free()
    verified = None
    if verify:  # the reference's acceptance criterion (HyperPlonkProof::verify, proof.rs:493-523) restated in oracle/: a
        # CHECK of the timed proof, run after and outside the timed region; nothing on the proving path touches it
        from oracle import pyref as py
        from oracle import verifier as vf
        from tests import util
        t0 = time.perf_counter()
        circuits_py = [py.fibonacci_circuit_and_trace(2)[0], py.modified_fibonacci_circuit_and_trace(2)[0]]
        for c in circuits_py:
            c.num_rows = rows  # the verifier reads only the circuit's shape and constraint expressions
        gx = int.from_bytes(bytes(g_bytes[:32]), "little") * pow(1 << 256, -1, py.FQ) % py.FQ
        gy = int.from_bytes(bytes(g_bytes[32:]), "little") * pow(1 << 256, -1, py.FQ) % py.FQ
        vk = vf.VerifierKey((gx, gy), TAU, g2_scalar=11)
        proof = util.hyperplonk_py(out["p"])
        try:
            verified = vf.hyperplonk_verify(proof, util.hyperplonk_vk_py(prover.trace_vks, circuits_py), vk) == proof["state_end"]
        except ValueError as e:
            verified = False
            print("hyperplonk verifier rejected:", e, file=sys.stderr)
        verify_s = time.perf_counter() - t0
    return {"value": ms * 1e-3, "unit": "s per proof", "rows_per_trace": rows, "traces": 2, "columns": [4, 8],
            "verified": verified, "verified_by": "oracle/verifier.py hyperplonk_verify (restated reference verifier incl. BN254 pairings), "
            f"{verify_s:.1f} s on the host after the timed region" if verify else None,
            "gpu_launches": launches // steps, "workload": "HyperPlonk::prove of Fibonacci + modified-Fibonacci transition circuits "
            "(2 witness commits, 2 zero-checks, 2 logup permutation checks, 2 x (cols + public + 5) MLPCS openings)",
            "final_transcript_state": out["p"].transcript_state.hex(), "_acc_stats": acc_stats, "_ms": ms, "_proof": out["p"]}


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import quill_zkvm_b200 as q
    from quill_zkvm_b200 import parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()
    ctx = q.Context(local, stream.cuda_stream)
    if world > 1:
        parallel.init_comm(ctx)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    FQ = 21888242871839275222246405745257275088696311157297823662689037894645226208583

    def mont(v, mod=FR):
        return np.frombuffer(((v % mod) * (1 << 256) % mod).to_bytes(32, "little"), dtype=np.uint8).copy()

    n = 1 << args.log_n
    lo, hi = parallel.shard_range(n, rank, world)
    n_loc = hi - lo
    g_bytes = np.concatenate([mont(1, FQ), mont(2, FQ)])  # the standard generator (1, 2)
    if lo:
        g_bytes = ctx.g1_mul(g_bytes.reshape(1, 64), mont(pow(TAU, lo, FR)).reshape(1, 32))[0]  # g * tau^lo on the device
    kzg = q.KZG.trusted_setup(ctx, n_loc - 1, g_bytes, mont(TAU))  # SRS shard: g * tau^(lo + i)
    if not args.no_precompute:
        kzg.precompute(args.precompute_bits)  # one-time, like the SRS upload: window multiples 2^(c w) P_i in HBM
    scal_dev = ctx.random_fr(n_loc, shard_seed(0x5155494C4C, lo))  # seeded by GLOBAL index: the same scalars at every N
    pin_scal = torch.empty(n_loc * 32, dtype=torch.uint8, pin_memory=True)
    scal_host = pin_scal.numpy()
    scal_host[:] = scal_dev.download()
    commit = (kzg.msm_sharded if world > 1 else kzg.commit)

    sampler = ClockSampler(local)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_loop(fn, steps, warmup, collect=None):
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                fn()
            barrier()
            l0 = ctx.kernel_launches
            ev0.record(stream)
            for _ in range(steps):
                fn()
                if collect is not None:
                    collect.append(ctx.last_elapsed_ms(1))
            ev1.record(stream)
            barrier()
            return max_over_ranks(ev0.elapsed_time(ev1) / steps), ctx.kernel_launches - l0

    if rank == 0:
        sampler.start()
    # ---- MSM: device-resident scalars (value) and pinned-host scalars (e2e) ----
    acc_ms: list = []
    results = {}
    msm_ms, msm_launches = timed_loop(lambda: results.__setitem__("dev", commit(scal_dev)), args.steps, args.warmup, acc_ms)
    e2e_ms, _ = timed_loop(lambda: results.__setitem__("host", commit(scal_host.reshape(-1, 32))), args.steps, args.warmup)
    assert np.array_equal(results["dev"], results["host"]), "device-resident and host-input commitments differ"
    msm_c, msm_digits, msm_shared, msm_adds = (ctx.last_stat(i) for i in range(4))
    # side leg (N = 1): the same commitment with the opt-in pair levels (QZ_MSM_PAIR_LEVELS, csrc/msm.cu msm_pair_*:
    # batched affine additions ahead of the XYZZ accumulation; DESIGN.md section 3) -- reported beside the default path
    pair_leg = None
    if world == 1 and not args.no_pair_leg:
        os.environ["QZ_MSM_PAIR_LEVELS"] = str(args.pair_levels)
        try:
            pair_acc: list = []
            pair_ms, pair_launches = timed_loop(lambda: results.__setitem__("pair", commit(scal_dev)), args.steps, args.warmup, pair_acc)
            pair_leg = {"ms_per_step": pair_ms, "value": n / (pair_ms * 1e-3), "unit": "points/s", "levels": args.pair_levels,
                        "pair_levels_plus_accumulate_ms": sum(pair_acc) / len(pair_acc),
                        "gpu_launches": pair_launches // args.steps,
                        "same_commitment": bool(np.array_equal(results["pair"], results["dev"])),
                        "default": "off (loses with host scalars: the streamed ranges' sort and the level-1 gathers share the "
                                   "memory system; neutral below 2^23 points)"}
        except Exception as e:  # noqa: BLE001  (a side leg never takes the line down)
            pair_leg = {"error": str(e)[:200]}
        finally:
            os.environ.pop("QZ_MSM_PAIR_LEVELS", None)

    # ---- sumcheck: three 2^log_n tables, degree-3 product ----
    nv = args.log_n
    slo, shi = parallel.table_shard_range(nv, rank, world)
    t_loc = shi - slo
    tabs_dev = [ctx.random_fr(t_loc, shard_seed(1000 * (t + 1), slo)) for t in range(3)]  # global-index seeds
    pins = [torch.empty(t_loc * 32, dtype=torch.uint8, pin_memory=True) for _ in range(3)]
    tabs_host = [p.numpy().reshape(-1, 32) for p in pins]
    for th, td in zip(tabs_host, tabs_dev):
        th[:] = td.download().reshape(-1, 32)
    claimed = mont(0)  # replaced below by the true sum (SURVEY 8d), read off an untimed proof's round-0 polynomial

    def make_store(tabs):
        st = q.VirtualPolynomialStore(nv if world == 1 else nv)
        st.num_vars = nv
        st.polynomials = list(tabs)  # shards when world > 1 (allocate_polynomial would insist on 2^nv entries)
        st.virtual_polys = [product_expr(q, 3)]
        return st

    st_dev, st_host = make_store(tabs_dev), make_store(tabs_host)
    sc_out = {}

    def prove(store, key):
        tr = q.Transcript(b"sumcheck_bench", ctx)
        sc_out[key] = q.SumcheckProof.prove(ctx, nv, store, 0, claimed, tr, sharded=world > 1)
        sc_out[key + "_state"] = tr.state.copy()

    # claimed_sum = the true sum: s_0(0) + s_0(1) = 2 c_0 + c_1 + c_2 + c_3 of the round-0 polynomial, which does not
    # depend on the claim (only the transcript does)
    prove(st_dev, "dev")
    c0 = [int.from_bytes(bytes(c), "little") * pow(1 << 256, -1, FR) % FR for c in sc_out["dev"][0].r_polys[0]]
    true_sum = (2 * c0[0] + sum(c0[1:])) % FR
    claimed[:] = mont(true_sum)
    rounds_ms: list = []
    sc_ms, sc_launches = timed_loop(lambda: prove(st_dev, "dev"), args.steps, args.warmup, rounds_ms)
    sc_e2e_ms, _ = timed_loop(lambda: prove(st_host, "host"), args.steps, args.warmup)
    assert sc_out["dev_state"].tobytes() == sc_out["host_state"].tobytes()
    # zero-check form of the same workload (config 3): eq table built on the device as a fourth factor, degree 4
    def zc_prove():
        tr = q.Transcript(b"zerocheck_bench", ctx)
        sc_out["zc"] = q.ZeroCheckProof.prove(ctx, st_dev, 0, tr, sharded=world > 1)
        sc_out["zc_state"] = tr.state.copy()

    zc_err = None
    try:
        zc_rounds_ms: list = []
        zc_ms, zc_launches = timed_loop(zc_prove, args.steps, args.warmup, zc_rounds_ms)
    except q.QuillError as e:  # an auxiliary leg: report it in the line instead of losing the headline legs above
        if world == 1:
            raise
        zc_ms, zc_launches, zc_err = None, 0, str(e)
    clocks = sampler.stop() if rank == 0 else None

    # (the nvidia-smi sampler is stopped first: its 200 ms polling contends for the driver and slows these
    # launch- and allocation-heavy legs several times over; the headline legs above are one call per step)
    # ---- config 2: KZG commit MSM of 2^20 scalars on one B200 (its own SRS and window table), N = 1 only ----
    msm20 = None
    if world == 1 and args.log_n >= 20 and not args.no_precompute:
        k20 = q.KZG.trusted_setup(ctx, (1 << 20) - 1, g_bytes, mont(TAU)).precompute()
        s20 = ctx.random_fr(1 << 20, shard_seed(0x5155494C4C, 0))
        ms20, l20 = timed_loop(lambda: results.__setitem__("c20", k20.commit(s20)), args.steps, args.warmup)
        msm20 = {"value": (1 << 20) / (ms20 * 1e-3), "unit": "points/s", "ms_per_step": ms20, "gpu_launches": l20 // args.steps,
                 "window_bits": ctx.last_stat(0), "mixed_adds_per_point": ctx.last_stat(1),
                 "commitment_xy": bytes(results["c20"]).hex(),
                 "workload": "KZG::commit of 2^20 random Fr scalars, device-resident, precomputed windows (BASELINE config 2)"}
        s20.free()
        k20.srs.free()

    # ---- config 4: multilinear PCS commit + open (MLEvalProof::prove: 5 MSMs + NTT), N = 1 only ----
    mlpcs = None
    if world == 1 and args.mlpcs_log_n > 0:
        nm = min(args.mlpcs_log_n, args.log_n)
        poly = ctx.random_fr(1 << nm, 777)
        point = np.frombuffer(b"".join(((i * 0x9E3779B97F4A7C15 + 12345) % FR).to_bytes(32, "little") for i in range(nm)),
                              dtype=np.uint8).reshape(nm, 32).copy()

        def commit_open():
            results["ml_c"] = kzg.commit(poly)
            results["ml_o"] = kzg.open_multilinear(poly, point, q.Transcript(b"mlpcs_bench", ctx))

        commit_open()  # warm-up (untimed)
        ctx.msm_accumulate_stats(1)
        ml_ms, ml_launches = timed_loop(commit_open, args.steps, 0)
        ml_stats = ctx.msm_accumulate_stats(-1)
        mlpcs = {"_acc_stats": ml_stats, "_ms": ml_ms, "value": ml_ms * 1e-3, "unit": "s per commit+open", "log_n": nm, "gpu_launches": ml_launches // args.steps,
                 "workload": f"MultilinearPCS::commit + ::open of a 2^{nm}-entry MLE (6 MSMs, eq table, NTT 2^{nm + 1}, 4 quotients)"}
        poly.free()

    # ---- config 5: HyperPlonk prove of two transition-circuit traces (Fibonacci + modified Fibonacci); with N > 1 every
    # rank holds the traces and the full SRS and the MLPCS openings (5 MSMs each) are dealt to the ranks ----
    hplonk = None
    if args.hyperplonk_log_rows > 0:
        hplonk = bench_hyperplonk(ctx, q, args.hyperplonk_log_rows, np.concatenate([mont(1, FQ), mont(2, FQ)]), mont(TAU),
                                  timed_loop, args.steps, verify=rank == 0 and not args.no_verify)
        hplonk["n_gpus"] = world


    # ---- roofline denominators ----
    imad_peak = ctx.bench_imad(0)  # 32x32->64 multiply-accumulates per second (IMAD.WIDE carry chains), measured now
    hbm_peak, hbm_src = peaks()
    out_bytes = nv * (33 * 32 + 4 + 32) + 32 + 32 + 64

    if rank == 0:
        msm_traffic, msm_traffic_src = profile_traffic("msm")
        sc_traffic, sc_traffic_src = profile_traffic("sumcheck")
        acc_avg = sum(acc_ms) / len(acc_ms)
        rounds_avg = sum(rounds_ms) / len(rounds_ms)
        msm_v = n / (msm_ms * 1e-3)
        sc_v = 3 * n / (sc_ms * 1e-3)
        line = {
            "metric": "KZG MSM points/s (sumcheck field-elems/s in `sumcheck`)",
            "value": msm_v, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": msm_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32x8 (254-bit modular integer)", "data": "synthetic",
            "config": workload_config(args, world, bool(ctx.peer_memory)),
            "e2e": {"value": n / (e2e_ms * 1e-3), "unit": "points/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": n_loc * 32 * world, "d2h_bytes_per_step": 64 * world},
            "roofline": {
                # frac = the work the kernel EXECUTES (mixed additions x 1280 limb products) against the measured
                # IMAD.WIDE rate; `canonical` restates SURVEY 8(d)'s 16-window model, which the precomputed-window table
                # beats by doing fewer additions per point (its fraction can exceed 1 and is not a utilisation)
                "kernel": "msm_accumulate", "bound": "int32-imad (integer multiply pipe; not hbm / tensor, see DESIGN.md)",
                "achieved": msm_adds * 1280 / (acc_avg * 1e-3) / 1e12, "peak": imad_peak / 1e12,
                "unit": "T limb-MAC/s", "frac": msm_adds * 1280 / (acc_avg * 1e-3) / imad_peak,
                "model": f"executed work: {msm_digits:.0f} mixed additions per point (c = {msm_c:.0f}"
                         f"{', one shared bucket set over precomputed window multiples' if msm_shared else ''}) x (8M + 2S) x 128 "
                         "limb products = 1280 per addition",
                "canonical": {"model": "SURVEY 8(d): 16 windows x (8M+2S) x 128 limb products = 20480 per point",
                              "achieved": n_loc * MSM_LIMB_PRODUCTS_PER_POINT / (acc_avg * 1e-3) / 1e12,
                              "frac": n_loc * MSM_LIMB_PRODUCTS_PER_POINT / (acc_avg * 1e-3) / imad_peak},
                "kernel_ms": acc_avg, "kernel_share_of_step": acc_avg / msm_ms,
                "traffic": msm_traffic if (world == 1 and args.log_n == 24 and not args.no_precompute) else None,
                "traffic_source": msm_traffic_src if (world == 1 and args.log_n == 24 and not args.no_precompute) else None,
                "peak_source": "qz_bench_imad (IMAD.WIDE.U32 carry chains) measured in this run"},
            "sumcheck": {
                "value": sc_v, "unit": "field-elems/s", "ms_per_step": sc_ms, "gpu_launches": sc_launches // args.steps,
                "e2e": {"value": 3 * n / (sc_e2e_ms * 1e-3), "unit": "field-elems/s", "ms_per_step": sc_e2e_ms,
                        "h2d_bytes_per_step": 3 * t_loc * 32 * world, "d2h_bytes_per_step": out_bytes * world},
                "roofline": {"kernel": "sc_round_prod<3> (streaming rounds, fold fused)", "bound": "hbm",
                             "achieved": SC_BYTES_PER_ELEM * 3 * t_loc / (rounds_avg * 1e-3) / 1e9, "peak": hbm_peak,
                             "unit": "GB/s", "frac": SC_BYTES_PER_ELEM * 3 * t_loc / (rounds_avg * 1e-3) / 1e9 / hbm_peak,
                             "kernel_ms": rounds_avg, "kernel_share_of_step": rounds_avg / sc_ms,
                             "traffic": sc_traffic if (world == 1 and args.log_n == 24) else None,
                             "traffic_source": sc_traffic_src if (world == 1 and args.log_n == 24) else None,
                             "peak_source": hbm_src},
            },
            "gpu_launches": msm_launches // args.steps,
            "clocks": clocks,
            # N-invariance evidence: inputs are seeded by global index, so these must be identical at N = 1, 2, 4, 8
            "digests": {"commitment_xy": bytes(results["dev"]).hex(),
                        "commitment_serialized": ctx.g1_serialize(results["dev"]).hex(),
                        "sumcheck_claimed_sum": "%064x" % true_sum,
                        "sumcheck_final_transcript_state": sc_out["dev_state"].tobytes().hex(),
                        "sumcheck_evaluation": bytes(sc_out["dev"][1].evaluation).hex(),
                        "zerocheck_final_transcript_state": sc_out["zc_state"].tobytes().hex() if "zc_state" in sc_out else None},
        }
        # parity carried into every run: the digests of the default workload are pinned against the oracle by
        # tests/test_gpu_config_sizes.py::test_bench_digests_pinned_by_the_oracle; any N must reproduce them
        gpath = os.path.join(ROOT, "tests", "golden", f"bench_digests_2_{args.log_n}.json")
        if os.path.exists(gpath):
            gold = json.load(open(gpath))["digests"]
            line["digests_match_golden"] = all(line["digests"].get(k) == v for k, v in gold.items() if line["digests"].get(k) is not None)
            line["digests_golden"] = os.path.relpath(gpath, ROOT)
        if zc_err is not None:
            line["zerocheck"] = {"error": zc_err}
        if zc_ms is not None:
            line["zerocheck"] = {"value": 3 * n / (zc_ms * 1e-3), "unit": "field-elems/s", "ms_per_step": zc_ms,
                                 "gpu_launches": zc_launches // args.steps,
                                 "roofline": zc_roofline(zc_rounds_ms, t_loc, hbm_peak, hbm_src, zc_ms),
                                 "workload": f"ZeroCheckProof::prove of f*g*e over three 2^{args.log_n}-entry tables: z drawn on the device, "
                                             "eq-factored rounds (degree-3 sums weighted by the eq table of the remaining variables, "
                                             "times the round's linear eq factor)"}
        if msm20:
            line["msm_2_20"] = msm20
        if pair_leg:
            line["msm_pair_levels"] = pair_leg
        if mlpcs:
            mlpcs["roofline"] = imad_roofline(mlpcs.pop("_acc_stats"), imad_peak, mlpcs.pop("_ms"), args.steps)
            line["mlpcs_commit_open"] = mlpcs
        hp_proof = None
        if hplonk:
            hp_proof = hplonk.pop("_proof")
            hplonk["roofline"] = imad_roofline(hplonk.pop("_acc_stats"), imad_peak, hplonk.pop("_ms"), args.steps)
            line["hyperplonk_prove"] = hplonk
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line))
        if args.dump_outputs:
            # what each timed leg returned to its caller in its last step
            outputs = {"msm_commitment": results["dev"], "msm_commitment_host_scalars": results["host"],
                       "msm_pair_levels_commitment": results.get("pair") if pair_leg and "error" not in pair_leg else None,
                       "sumcheck_proof": sc_out["dev"], "sumcheck_transcript_state": sc_out["dev_state"],
                       "sumcheck_proof_host_tables": sc_out["host"],
                       "sumcheck_transcript_state_host_tables": sc_out["host_state"],
                       "zerocheck_proof": sc_out.get("zc") if zc_err is None else None,
                       "zerocheck_transcript_state": sc_out.get("zc_state") if zc_err is None else None,
                       "msm_2_20_commitment": results.get("c20"),
                       "mlpcs_commitment": results.get("ml_c"), "mlpcs_opening": results.get("ml_o"),
                       "hyperplonk_proof": hp_proof}
            dump_outputs(args.dump_outputs, {k: v for k, v in outputs.items() if v is not None})
    for b in tabs_dev + [scal_dev]:
        b.free()
    kzg.srs.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=24, help="problem size 2^log_n (BASELINE.json metric: 24)")
    ap.add_argument("--cpu-log-n", type=int, default=18, help="CPU baseline MSM sample size")
    ap.add_argument("--cpu-sc-log-n", type=int, default=20, help="CPU baseline sumcheck sample size")
    ap.add_argument("--ref-log-n", type=int, default=18, help="--impl reference: MSM sample size per step")
    ap.add_argument("--ref-sc-log-n", type=int, default=20, help="--impl reference: sumcheck sample size per step")
    ap.add_argument("--mlpcs-log-n", type=int, default=22, help="config 4: MLPCS commit+open size (0 = skip)")
    ap.add_argument("--hyperplonk-log-rows", type=int, default=20,
                    help="config 5: rows per trace of the two-trace HyperPlonk proof (0 = skip; BASELINE names 20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pair-leg", action="store_true", help="skip the side leg with the MSM pair levels switched on")
    ap.add_argument("--pair-levels", type=int, default=3, help="QZ_MSM_PAIR_LEVELS of the side leg")
    ap.add_argument("--no-verify", action="store_true", help="skip the verifier check of the HyperPlonk proof")
    ap.add_argument("--no-precompute", action="store_true", help="MSM without the precomputed window multiples")
    ap.add_argument("--precompute-bits", type=int, default=0, help="window bits of the precomputed table (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what every timed leg returned in "
                    "its last step as DIR/<name>.npy (float64 32-bit limbs; the inputs are seeded, so runs with the same "
                    "arguments compare output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
