#!/usr/bin/env python
"""bench.py — proofs/s on the BASELINE.json workload (Groth16, BN254, domain 2^20 synthetic chain circuit).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--log-n 20] [--impl reference]
                    [--workload groth16|plonk|fflonk] [--curve bn128|bls12381] [--dump-outputs DIR]

One step = one proof.  N = 1: the whole prover on one B200.  N > 1 (torchrun, one rank per GPU): every MSM is sharded
by point range across the ranks (north star / SURVEY §8e) and the three A/B/C transform chains run on different ranks;
the exchange steps run inside libsnarkb200.so over NCCL.  `value` is the sharded single-proof rate (strong scaling);
`replicas` reports N independent provers beside it.

JSON keys follow the task contract; extra keys: roofline (dominant kernel vs measured HBM peak), roofline_int (same
kernel vs the calibrated integer-pipe peak — the bound that actually applies, SURVEY §8d), cpu_baseline (the oracle's
restated reference prover on the host cores, same key, full size), breakdown_ms (per kernel class, serialised proof),
oracle_match (the timed workload's proof equals the CPU oracle's: committed hash and, at N = 1, a live comparison).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="groth16", choices=["groth16", "plonk", "fflonk"])
    ap.add_argument("--curve", default=None, choices=["bn128", "bls12381"], help="default: bn128 (groth16, fflonk), bls12381 (plonk: BASELINE config #5)")
    ap.add_argument("--cpu-log-n", type=int, default=0, help="log2 domain of the CPU arm's sample (0 = the full workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--witness-like", action="store_true", help="witness distribution of real circuits (SURVEY 8d): 50%% zeros, 25%% ones, 25%% uniform")
    ap.add_argument("--tune", action="append", default=[], help="experimental kernel-variant switch k=v (sb_set_tuning), e.g. 1=1 = legacy bucket reduction")
    ap.add_argument("--mode", default="shard", choices=["shard", "replicas"], help="N > 1: which number is `value` (the other one is reported beside it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the proof of the last timed step to DIR/proof.npy (B200 arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the B200 arm's outputs; the reference arm has none to write")
    return a


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples = []
        self.stop = False
        self.index = index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.samples.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for i, nm in enumerate(names):
                if len(s) > 3 + i and s[3 + i].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ host cores
def host_cores() -> int:
    """Threads the CPU arm may use: the affinity mask, capped by a cgroup CPU quota if one is set.  torchrun exports
    OMP_NUM_THREADS=1 to its children; the CPU arm ignores it (it is the arm's whole job to use the host)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    return n


def proof_hash(proof_obj) -> str:
    """sha256 of the canonical JSON text of the proof object (SURVEY §8c: proof.json text identical)."""
    return hashlib.sha256(json.dumps(proof_obj, sort_keys=True, separators=(",", ":")).encode()).hexdigest()


def dump_outputs(out_dir: str | None, proof: np.ndarray) -> None:
    """--dump-outputs: the proof bytes a prove call returns (affine points and field elements in the library's Montgomery
    form), one float64 per byte so that the values are exact.  The inputs are fixed by the flags, so two builds given the
    same flags must write the same file."""
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "proof.npy"), np.asarray(proof, np.uint8).astype(np.float64))


def golden_hash(workload: str, curve: str, L: int, witness_like: bool):
    if workload != "groth16" or curve != "bn128" or witness_like:
        return None
    try:
        tab = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_proof_hashes.json")))
        return tab["groth16_bn128_chain_r5_s7"].get(str(L))
    except Exception:
        return None


def workload_config(L: int, world: int, witness_like: bool) -> dict:
    """`config` of the JSON line; the B200 arm and the reference arm print the same dictionary for the same flags."""
    return {"workload": f"groth16 prove, BN254, synthetic chain R1CS, domain 2^{L} (nVars 2^{L}, {2 * ((1 << L) - 3) + 2} QAP coefficients); 4 G1 MSM + 1 G2 MSM of 2^{L} points, 6 NTT of 2^{L}",
            "curve": "bn128", "witness": "witness-like (50% zeros, 25% ones)" if witness_like else "uniform field elements (chain circuit)",
            "parallelism": f"one proof over {world} GPUs: MSM point-range shards, A/B/C transform chains on ranks 0..2, NCCL exchange inside the library" if world > 1 else "single GPU",
            "l2_policy": "inputs larger than L2 (384 MiB of bases + 32 MiB witness per proof vs 126 MB L2)"}


# ------------------------------------------------------------------------------------------------ reference arm / cpu baseline
def oracle_groth16(log_n: int, steps: int, warmup: int, zkey: bytes | None = None, witness: np.ndarray | None = None):
    """Times the oracle's restatement of groth16_prove.js (reference algorithms: pTSizes Pippenger, radix-2 DIT NTT,
    serial buildABC1) on all host cores.  Without a zkey the key is built with the oracle's own point generator (same
    points as sb_gen_points), so this arm needs no GPU and proves the very key the B200 arm proves."""
    from oracle import oracle as O
    from snarkjs_b200 import synth
    ci = O.CURVES[O.BN254]
    cores = host_cores()
    O.lib().or_set_threads(cores)
    if zkey is None:
        zkey = synth.groth16_zkey_image(ci.q, ci.r, 32, log_n, lambda g, s, k: O.gen_points(O.BN254, g, s, k).tobytes())
    if witness is None:
        witness = synth.chain_witness(ci.r, log_n)
    wt = synth.wtns_container(ci.r, witness)
    r, s = ci.fr_to_mont(5), ci.fr_to_mont(7)
    proof = None
    for _ in range(warmup):
        proof, _ = O.groth16_prove(zkey, wt, r, s, concurrency=cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        proof, _ = O.groth16_prove(zkey, wt, r, s, concurrency=cores)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return dt, cores, proof


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "groth16":
        import bench_plonk
        return bench_plonk.run_reference(args)
    L = args.cpu_log_n or args.log_n
    steps = max(1, min(args.steps, 2))
    warm = 1 if args.warmup > 0 else 0
    dt, cores, proof = oracle_groth16(L, steps, warm)
    scale = (1 << args.log_n) / (1 << L)
    val = 1.0 / (dt * scale)
    sample = f"oracle groth16_prove (restated reference prover) on the chain circuit at domain 2^{L}: {steps} proofs after {warm} warm-up, {dt:.3f} s each, {cores} OpenMP threads"
    if scale != 1:
        sample += f", scaled x{scale:g} (linear in constraints) to domain 2^{args.log_n}"
    ph = proof_hash(proof)
    gold = golden_hash("groth16", "bn128", L, False)
    line = {"metric": "groth16_proofs_per_sec", "value": val, "unit": "proofs/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt * scale * 1e3, "higher_is_better": True, "scaling": "weak" if args.mode == "replicas" else "strong", "vs_baseline": None,
            "dtype": "u32x8 (256-bit modular integers)", "data": "synthetic", "impl": "reference",
            "config": workload_config(args.log_n, args.gpus, False), "same_key_as_b200_arm": True,
            "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample, "nproc": os.cpu_count()},
            "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "proof_sha256": ph, "oracle_match": (ph == gold) if gold else None}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import snarkjs_b200
    from snarkjs_b200 import groth16, synth
    from snarkjs_b200.curve import _ptr

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    L = args.log_n
    curve = snarkjs_b200.getCurveFromName("bn128", device=local)
    for kv in args.tune:
        k_, v_ = kv.split("=")
        curve.lib.sb_set_tuning(int(k_), int(v_))
    peak_modmul = curve.lib.sb_calibrate(curve.handle, 1) if rank == 0 else 0.0
    peak_imad = curve.lib.sb_calibrate(curve.handle, 0) if rank == 0 else 0.0
    t0 = time.perf_counter()
    zkey = synth.synth_groth16_zkey(curve, L, seed=1)
    pk = groth16.ProvingKey(zkey, curve=curve, shard=rank, n_shards=world)
    t_setup = time.perf_counter() - t0
    wit_np = synth.chain_witness(curve.r, L)
    if args.witness_like:
        wit_np = synth.witness_like(wit_np)
    wit = torch.from_numpy(wit_np.copy()).pin_memory()           # pinned host witness: the e2e input
    wptr = wit.data_ptr()
    nwit = wit.numel() // 32
    r = (5 * (1 << 256) % curve.r).to_bytes(32, "little")
    s = (7 * (1 << 256) % curve.r).to_bytes(32, "little")
    proof = np.empty(8 * curve.n8q, np.uint8)
    lib, h = curve.lib, curve.handle
    if world > 1:
        # the library's own communicator (NCCL inside libsnarkb200.so): torch.distributed only carries the 128-byte id
        idt = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            idt = torch.frombuffer(bytearray(curve.comm_unique_id()), dtype=torch.uint8).clone()
        idt = idt.cuda()
        dist.broadcast(idt, 0)
        curve.comm_init(world, rank, bytes(idt.cpu().numpy().tobytes()))

    def step(resident: bool):
        if world == 1:
            if resident:
                curve.check(lib.sb_groth16_prove_resident(h, pk.handle, r, s, _ptr(proof)))
            else:
                curve.check(lib.sb_groth16_prove(h, pk.handle, wptr, nwit, r, s, _ptr(proof)))
        else:   # one collective call: witness slices + all-gather, chain exchange, partial all-gather all inside the library
            curve.check(lib.sb_groth16_prove_dist(h, pk.handle, None if resident else wptr, nwit, r, s, _ptr(proof) if rank == 0 else None))

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        t = time.perf_counter()
        for _ in range(steps):
            fn()
        sync()
        dt = time.perf_counter() - t
        if dist is not None:
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        return dt

    for _ in range(max(args.warmup, 3)):
        step(False)
    l0 = curve.launch_count()
    with ClockSampler(local) as cs:
        dt_e2e = timed(lambda: step(False), args.steps)
        proof_e2e = proof.copy()
        l1 = curve.launch_count()
        # per-stage breakdown of the last e2e step (CUDA events on the library's stream)
        brk = {"h2d_witness": curve.last_ms(1), "device_total": curve.last_ms(0)}
        dt_res = timed(lambda: step(True), args.steps)
        proof_res = proof.copy()
    clocks = cs.summary()
    replicas = None
    if world > 1:
        # N independent provers (SURVEY §8e "8 independent provers"): every rank proves its own copy of the workload with
        # a full key; no exchange at all.  Reported beside the sharded single-proof rate.
        pk_full = groth16.ProvingKey(zkey, curve=curve)
        rproof = np.empty(8 * curve.n8q, np.uint8)

        def rstep(resident):
            if resident:
                curve.check(lib.sb_groth16_prove_resident(h, pk_full.handle, r, s, _ptr(rproof)))
            else:
                curve.check(lib.sb_groth16_prove(h, pk_full.handle, wptr, nwit, r, s, _ptr(rproof)))
        for _ in range(3):
            rstep(False)
        dt_r_e2e = timed(lambda: rstep(False), args.steps)
        dt_r_res = timed(lambda: rstep(True), args.steps)
        same = torch.tensor([1 if (rank != 0 or np.array_equal(rproof, proof_e2e)) else 0], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        replicas = {"value": world * args.steps / dt_r_res, "unit": "proofs/s", "e2e": world * args.steps / dt_r_e2e,
                    "ms_per_proof_per_gpu": dt_r_res / args.steps * 1e3, "scaling": "weak",
                    "same_proof_as_sharded": bool(same.item()),
                    "note": f"{world} independent provers, one full key per GPU, each proving its own copy of the workload"}
        pk_full.release()
    # kernel-level numbers for the rooflines: one extra proof with every stream serialised (in the overlapped schedule
    # kernels share the SMs, so their event-bracketed durations are not per-kernel costs)
    lib.sb_set_tuning(2, 1)
    for _ in range(2):
        step(True)
    acc = {"g1_ms": lib.sb_last_stat(h, 0), "g2_ms": lib.sb_last_stat(h, 1), "g1_launches": lib.sb_last_stat(h, 2),
           "g2_launches": lib.sb_last_stat(h, 3), "g1_entries": lib.sb_last_stat(h, 4), "g2_entries": lib.sb_last_stat(h, 5)}
    brk["serialised_device_total"] = curve.last_ms(0)
    try:
        names = ["digits_sort", "accumulate_g1", "accumulate_g2", "fold", "bucket_reduce", "qap_rows", "ntt_passes", "join_abc"]
        for i, nm in enumerate(names):
            brk[nm] = lib.sb_last_stat(h, 8 + i)
    except Exception:
        pass
    lib.sb_set_tuning(2, 0)
    assert np.array_equal(proof, proof_e2e), "resident and e2e proofs differ"

    if rank != 0:
        return
    # dominant kernel: the bucket-accumulation kernel (XYZZ mixed add 8M+2S per entry; G2: 8 Fq2 mul + 2 Fq2 sqr).  Algorithmic bytes per entry: 8 B sorted (key,val) +
    # one affine base (64 / 128 B), plus the bucket array written once.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    # multiply-equivalents per entry from the wide-MAC count (one 8-limb Montgomery multiply = 2*64 + 8 = 136 wide MACs, a
    # dual-product multiply = 3*64 + 8 = 200): G1 mixed add = 8 multiplies + 1 dual = 1288 MACs = 9.47; G2 = 16 duals + 4
    # multiplies = 3744 MACs = 27.53
    g1_mod = acc["g1_entries"] * (1288.0 / 136.0)
    g2_mod = acc["g2_entries"] * (3744.0 / 136.0)
    dom = "g2" if acc["g2_ms"] >= acc["g1_ms"] / max(acc["g1_launches"], 1) else "g1"
    traffic = None
    try:   # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = tj.get("k_accumulate_g2" if dom == "g2" else "k_accumulate_g1", {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    if dom == "g2":
        k_ms, k_launch, k_entries, k_mod, base_b, name = acc["g2_ms"], acc["g2_launches"], acc["g2_entries"], g2_mod, 128, "k_accumulate<Fp2<BnFq>> (G2 bucket accumulation)"
    else:
        k_ms, k_launch, k_entries, k_mod, base_b, name = acc["g1_ms"], acc["g1_launches"], acc["g1_entries"], g1_mod, 64, "k_accumulate<Fp<BnFq>> (G1 bucket accumulation)"
    k_launch = max(k_launch, 1)
    alg_bytes = (k_entries * (8 + base_b)) / k_launch
    avg_ms = k_ms / k_launch
    ach_gbs = alg_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    ach_mod = (k_mod / k_launch) / (avg_ms * 1e-3) if avg_ms > 0 else 0.0
    all_mod = (g1_mod + g2_mod)
    all_ms = acc["g1_ms"] + acc["g2_ms"]
    pobj = groth16.proof_to_object(curve, proof.tobytes())
    ph = proof_hash(pobj)
    gold = golden_hash("groth16", "bn128", L, args.witness_like)
    line = {
        "metric": "groth16_proofs_per_sec", "value": args.steps / dt_res, "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dt_res / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak" if args.mode == "replicas" else "strong", "vs_baseline": None,   # one label for the whole 1..N sweep: the sharded proof is the same total work at every N
        "dtype": "u32x8 (256-bit modular integers, 32-bit limbs)", "data": "synthetic",
        "config": workload_config(L, world, args.witness_like),
        "e2e": {"value": args.steps / dt_e2e, "unit": "proofs/s", "h2d_bytes_per_step": int(nwit * 32), "d2h_bytes_per_step": int(proof.size),
                "ms_per_step": dt_e2e / args.steps * 1e3, "api": ("sb_groth16_prove_dist (pinned host witness on every rank, 1/N uploaded per rank -> affine proof bytes on rank 0's host)" if world > 1 else "sb_groth16_prove (pinned host witness -> affine proof bytes on host)")},
        "gpu_launches": int(l1 - l0),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": name, "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak if hbm_peak else None,
                     "traffic": traffic, "peak_source": peak_src, "launch_ms": avg_ms, "algorithmic_bytes_per_launch": alg_bytes,
                     "note": "integer-pipe bound kernel: see roofline_int; HBM fraction is low by construction"},
        "roofline_int": {"bound": "int32 IMAD pipe (modmul-bound roofline, SURVEY 8d)", "kernel": name, "achieved": ach_mod / 1e9, "unit": "G Fq-modmul/s",
                         "peak": peak_modmul / 1e9, "frac": ach_mod / peak_modmul if peak_modmul > 0 else None,
                         "peak_source": "sb_calibrate(1): four independent per-thread BN254 Fq Montgomery-multiply chains (IMAD.WIDE.U32.X issue-bound), measured on this GPU in this run",
                         "imad_wide_per_s": peak_imad, "imad_wide_per_clk_per_sm": (peak_imad / 148.0 / (clocks["sm_mhz"] * 1e6)) if clocks.get("sm_mhz") else None,
                         "all_accumulate_kernels_frac": (all_mod / (all_ms * 1e-3)) / peak_modmul if (all_ms > 0 and peak_modmul > 0) else None},
        "breakdown_ms": brk, "accumulate": acc, "setup_s": t_setup, "replicas": replicas,
        "proof_sha256": ph,                      # same inputs => same bytes at every N
        "oracle_match": (ph == gold) if gold else None,
        "oracle_match_source": "tests/golden/bench_proof_hashes.json (CPU oracle proof of this key, made by tests/golden/make_bench_hashes.py)" if gold else "no committed oracle hash for this size",
    }
    if gold and ph != gold:
        line["oracle_mismatch"] = {"got": ph, "want": gold}
    if args.mode == "replicas" and replicas:      # report the independent-prover rate as `value`, the sharded one beside it
        line["sharded"] = {"value": line["value"], "e2e": line["e2e"]["value"], "ms_per_step": line["ms_per_step"], "scaling": "strong"}
        line["value"], line["ms_per_step"], line["scaling"] = replicas["value"], 1e3 / replicas["value"], "weak"
        line["e2e"]["value"] = replicas["e2e"]
    if not args.no_cpu_baseline and world == 1:
        try:   # the CPU oracle proves the SAME key and witness (full size unless --cpu-log-n): baseline + live parity check
            Ls = args.cpu_log_n or L
            if Ls == L:
                dt, cores, oproof = oracle_groth16(L, 1, 0, zkey=zkey, witness=wit_np)
                line["oracle_live_match"] = (oproof == pobj)
                sample = f"oracle (restated reference prover) proving the same key and witness at domain 2^{L}: one proof, {dt:.3f} s, {cores} OpenMP threads"
                val = 1.0 / dt
            else:
                dt, cores, _ = oracle_groth16(Ls, 1, 0)
                scale = (1 << L) / (1 << Ls)
                sample = f"oracle (restated reference prover) on the chain circuit at domain 2^{Ls}: {dt:.3f} s, {cores} OpenMP threads, scaled x{scale:g} linearly to 2^{L}"
                val = 1.0 / (dt * scale)
            line["cpu_baseline"] = {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample, "nproc": os.cpu_count()}
        except Exception as e:  # the baseline is a report, never a reason to lose the GPU number
            line["cpu_baseline"] = {"error": str(e)}
    print(json.dumps(line))
    dump_outputs(args.dump_outputs, proof_res)
    pk.release()
    curve.terminate()
    if dist is not None:
        dist.destroy_process_group()
    if gold and ph != gold:
        sys.exit("proof does not match the CPU oracle's (tests/golden/bench_proof_hashes.json)")


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload != "groth16":
        import bench_plonk
        bench_plonk.run_b200(a)
    else:
        run_b200(a)
