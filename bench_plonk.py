"""bench_plonk.py — BASELINE.json config #5: `plonk prove` / `fflonk prove` at domain 2^L on one B200 (bench.py --workload
plonk|fflonk).  Same JSON contract as bench.py's Groth16 line.

One step = one proof of the synthetic chain circuit (snarkjs_b200/synth.py: 2^L - 6 gates, ~n/4 additions on two dependency
levels, one public signal; the PTau section holds pseudo-random valid points).  `value` = proofs/s with the witness
already in HBM (sb_*_prove_resident), `e2e` = sb_*_prove from a pinned host witness to proof bytes on the host.  PLONK runs on
BLS12-381 by default (config #5), fflonk on BN254 (the only curve the reference's fflonk supports, src/fflonk_setup.js:534-557).

Reference arm (--impl reference) and cpu_baseline: the same control flow and per-element functions compiled with g++ -O3
-fopenmp behind the host backend of tests/host/ (NTT and MSM from the CPU oracle, OpenMP over all host cores): a C++ port of the
prover, "kind": "port".  It proves the same key (built with the oracle's NTT instead of the library's: same bytes, checked
in tests/test_py_mirror.py), so at N = 1 the B200 proof is compared with it byte for byte (`cpu_live_match`).
"""
from __future__ import annotations

import ctypes
import functools
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_BLINDERS = {"plonk": 11, "fflonk": 9}


def _curve_name(args) -> str:
    if args.workload == "fflonk":
        return "bn128"
    return args.curve or "bls12381"


def _blinders(r: int, proto: str) -> bytes:
    return b"".join((((7 + i) << 256) % r).to_bytes(32, "little") for i in range(N_BLINDERS[proto]))


def _proof_bytes(proto: str, n8q: int) -> int:
    return 9 * 2 * n8q + 6 * 32 if proto == "plonk" else 4 * 2 * n8q + 16 * 32


# ------------------------------------------------------------------------------------------------ CPU port (reference arm)
@functools.lru_cache(maxsize=None)
def host_flow_lib(proto: str):
    """tests/host/host_<proto>.cpp compiled with OpenMP, once per process, in a temporary directory: the source tree may be
    read-only, and a -march=native build must not be reused on another host."""
    src = os.path.join(ROOT, "tests", "host", f"host_{proto}.cpp")
    with tempfile.TemporaryDirectory(prefix="snarkjs_b200_host_") as tmp:
        so = os.path.join(tmp, f"libhost{proto}_omp.so")
        subprocess.check_call(["g++", "-O3", "-march=native", "-fopenmp", "-std=c++17", "-shared", "-fPIC", "-o", so, src, "-ldl"])
        lib = ctypes.CDLL(so)     # stays mapped after the file is removed
    fn = getattr(lib, f"hp_{proto}_prove")
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int]
    return fn


def oracle_key(proto: str, curve_name: str, L: int):
    """(zkey bytes, witness uint8 array) built with the CPU oracle behind synth's callables (no GPU needed)."""
    from oracle import oracle as O
    from snarkjs_b200 import synth
    ci = O.CURVES[O.BN254 if curve_name == "bn128" else O.BLS12_381]
    cb = (lambda p: ci.fr_from_mont(O.fr_root(ci.id, p)), lambda b, inv: O.fr_fft(ci.id, b, inv), lambda b, f, i: O.fr_batch_apply_key(ci.id, b, f, i),
          lambda grp, sd, k: O.gen_points(ci.id, grp, sd, k), ci.g2_affine_bytes(ci.g2))
    circ = synth.plonk_chain_circuit((1 << L) - 6, ci.r)
    image = synth.plonk_zkey_image if proto == "plonk" else synth.fflonk_zkey_image
    return image(ci.q, ci.r, ci.n8q, circ, *cb), circ["witness"], ci


def cpu_prove(proto: str, zkey, witness: np.ndarray, r: int, n8q: int, cores: int):
    """One proof by the CPU port; returns (seconds, raw proof bytes)."""
    from oracle import oracle as O
    O.lib().or_set_threads(cores)
    os.environ["OMP_NUM_THREADS"] = str(cores)          # torchrun exports 1; the CPU arm's whole job is to use the host
    fn = host_flow_lib(proto)
    zk = np.frombuffer(zkey, np.uint8) if not isinstance(zkey, np.ndarray) else zkey
    out = np.zeros(_proof_bytes(proto, n8q), np.uint8)
    err = ctypes.create_string_buffer(256)
    t = time.perf_counter()
    rc = fn(O.build().encode(), zk.ctypes.data, zk.size, witness.ctypes.data, witness.size // 32, _blinders(r, proto), out.ctypes.data, err, 256)
    dt = time.perf_counter() - t
    if rc != 0:
        raise RuntimeError(f"host flow failed rc={rc}: {err.value.decode()}")
    return dt, out.tobytes()


def _proof_object(proto: str, curve_ns, raw: bytes):
    from snarkjs_b200 import fflonk, plonk
    return (plonk if proto == "plonk" else fflonk).proof_to_object(curve_ns, raw)


def golden_hash(proto: str, curve_name: str, L: int):
    try:
        tab = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_proof_hashes.json")))
        return tab.get(f"{proto}_{curve_name}_chain_b7", {}).get(str(L))
    except Exception:
        return None


def run_reference(args):
    from types import SimpleNamespace
    from bench import host_cores, proof_hash
    proto, cname = args.workload, _curve_name(args)
    L = args.cpu_log_n or args.log_n
    cores = host_cores()
    from oracle import oracle as O
    O.lib().or_set_threads(cores)
    t0 = time.perf_counter()
    zkey, wit, ci = oracle_key(proto, cname, L)
    t_setup = time.perf_counter() - t0
    steps = max(1, min(args.steps, 2))
    warm = 1 if (args.warmup > 0 and L <= 16) else 0
    raw = None
    for _ in range(warm):
        cpu_prove(proto, zkey, wit, ci.r, ci.n8q, cores)
    t = time.perf_counter()
    for _ in range(steps):
        _, raw = cpu_prove(proto, zkey, wit, ci.r, ci.n8q, cores)
    dt = (time.perf_counter() - t) / steps
    scale = (1 << args.log_n) / (1 << L)
    val = 1.0 / (dt * scale)
    ns = SimpleNamespace(name=cname, n8q=ci.n8q, q=ci.q, r=ci.r)
    ph = proof_hash(_proof_object(proto, ns, raw))
    gold = golden_hash(proto, cname, L)
    sample = f"C++ port of {proto} prove (product control flow + element functions on a host backend, oracle NTT/MSM) on the chain circuit at domain 2^{L}: {steps} proof(s) after {warm} warm-up, {dt:.2f} s each, {cores} OpenMP threads"
    if scale != 1:
        sample += f", scaled x{scale:g} (linear in gates) to domain 2^{args.log_n}"
    line = {"metric": f"{proto}_proofs_per_sec", "value": val, "unit": "proofs/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt * scale * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 scalar field / u32x%d base field (modular integers)" % (ci.n8q // 4), "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{proto} prove, {cname}, synthetic chain circuit, domain 2^{args.log_n}", "curve": cname, "same_key_as_b200_arm": True},
            "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample, "nproc": os.cpu_count()},
            "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "proof_sha256": ph, "oracle_match": (ph == gold) if gold else None, "setup_s": t_setup}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import snarkjs_b200
    from snarkjs_b200 import fflonk, plonk, synth
    from snarkjs_b200.curve import _ptr
    from bench import ClockSampler, dump_outputs, host_cores, proof_hash

    proto, cname, L = args.workload, _curve_name(args), args.log_n
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:    # the rounds are serialised by the transcript: N GPUs = N independent provers (replicas), no exchange
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    curve = snarkjs_b200.getCurveFromName(cname, device=local)
    lib, h = curve.lib, curve.handle
    for kv in args.tune:
        k_, v_ = kv.split("=")
        lib.sb_set_tuning(int(k_), int(v_))
    peak_modmul_bn = lib.sb_calibrate(h, 1) if rank == 0 else 0.0
    t0 = time.perf_counter()
    mod = plonk if proto == "plonk" else fflonk
    zkey, wit_np = (synth.synth_plonk_zkey if proto == "plonk" else synth.synth_fflonk_zkey)(curve, L)
    t_key = time.perf_counter() - t0
    t0 = time.perf_counter()
    pk = mod.ProvingKey(zkey, curve)
    t_load = time.perf_counter() - t0
    zkey_len = len(zkey)
    if not (rank == 0 and world == 1 and not args.no_cpu_baseline):
        del zkey
    wit = torch.from_numpy(wit_np.copy()).pin_memory()
    wptr, nwit = wit.data_ptr(), wit.numel() // 32
    bl = _blinders(curve.r, proto)
    proof = np.empty(_proof_bytes(proto, curve.n8q), np.uint8)
    prove = lib.sb_plonk_prove if proto == "plonk" else lib.sb_fflonk_prove
    prove_res = lib.sb_plonk_prove_resident if proto == "plonk" else lib.sb_fflonk_prove_resident

    def step(resident):
        if resident:
            curve.check(prove_res(h, pk.handle, bl, _ptr(proof)))
        else:
            curve.check(prove(h, pk.handle, wptr, nwit, bl, _ptr(proof)))

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

    W = max(args.warmup, 3)
    for _ in range(W):
        step(False)
    l0 = curve.launch_count()
    with ClockSampler(local) as cs:
        dt_e2e = timed(lambda: step(False), args.steps)
        proof_e2e = proof.copy()
        l1 = curve.launch_count()
        dt_res = timed(lambda: step(True), args.steps)
    clocks = cs.summary()
    assert np.array_equal(proof, proof_e2e), "resident and e2e proofs differ"
    # per-class device times of the last proof (the flow runs on one stream: event-bracketed durations are per-kernel costs)
    names = ["digits_sort", "accumulate_g1", "accumulate_g2", "fold", "bucket_reduce", "qap_rows", "ntt_passes", "join_abc"]
    brk = {"device_total": curve.last_ms(0), "rounds_1_to_5_host_clock": [curve.last_ms(i) for i in range(1, 6)]}
    for i, nm in enumerate(names):
        v = lib.sb_last_stat(h, 8 + i)
        if v:
            brk[nm] = v
    brk["elementwise_scans_transcript_and_syncs"] = brk["device_total"] - sum(v for k, v in brk.items() if k in names)
    acc_ms, acc_launches, acc_entries = lib.sb_last_stat(h, 0), max(lib.sb_last_stat(h, 2), 1.0), lib.sb_last_stat(h, 4)
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    n32 = curve.n8q // 4
    # dominant kernel: G1 bucket accumulation over the PTau window table (8 B entry + one affine base per entry)
    alg_bytes = acc_entries * (8 + 2 * curve.n8q) / acc_launches
    avg_ms = acc_ms / acc_launches
    ach_gbs = alg_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    # 8 multiplies + 1 dual-product multiply per mixed add, in multiply-equivalents by wide-MAC count (N = limbs)
    mod_per_entry = (8 * (2 * n32 * n32 + n32) + (3 * n32 * n32 + n32)) / (2 * n32 * n32 + n32)   # 3p < 2^(32 N) for both base fields: the dual product applies
    ach_mod = (acc_entries * mod_per_entry / acc_launches) / (avg_ms * 1e-3) if avg_ms > 0 else 0.0
    # integer-pipe peak for this base field: the calibrated BN254 rate scaled by the wide-MAC count of one multiply (2N^2 + N)
    peak_mod = peak_modmul_bn * (2 * 8 * 8 + 8) / (2 * n32 * n32 + n32)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = tj.get(f"k_accumulate_g1_{cname}", {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    ns = curve
    pobj = mod.proof_to_object(ns, proof.tobytes())
    ph = proof_hash(pobj)
    gold = golden_hash(proto, cname, L)
    kname = f"k_accumulate<Fp<{'BnFq' if cname == 'bn128' else 'BlsFq'}>> (G1 bucket accumulation, {int(acc_launches)} launches per proof)"
    n = 1 << L
    wl = (f"plonk prove, {cname}, synthetic chain circuit, domain 2^{L}: 9 G1 MSM of n+6 points, 4 iNTT(n) + 4 NTT(4n) + 2 iNTT(4n), round kernels" if proto == "plonk"
          else f"fflonk prove, {cname}, synthetic chain circuit, domain 2^{L}: 4 G1 MSM of 8n..9n points, NTTs up to 4n, round kernels")
    line = {
        "metric": f"{proto}_proofs_per_sec", "value": world * args.steps / dt_res, "unit": "proofs/s", "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": dt_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"u32x8 scalar field / u32x{n32} base field (modular integers, 32-bit limbs)", "data": "synthetic",
        "config": {"workload": wl, "curve": cname, "gates": n - 6, "n_additions": int(pk.nAdditions), "parallelism": "single GPU" if world == 1 else f"{world} independent provers (replicas: the rounds are serialised by the transcript)",
                   "l2_policy": "inputs larger than L2 (key %.1f GB in HBM, %d MiB witness per proof vs 126 MB L2)" % (zkey_len / 1e9, nwit * 32 >> 20)},
        "e2e": {"value": world * args.steps / dt_e2e, "unit": "proofs/s", "h2d_bytes_per_step": int(nwit * 32), "d2h_bytes_per_step": int(proof.size),
                "ms_per_step": dt_e2e / args.steps * 1e3, "api": f"sb_{proto}_prove (pinned host witness -> proof bytes on host)"},
        "gpu_launches": int(l1 - l0), "launches_per_proof": int((l1 - l0) // max(args.steps, 1)), "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": kname, "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak if hbm_peak else None,
                     "traffic": traffic, "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                     "launch_ms": avg_ms, "algorithmic_bytes_per_launch": alg_bytes, "note": "integer-pipe bound kernel: see roofline_int"},
        "roofline_int": {"bound": "int32 IMAD pipe (modmul-bound roofline, SURVEY 8d)", "kernel": kname, "achieved": ach_mod / 1e9, "unit": "G Fq-modmul/s",
                         "peak": peak_mod / 1e9, "frac": ach_mod / peak_mod if peak_mod > 0 else None,
                         "peak_source": f"sb_calibrate(1) (BN254 Fq multiplies/s measured on this GPU in this run) x 136/{2 * n32 * n32 + n32} wide MACs per multiply of this base field"},
        "breakdown_ms": brk, "key_build_s": t_key, "key_load_s": t_load, "proof_sha256": ph,
        "oracle_match": (ph == gold) if gold else None,
        "oracle_match_source": "tests/golden/bench_proof_hashes.json (CPU port's proof of this key, tests/golden/make_bench_hashes.py)" if gold else "no committed hash for this size",
    }
    if not args.no_cpu_baseline and world == 1:
        try:
            Ls = args.cpu_log_n or L
            cores = host_cores()
            if Ls == L:
                dt, raw = cpu_prove(proto, zkey, wit_np, curve.r, curve.n8q, cores)
                line["cpu_live_match"] = (raw == proof.tobytes())
                sample = f"C++ port of {proto} prove (host backend, oracle NTT/MSM) proving the same key and witness at domain 2^{L}: one proof, {dt:.2f} s, {cores} OpenMP threads"
                val = 1.0 / dt
            else:
                zk2, w2, ci = oracle_key(proto, cname, Ls)
                dt, _ = cpu_prove(proto, zk2, w2, ci.r, ci.n8q, cores)
                scale = (1 << L) / (1 << Ls)
                sample = f"C++ port of {proto} prove at domain 2^{Ls}: {dt:.2f} s, {cores} OpenMP threads, scaled x{scale:g} linearly to 2^{L}"
                val = 1.0 / (dt * scale)
            line["cpu_baseline"] = {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample, "nproc": os.cpu_count()}
        except Exception as e:
            line["cpu_baseline"] = {"error": str(e)}
    print(json.dumps(line))
    dump_outputs(args.dump_outputs, proof)
    pk.release()
    curve.terminate()
    if dist is not None:
        dist.destroy_process_group()
    if gold and ph != gold:
        sys.exit("proof does not match the committed CPU-port hash (tests/golden/bench_proof_hashes.json)")
