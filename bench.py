#!/usr/bin/env python
"""bench.py -- Groth16 prove() on a synthetic DummyCircuit-shaped R1CS (BLS12-381), the hot path that
BASELINE.json's metric is quoted on, through libb200snark.so on 1..8 B200s; plus the CPU reference arm.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference ...                     (CPU restatement of the reference algorithms)
  python bench.py ... --dump-outputs DIR                   (also write the last timed proof to DIR/proof_{a,b,c}.npy)

One "step" = one proof: R1CS matrices x witness (SpMV) -> witness_map (the reference algorithm's 7 NTTs; 6 are executed, r1cs.cu) ->
4 G1 MSMs + 1 G2 MSM -> epilogue.  Algorithmic bytes stay SURVEY 8(d)'s figure for the reference algorithm (7 transforms).
`value` times proofs with z already resident in HBM; `e2e` times the public C-ABI call with z in pinned
host memory (H2D inside) and the proof read back to the host.  N > 1: strong scaling -- the five MSMs
are cut by base range over the ranks (each rank holds 1/N of the proving key), partial sums are
all-gathered with NCCL and rank 0 applies the epilogue.  See DESIGN.md for the roofline accounting.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLS_R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
R256 = 1 << 256
SEED_PK, SEED_RS, SEED_Z = 0xB2000003, 0xB2000004, 0xB2000005


def limbs(x):
    return np.array([(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)], dtype=np.uint32)


def mont(x):
    return limbs(x * R256 % BLS_R)


def ark_window_bits(n):
    if n < 32:
        return 3
    return (n - 1).bit_length() * 69 // 100 + 2


def msm_window_choice(n, point_bytes, bits=255):
    """(c, windows) the library picks for an n-point MSM (same cost model as msm_shape in csrc/msm.cu)."""
    best, best_c = None, 5
    for c in range(5, 21):
        nw = -(-bits // c)
        if bits - (nw - 1) * c >= c:
            nw += 1
        buckets = nw * (1 << (c - 1))
        if buckets * point_bytes > 4 << 30:
            break
        cost = n * nw + buckets * 4.7
        if best is None or cost < best:
            best, best_c, best_nw = cost, c, nw
    return best_c, best_nw


def reference_add_count(n, bits=255):
    """G1 additions ark-ec's Pippenger performs for an n-point MSM (SURVEY 8d): N*ceil(l/c) + ceil(l/c)*2^c."""
    c = ark_window_bits(n)
    w = -(-bits // c)
    return n * w + w * (1 << c)


# ------------------------------------------------------------------------------------------------
# synthetic instance (shared by both arms): DummyCircuit shape (relations/src/sr1cs/mod.rs:296-317)
# emitted directly as CSR, with n_rows + n_instance == 2^log_n so the QAP domain is exactly 2^log_n.
# ------------------------------------------------------------------------------------------------
def cpu_scale(log_s, log_n):
    """Fraction of a domain-2^log_n proof that a domain-2^log_s proof represents on the CPU, by the reference
    algorithm's own Pippenger addition count (MSMs are ~95 % of a CPU proof).  Slightly above the plain size ratio: the
    window grows with n (c = 15 at 2^20, 18 at 2^24), so a large MSM spends fewer additions per point -- scaling a small
    sample linearly would understate the CPU."""
    return reference_add_count(1 << log_s) / reference_add_count(1 << log_n)


def dummy_instance(log_n):
    N = 1 << log_n
    n_rows, n_inst = N - 2, 2
    n_wit = N - 3                      # a, b and N-5 copies of a  (n_vars = N - 1, h_query has N - 1 points)
    one = mont(1)
    nnz = n_rows - 1                   # the last constraint is empty (lc![] * lc![] = lc![])
    row_ptr = np.minimum(np.arange(n_rows + 1, dtype=np.uint64), np.uint64(nnz))
    coeff = np.tile(one, nnz)
    csr = [(row_ptr, np.full(nnz, col, dtype=np.uint32), coeff) for col in (2, 3, 1)]   # A: a, B: b, C: c = a*b
    rng = np.random.default_rng(SEED_Z)
    a = int.from_bytes(rng.bytes(32), "little") % BLS_R
    b = int.from_bytes(rng.bytes(32), "little") % BLS_R
    z_inst = np.concatenate([one, mont(a * b % BLS_R)])
    z_wit = np.tile(mont(a), n_wit)
    z_wit[8:16] = mont(b)
    return dict(N=N, n_rows=n_rows, n_inst=n_inst, n_wit=n_wit, csr=csr, z_inst=z_inst, z_wit=z_wit)


def rs_scalars():
    rng = np.random.default_rng(SEED_RS)
    r = int.from_bytes(rng.bytes(32), "little") % BLS_R
    s = int.from_bytes(rng.bytes(32), "little") % BLS_R
    return mont(r), mont(s)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, reasons, mx = [], set(), None
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
# CPU arm: the C++ restatement of ark-ec / ark-poly / ark-groth16 (oracle/c/oracle.cpp) on all host cores
# ------------------------------------------------------------------------------------------------
def cpu_prove_sample(log_n_sample, steps, warmup, threads=None):
    from oracle import cnative   # the one place outside tests/ that executes oracle/: the CPU baseline

    threads = threads or cnative.threads_default()
    inst = dummy_instance(log_n_sample)
    N, n_vars = inst["N"], inst["n_inst"] + inst["n_wit"]
    # synthetic key: multiples of the generators (distinct valid points; structure does not affect timing)
    g1 = np.array(_G1_GEN_MONT, dtype=np.uint32)
    g2 = np.array(_G2_GEN_MONT, dtype=np.uint32)
    mk1 = lambda start, n: cnative.multiples(0, 1, g1, start, n, threads)
    mk2 = lambda start, n: cnative.multiples(0, 2, g2, start, n, threads)
    pk = [mk1(3, 1), mk1(5, 1), mk1(7, 1), mk2(5, 1), mk2(7, 1), mk1(11, n_vars), mk1(11 + N, n_vars), mk2(13, n_vars),
          mk1(11 + 2 * N, N - 1), mk1(11 + 3 * N, inst["n_wit"])]
    r, s = rs_scalars()
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        cnative.groth16_prove(0, inst["csr"], inst["n_rows"], inst["n_inst"], inst["n_wit"], pk, inst["z_inst"], inst["z_wit"], r, s,
                              threads=threads)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return float(np.mean(times)), threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    from oracle import cnative
    cores = cnative.threads_default()
    log_s = args.ref_log_n or (20 if cores >= 16 else 16)
    log_s = min(log_s, args.log_n)
    sec, threads = cpu_prove_sample(log_s, args.steps, args.warmup)
    scale = cpu_scale(log_s, args.log_n)
    value = scale / sec
    sample = (f"Groth16 prove of the same DummyCircuit-shaped R1CS at domain 2^{log_s} ({sec:.3f} s/proof on {threads} threads), "
              f"scaled to 2^{args.log_n} by the reference's Pippenger addition count (x{1 / scale:.2f})")
    out = {
        "impl": "reference", "metric": "groth16_proofs_per_sec", "value": value, "unit": "proofs/s", "n_gpus": args.gpus,
        # ms_per_step is the time of one step AS RUN (a bounded sample: one proof at domain 2^log_s); `value` scales it to
        # the stated configuration -- the line says so instead of printing a 2^24 step time that was never measured
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "extrapolated": True,
        "sample_fraction_of_config": scale, "ms_per_step_extrapolated_to_config": 1e3 / value,
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 limbs (255/381-bit modular integers)", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": "proofs/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "C++ restatement of the ark-ec/ark-poly/ark-groth16 algorithms (no Rust toolchain here); MSMs are chunked over "
                "all host threads, which is stronger than ark-ec's per-window rayon parallelism",
    }
    emit(out)


def workload_config(args, world):
    return {"workload": f"Groth16 prove, BLS12-381, DummyCircuit-shaped R1CS, QAP domain 2^{args.log_n} "
                        f"({(1 << args.log_n) - 2} constraints, {(1 << args.log_n) - 1} variables)",
            "log_domain": args.log_n, "curve": "bls12_381", "parallelism": f"msm base-range shard x{world}" + (", witness map by four-step NTT over column slabs (one all-to-all per transform)" if world > 1 else ""),
            "l2": "inputs larger than L2 (proving key 9 GiB at 2^24); no flush needed"}


# ------------------------------------------------------------------------------------------------
# roofline of the dominant kernel, from the per-kernel CUDA-event totals of the timed region
# ------------------------------------------------------------------------------------------------
# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the bucket-accumulation launches of the h-query MSM of one
# proof at domain 2^24 on one GPU (uniform scalars: five halving rounds + the XYZZ pass, 92 % of the group's time), summed over
# the ncu pass of profiles/r02_msm_traffic_summary.txt; the three multiplicity-collapsed MSMs add one streaming round over
# their heavy list each (~5 GB apiece, not captured).  ~20x the algorithmic bytes BY CONSTRUCTION: the bucket method touches
# every base once per window, and the batched-affine rounds trade multiplications for two more streaming passes per round --
# DRAM stays under 45 % busy (same file).
NCU_TRAFFIC = {("g1", 24, 1): 1.63e11, ("g2", 24, 1): None}


def roofline_from_report(rep, N, world, log_n, peak, peak_src):
    """rep: {kernel: (launches, total_ms)} of ONE proof.  The dominant kernel GROUP is reported as one unit of work: the bucket
    accumulation of all G1 (or G2) MSMs of a proof = msm_ba_p1/inv/p2 (halving rounds) + msm_accumulate (XYZZ pass)."""
    groups_ = {}
    for name, (cnt, ms) in rep.items():
        grp = None
        if name in ("msm_accumulate_g1", "msm_ba_p1_g1", "msm_ba_inv_g1", "msm_ba_p2_g1"):
            grp = "g1"
        elif name in ("msm_accumulate_g2", "msm_ba_p1_g2", "msm_ba_inv_g2", "msm_ba_p2_g2"):
            grp = "g2"
        key = f"msm bucket accumulation {grp} (msm_ba_p1/inv/p2_{grp} + msm_accumulate_{grp})" if grp else name
        g = groups_.setdefault(key, {"ms": 0.0, "launches": 0, "grp": grp, "parts": {}})
        g["ms"] += ms
        g["launches"] += cnt
        g["parts"][name] = round(ms, 3)
    total_ms = sum(v[1] for v in rep.values())
    kern, g = max(groups_.items(), key=lambda kv: kv[1]["ms"])
    roof = {"kernel": kern, "bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src, "traffic": None,
            "launches": g["launches"], "share_of_step": g["ms"] / total_ms if total_ms else None, "parts_ms": g["parts"]}
    if g["grp"]:
        # (point, scalar) pairs this group consumes per proof on this rank: G1 = a, b_g1 (n_vars each), l (n_wit), h (N - 1)
        n_vars, n_wit = N - 1, N - 3
        pairs = ((2 * n_vars + n_wit + (N - 1)) if g["grp"] == "g1" else n_vars) / world
        alg = pairs * (128 if g["grp"] == "g1" else 224)
        ach = alg / (g["ms"] * 1e-3) / 1e9
        roof.update({"achieved": ach, "frac": ach / peak, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": g["ms"],
                     "launch_unit": f"all {'four G1 MSMs' if g['grp'] == 'g1' else 'G2 MSM work'} of one proof ({g['launches']} kernel launches: halving "
                                    "rounds of the h-query MSM and of the heavy lists of the multiplicity-collapsed MSMs, XYZZ passes)",
                     "traffic": NCU_TRAFFIC.get((g["grp"], log_n, world))})
        c_bits, nwin = msm_window_choice(int((N - 1) / world), 192 if g["grp"] == "g1" else 384)
        adds = pairs * nwin / (g["ms"] * 1e-3)
        ceil_ = 2.9e9 if g["grp"] == "g1" else None
        roof["alu"] = {"unit": f"Pippenger bucket additions/s a plain pipeline would perform (c={c_bits}, {nwin} windows per pair)", "achieved": adds,
                       "peak": ceil_, "frac": adds / ceil_ if ceil_ else None,
                       "note": "peak = XYZZ mixed G1 additions/s of tools/microbench.cu (10 Fq mul each, fmaheavy-pipe bound).  The fraction exceeds 1 "
                               "because the work is done with fewer multiplications: affine additions with shared inversions (6 mul) and ONE addition "
                               "per point for repeated scalar values; the fmaheavy utilisation of the kernels themselves is in profiles/ "
                               "(78 % in streaming rounds, 57 % in the gathered first round)"}
    else:
        roof["avg_launch_ms"] = g["ms"] / max(g["launches"], 1)
    return roof


# ------------------------------------------------------------------------------------------------
# one-off correctness check of the benchmarked proof (outside every timed region; the oracle is the checker)
# ------------------------------------------------------------------------------------------------
def verify_proof(be, mat, z_host_np, proof, key_scalars, consts, r_m, s_m, n_inst, check_h=True):
    """The synthetic key is k_j * G for known k_j, so A, B, C have known discrete logs (SURVEY App. A.6):
         a* = alpha + <k_a, z> + r delta      b* = beta + <k_b, z> + s delta
         c* = s a* + r b1* - r s delta + <k_l, w> + <k_h, h>
    The dot products are plain Fr arithmetic on the host (oracle/c), the three expected points three scalar
    multiplications of the big-int oracle.  h is the GPU's witness_map output and is itself compared, element by element,
    with the CPU oracle's witness_map (check_h)."""
    from oracle import cnative
    from oracle.ec import groups
    from oracle.params import BLS12_381 as curve
    from tests.util import unpack_fr, unpack_points

    rmod = curve.r
    n_vars = len(z_host_np) // 8
    t0 = time.time()
    h = be.witness_map(mat, z_host_np)
    info = {}
    if check_h:
        N = len(h) // 8
        inst = dummy_instance(N.bit_length() - 1)
        info["h_equals_cpu_oracle"] = bool(np.array_equal(h, cnative.witness_map(0, inst["csr"], inst["n_rows"], n_inst, z_host_np)))
        assert info["h_equals_cpu_oracle"], "witness_map differs from the CPU oracle"
    dot = lambda k, v, n: unpack_fr(curve, cnative.fr_dot(0, np.ascontiguousarray(k), np.ascontiguousarray(v), n), mont=False)[0]
    za = dot(key_scalars["a_query"], z_host_np, n_vars)
    zb1 = dot(key_scalars["b_g1_query"], z_host_np, n_vars)
    zb2 = dot(key_scalars["b_g2_query"], z_host_np, n_vars)
    wl = dot(key_scalars["l_query"], z_host_np[n_inst * 8:], n_vars - n_inst)
    hh = dot(key_scalars["h_query"], h, len(key_scalars["h_query"]) // 8)
    rr, ss = unpack_fr(curve, r_m)[0], unpack_fr(curve, s_m)[0]
    alpha, beta1, delta1, beta2, delta2 = consts
    a_star = (alpha + za + rr * delta1) % rmod
    b1_star = (beta1 + zb1 + ss * delta1) % rmod
    b2_star = (beta2 + zb2 + ss * delta2) % rmod
    c_star = (ss * a_star + rr * b1_star - rr * ss % rmod * delta1 + wl + hh) % rmod
    G1, G2 = groups(curve)
    ok = (unpack_points(curve, 1, proof[0])[0] == G1.mul(G1.gen, a_star) and unpack_points(curve, 2, proof[1])[0] == G2.mul(G2.gen, b2_star)
          and unpack_points(curve, 1, proof[2])[0] == G1.mul(G1.gen, c_star))
    assert ok, "benchmarked proof does not match its known discrete logs"
    info.update({"proof_equals_known_discrete_logs": True, "seconds": round(time.time() - t0, 1)})
    return info


def bind_to_gpu_numa_node(torch, index):
    """Run this process on the CPUs local to GPU `index` (sysfs local_cpulist of its PCI function), so that the pinned host buffer
    of the end-to-end leg is allocated on the GPU's NUMA node: a 512 MiB witness copied across sockets moves at a fraction of
    the PCIe rate (observed: end-to-end 210 vs 380 ms per proof on otherwise identical boxes).  Best effort; returns what it did."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        txt = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        cpus = set()
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"gpu": bdf, "cpus": txt}
    except Exception as e:   # noqa: BLE001 -- affinity is an optimisation, never a failure
        return {"error": repr(e)[:120]}
    return None


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import snark_b200
    from snark_b200 import shard
    from snark_b200.lib import MEM_DEVICE, PkDesc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpus_before = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(torch, local)       # before any pinned allocation: the host z buffer must sit next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    be = snark_b200.Backend(curve=0, device=local)   # raises (no fallback) without the .so or a B200
    ext = torch.cuda.ExternalStream(be.stream, device=dev)

    inst = dummy_instance(args.log_n)
    N, n_inst, n_wit = inst["N"], inst["n_inst"], inst["n_wit"]
    n_vars = n_inst + n_wit
    mat = be.r1cs_upload(inst["n_rows"], n_inst, n_wit, inst["csr"])
    inst["csr"] = None

    # --- synthetic proving key with known discrete logs, built on the GPU by the fixed-base kernel ----
    def rand_scalars(n, seed):
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        t = torch.randint(-(1 << 31), (1 << 31) - 1, (n, 8), dtype=torch.int32, device=dev, generator=g)
        t[:, 7] &= 0x1FFFFFFF           # < 2^253 < r: canonical scalars
        return t

    def q_range(name, total, rk):
        # every query is cut by base range; h by coefficient slab (what the distributed witness map hands each rank)
        return shard.slab_range(N, rk, world) if name == "h_query" else shard.shard_range(total, rk, world)

    def make_query(name, group, total, seed):
        lo, hi = q_range(name, total, rank)
        k = rand_scalars(hi - lo, seed * 1000 + rank)
        out = torch.empty(((hi - lo) * (be.g1_bytes if group == 1 else be.g2_bytes)) // 4, dtype=torch.int32, device=dev)
        be.fixed_base(group, k, hi - lo, mont=False, out=out)
        be.sync()
        return out, lo, hi - lo

    consts1 = torch.empty(3 * be.g1_bytes // 4, dtype=torch.int32, device=dev)
    consts2 = torch.empty(2 * be.g2_bytes // 4, dtype=torch.int32, device=dev)
    # the library reads its inputs on its own stream: keep the scalar tensors alive until it is done with them
    kc1, kc2 = rand_scalars(3, SEED_PK), rand_scalars(2, SEED_PK + 1)
    be.fixed_base(1, kc1, 3, mont=False, out=consts1)
    be.fixed_base(2, kc2, 2, mont=False, out=consts2)
    be.sync()
    d = PkDesc()
    d.n_instance, d.n_witness, d.domain_size = n_inst, n_wit, N
    g1w, g2w = be.g1_bytes, be.g2_bytes
    d.alpha_g1, d.beta_g1, d.delta_g1 = consts1.data_ptr(), consts1.data_ptr() + g1w, consts1.data_ptr() + 2 * g1w
    d.beta_g2, d.delta_g2 = consts2.data_ptr(), consts2.data_ptr() + g2w
    keep = []
    for name, off, ln, group, total, seed in (("a_query", "a_off", "a_len", 1, n_vars, 11), ("b_g1_query", "b1_off", "b1_len", 1, n_vars, 12),
                                              ("b_g2_query", "b2_off", "b2_len", 2, n_vars, 13), ("h_query", "h_off", "h_len", 1, N - 1, 14),
                                              ("l_query", "l_off", "l_len", 1, n_wit, 15)):
        t, lo, cnt = make_query(name, group, total, SEED_PK + seed)
        keep.append(t)
        setattr(d, name, t.data_ptr()); setattr(d, off, lo); setattr(d, ln, cnt)
    pk = be.pk_upload(d, mem=MEM_DEVICE)
    keep.clear()
    torch.cuda.empty_cache()

    grp = None
    if world > 1:
        # the NCCL id travels over torch.distributed (any channel would do); the communicator lives inside the library
        uid = torch.from_numpy(be.group_unique_id() if rank == 0 else np.zeros(128, dtype=np.uint8)).to(dev)
        dist.broadcast(uid, 0)
        grp = be.group_create(uid.cpu().numpy(), rank, world)

    r, s = rs_scalars()
    z_host = torch.from_numpy(np.concatenate([inst["z_inst"], inst["z_wit"]]).view(np.int32)).pin_memory()
    z_dev = z_host.to(dev)

    def prove(resident):
        """One proof; returns the proof (rank 0) -- every rank takes part."""
        if world == 1:
            if resident:
                return be.groth16_prove_resident(pk, mat, z_dev, r, s)
            return be.groth16_prove(pk, mat, zi_ptr_obj, zw_ptr_obj, r, s)
        # one collective C-ABI call per rank: shard MSMs, ONE ncclAllGather of the five partial sums (device buffers, on the
        # library's stream, communicator owned by the library) and the join + epilogue on rank 0
        if resident:
            proof = be.groth16_prove_group_resident(grp, pk, mat, z_dev, r, s)
        else:
            proof = be.groth16_prove_group(grp, pk, mat, zi_ptr_obj, zw_ptr_obj, r, s)
        return proof if rank == 0 else None

    # views of the pinned host buffer (Backend passes their addresses through as HOST memory)
    zi_ptr_obj = z_host[: n_inst * 8].numpy()
    zw_ptr_obj = z_host[n_inst * 8:].numpy()

    def timed(resident, steps, warmup, profile=False):
        for _ in range(warmup):
            prove(resident)
        be.sync(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if profile:
            be.profile(True)
        launches0 = be.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        t0 = time.perf_counter()
        proof = None
        for _ in range(steps):
            proof = prove(resident)
        e1.record(ext)
        be.sync(); torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1), wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        rep = be.profile_report() if profile else None
        if profile:
            be.profile(False)
        return float(ms[0]), float(ms[1]), be.launches - launches0, rep, proof

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dev_ms, wall_ms, launches, _, proof_a = timed(True, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    e2e_ms, e2e_wall, _, _, proof_b = timed(False, args.steps, 1)
    # per-kernel breakdown from a separate profiled pass (an event pair around each of the ~1000 launches of a proof costs
    # tens of milliseconds per step, so it stays out of the two timed regions above)
    _, _, _, rep, _ = timed(True, 1, 0, profile=True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    assert all(np.array_equal(x, y) for x, y in zip(proof_a, proof_b)), "resident and host-buffer proofs differ"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof_a)
    verified = None
    if not args.no_verify:
        # regenerate every rank's key scalars on this GPU (same seeded generator) and check the proof in the exponent
        def canon(t):
            return t.cpu().numpy().view(np.uint32).reshape(-1)

        ks = {}
        for name, total, seed in (("a_query", n_vars, 11), ("b_g1_query", n_vars, 12), ("b_g2_query", n_vars, 13), ("h_query", N - 1, 14),
                                  ("l_query", n_wit, 15)):
            parts = []
            for rk in range(world):
                lo, hi = q_range(name, total, rk)
                parts.append(canon(rand_scalars(hi - lo, (SEED_PK + seed) * 1000 + rk)))
            ks[name] = np.concatenate(parts)
        lim = lambda row: sum(int(v) << (32 * i) for i, v in enumerate(row))
        c1 = canon(rand_scalars(3, SEED_PK)).reshape(3, 8)
        c2 = canon(rand_scalars(2, SEED_PK + 1)).reshape(2, 8)
        consts = [lim(c1[0]), lim(c1[1]), lim(c1[2]), lim(c2[0]), lim(c2[1])]
        verified = verify_proof(be, mat, z_host.numpy().view(np.uint32), proof_a, ks, consts, r, s, n_inst, check_h=(world == 1))
        del ks
    value = args.steps / (dev_ms / 1e3)
    e2e_value = args.steps / (e2e_ms / 1e3)

    peak, peak_src = hbm_peak()
    roof = roofline_from_report(rep, N, world, args.log_n, peak, peak_src)
    msm_adds = 4 * reference_add_count(N) * value   # four ~N-point G1 MSMs per proof, reference add count
    out = {
        "metric": "groth16_proofs_per_sec", "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 limbs (255/381-bit modular integers)", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": "proofs/s", "h2d_bytes_per_step": int(n_vars * 32 + 64), "d2h_bytes_per_step": int(2 * g1w + g2w),
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof,
        "kernel_ms_per_step": {k: round(v[1], 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])},
        "msm_g1_adds_per_sec_in_prove": msm_adds, "wall_ms_per_step": wall_ms / args.steps,
        "verified": verified, "host_affinity": numa,
    }
    if world == 1 and not args.no_extras:
        out["extras"] = extras(be, torch, dev, ext, peak)
    os.sched_setaffinity(0, cpus_before)             # the CPU baseline below may use every core the box allows
    if world == 1 and not args.no_cpu:
        from oracle import cnative
        cores = cnative.threads_default()
        log_s = min(args.ref_log_n or (20 if cores >= 16 else 16), args.log_n)
        sec, threads = cpu_prove_sample(log_s, 1, 0)
        scale = cpu_scale(log_s, args.log_n)
        out["cpu_baseline"] = {"value": scale / sec, "unit": "proofs/s", "cores": threads, "kind": "port",
                               "sample": f"one Groth16 prove at domain 2^{log_s} ({sec:.3f} s on {threads} threads), scaled to "
                                         f"2^{args.log_n} by the reference's Pippenger addition count (x{1 / scale:.2f})"}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(path, proof):
    """The proof of the last timed step as the caller receives it -- A (G1), B (G2), C (G1), affine, Montgomery u32 limbs --
    one float64 array per point (exact for 32-bit words), so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, arr in zip(("proof_a", "proof_b", "proof_c"), proof):
        np.save(os.path.join(path, f"{name}.npy"), arr.astype(np.float64))


def extras(be, torch, dev, ext, peak):
    """BASELINE configs 2 and 3 on one GPU: 2^22-point G1 MSM and 2^24-element NTT round trip."""
    res = {}

    def time_fn(fn, reps=3):
        fn(); be.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        for _ in range(reps):
            fn()
        e1.record(ext)
        be.sync()
        return e0.elapsed_time(e1) / reps

    g = torch.Generator(device=dev); g.manual_seed(0xB2000001)
    n = 1 << 22
    k = torch.randint(-(1 << 31), (1 << 31) - 1, (n, 8), dtype=torch.int32, device=dev, generator=g)
    k[:, 7] &= 0x1FFFFFFF
    bases = torch.empty(n * be.g1_bytes // 4, dtype=torch.int32, device=dev)
    be.fixed_base(1, k, n, mont=False, out=bases)
    sc = torch.randint(-(1 << 31), (1 << 31) - 1, (n, 8), dtype=torch.int32, device=dev, generator=g)
    sc[:, 7] &= 0x1FFFFFFF
    ms = time_fn(lambda: be.msm_g1(bases, sc, n, mont=True))
    res["msm_g1_2p22_uniform"] = {"ms": ms, "g1_adds_per_sec_reference_count": reference_add_count(n) / (ms / 1e3),
                                  "hbm_GBps_algorithmic": n * 128 / (ms / 1e3) / 1e9, "hbm_frac": n * 128 / (ms / 1e3) / 1e9 / peak}
    same = sc[:1].repeat(n, 1).contiguous()
    ms = time_fn(lambda: be.msm_g1(bases, same, n, mont=True))
    res["msm_g1_2p22_all_equal_scalars"] = {"ms": ms, "g1_adds_per_sec_reference_count": reference_add_count(n) / (ms / 1e3)}
    del bases, k, sc, same
    n = 1 << 24
    x = torch.randint(-(1 << 31), (1 << 31) - 1, (n, 8), dtype=torch.int32, device=dev, generator=g)
    x[:, 7] &= 0x1FFFFFFF
    ms = time_fn(lambda: be.ntt(x, 24))
    res["ntt_2p24_forward"] = {"ms": ms, "elements_per_sec": n / (ms / 1e3), "hbm_GBps_algorithmic": n * 64 / (ms / 1e3) / 1e9,
                               "hbm_frac": n * 64 / (ms / 1e3) / 1e9 / peak}
    return res


# standard generators in Montgomery limbs (the same constants as snark_b200/csrc/field_params.h)
def _gen_limbs():
    p = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
    R = 1 << 384
    g1 = (0x17F1D3A73197D7942695638C4FA9AC0FC3688C4F9774B905A14E3A3F171BAC586C55E83FF97A1AEFFB3AF00ADB22C6BB,
          0x08B3F481E3AAA0F1A09E30ED741D8AE4FCF5E095D5D00AF600DB18CB2C04B3EDD03CC744A2888AE40CAA232946C5E7E1)
    g2 = (0x024AA2B2F08F0A91260805272DC51051C6E47AD4FA403B02B4510B647AE3D1770BAC0326A805BBEFD48056C8C121BDB8,
          0x13E02B6052719F607DACD3A088274F65596BD0D09920B61AB5DA61BBDC7F5049334CF11213945D57E5AC7D055D042B7E,
          0x0CE5D527727D6E118CC9CDC6DA2E351AADFD9BAA8CBDD3A76D429A695160D12C923AC9CC3BACA289E193548608B82801,
          0x0606C4A02EA734CC32ACD2B02BC28B99CB3E287E85A763AF267492AB572E99AB3F370D275CEC1DA1AAA9075FF05F79BE)
    f = lambda v: [((v * R % p) >> (32 * i)) & 0xFFFFFFFF for i in range(12)]
    return sum((f(v) for v in g1), []), sum((f(v) for v in g2), [])


_G1_GEN_MONT, _G2_GEN_MONT = _gen_limbs()
_REAL_STDOUT = None


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=24, help="log2 of the QAP domain (24 = BASELINE's headline size)")
    ap.add_argument("--ref-log-n", type=int, default=0, help="domain of the bounded CPU sample (default: 20 with >= 64 cores, else 16)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the one-off check of the proof against its known discrete logs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step to DIR/proof_{a,b,c}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the B200 arm")
    # the contract is ONE JSON line on stdout: anything libraries print there (e.g. NCCL's version banner) goes
    # to stderr instead; emit() writes the result line to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
