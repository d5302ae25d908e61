#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on N GPUs of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference            # the reference's own CPU path on the host cores
    python bench.py --dump-outputs DIR          # also write a sample of the timed step's outputs to DIR/*.npy

Workload (BASELINE.json configs[1]): batched forward + inverse negacyclic NTT,
N = 2^16, 55-bit prime (GeneratePrimes(1, 55, true, N)), 8192 polynomials per GPU,
coefficients uniform in [0, q).  A "step" is one forward pass (x -> y) and one
inverse pass (y -> z) over the batch = 2 * 8192 transforms per GPU.  Batches of
independent polynomials shard across GPUs with no data-path collective
(scaling = weak: 8192 polynomials per GPU); the only torch.distributed calls
are the barrier and the max-over-ranks of the measured time.

`value`  : NTTs/sec, whole job, inputs resident in HBM, CUDA-event timed.
`e2e`    : the same metric through the C ABI's HOST-pointer path (pinned host
           buffers in, pinned host buffers out, copies inside the timed region).
`roofline`: the forward transform (all kernels of one hexl_b200_ntt_forward call)
           against the measured HBM copy bandwidth; 16*N algorithmic bytes/NTT.
`cpu_baseline`: the compiled reference (oracle/_ref) timed on the host cores
           (rank 0, N = 1 only), on a bounded sample of the same workload.
`eltwise` : BASELINE configs[2]: EltwiseMultMod / FMAMod / ReduceMod over N = 2^10..2^17 x {40,50,60}-bit q,
           batch 4096, algorithmic GB/s and fraction of the measured HBM peak.
`c4`      : BASELINE configs[3]: FwdNTT -> EltwiseMultMod -> InvNTT, N = 2^17, 16 x 60-bit moduli, the moduli
           split across the ranks (2 per GPU at 8 GPUs; strong scaling of one fixed job), residue products/s.
`c5`      : BASELINE configs[4]: CKKS KeySwitch, N = 2^15, 30 RNS moduli, sharded by ciphertext (every rank holds
           the keys and switches its own ciphertexts: no exchange on the data path), key switches/s; `e2e` =
           host buffers through hexl_b200_key_switch_resident with the keys resident on the GPU.
Every rank is bound to the NUMA node of its GPU before it allocates pinned memory.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = 16
MOD_BITS = 55
BATCH = 8192
METRIC = "ntt_per_sec_fwd_inv_N65536_q55_batch8192"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="polynomials per GPU")
    ap.add_argument("--logn", type=int, default=LOG_N)
    ap.add_argument("--bits", type=int, default=MOD_BITS)
    ap.add_argument("--e2e-batch", type=int, default=None, help="polynomials per GPU for the host-pointer leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-eltwise", action="store_true")
    ap.add_argument("--no-composites", action="store_true", help="skip the c4 / c5 legs")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of what the last one computed to DIR/*.npy "
                         "(b200 arm, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def wait_first(self, work=None, timeout=3.0):
        """Keep the GPU busy (work()) until nvidia-smi has printed its first sample, so that the tool's start-up
        (NVML initialisation, a few hundred ms) lands in the warm-up and only its periodic queries in the timed region."""
        t0 = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t0 < timeout:
            if work:
                work()
            else:
                time.sleep(0.01)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ NUMA
def bind_to_gpu_numa(local: int):
    """Pin this rank to the CPUs of the NUMA node its GPU hangs off, so that pinned staging buffers are allocated
    (first touch) in that node's DRAM and H2D/D2H copies do not cross the socket interconnect.  Returns a short
    description for the JSON line; a no-op on single-node hosts or when sysfs does not say."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read())
        if node < 0:
            return {"node": None, "note": "sysfs reports no NUMA affinity"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"node": node, "note": "no allowed CPU on that node"}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus": len(allowed)}
    except (OSError, ValueError, AttributeError, RuntimeError) as e:
        return {"node": None, "note": f"not bound ({type(e).__name__})"}


def source_hash() -> str:
    """sha256 over the sources of the transform kernels the roofline is about (hexl_b200_ntt_forward / _inverse):
    profiles/traffic.json is only believed when it was captured on this code"""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "hexl_b200", "csrc")
    for name in ("internal.h", "modarith.cuh", "ntt.cu", "ntt_kernels.cuh"):
        h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


# ------------------------------------------------------------ reference arm
def cpu_threads() -> int:
    """host threads this process can actually run concurrently: the affinity mask
    capped by the cgroup CPU quota (a container may see 128 CPUs but own 16)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:  # cgroup v2
        q, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = int(q) / int(period)
    except (OSError, ValueError):
        try:  # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / period
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def cpu_leg(n, q, threads, polys, reps, min_seconds=0.0):
    """forward + inverse over `polys` polynomials with the reference's CPU path;
    returns (NTTs/sec best-of-reps, description).  Uses oracle/_ref when it is
    here, else the C restatement."""
    import numpy as np
    import oracle
    chk = oracle.best_checker()
    rng = np.random.default_rng(42)
    x = rng.integers(0, q, size=n * polys, dtype=np.uint64)
    if chk.kind == "reference":
        y, z = np.empty_like(x), np.empty_like(x)
        fwd = lambda: chk.ntt_forward(x, n, q, 1, 1, threads=threads, out=y)
        inv = lambda: chk.ntt_inverse(y, n, q, 1, 1, threads=threads, out=z)
        tier = chk.tier(q)
    else:
        chk.tables(n, q)
        state = {}
        fwd = lambda: state.__setitem__("y", chk.ntt_forward(x, n, q, 1, 1, threads=threads))
        inv = lambda: state.__setitem__("z", chk.ntt_inverse(state["y"], n, q, 1, 1, threads=threads))
        tier = "scalar C restatement"
    fwd(); inv()  # warm: tables, page faults
    best, spent, done = float("inf"), 0.0, 0
    while done < reps or (spent < min_seconds and done < 64):
        t0 = time.perf_counter()
        fwd(); inv()
        dt = time.perf_counter() - t0
        best, spent, done = min(best, dt), spent + dt, done + 1
    cpu_leg.last = {"reps": done, "seconds": spent}
    if chk.kind == "reference":
        assert (z == x).all(), "reference round trip failed"
    return 2 * polys / best, chk.kind, tier


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    n = 1 << args.logn
    q = oracle.best_checker().generate_primes(1, args.bits, True, n)[0]
    threads = cpu_threads()
    polys = max(threads * 16, 64)
    # each step = one bounded sample (forward + inverse over `polys` polynomials)
    vals = []
    kind = tier = None
    for _ in range(args.warmup + args.steps):
        v, kind, tier = cpu_leg(n, q, threads, polys, 1)
        vals.append(v)
    vals = vals[args.warmup:]
    value = 2 * polys * len(vals) / sum(2 * polys / v for v in vals)
    ms = 1e3 * 2 * polys / value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "NTT/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"batched Fwd+Inv NTT, N=2^{args.logn}, {args.bits}-bit prime q={q}, "
                               f"sample of {polys} polynomials per step on the host cores",
                   "tier": tier},
        "cpu_baseline": {"value": value, "unit": "NTT/s", "cores": threads, "kind": kind,
                         "sample": f"{polys} polynomials x (forward + inverse) per step, {threads} threads, tier {tier}"},
        "e2e": {"value": value, "unit": "NTT/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------ multi-rank helpers
def max_over_ranks(value: float, world: int, device="cuda") -> float:
    """device-timed duration -> max over ranks (NCCL on GPUs, gloo in the CPU test)"""
    if world <= 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_value(units_per_rank: int, world: int, seconds: float, weak: bool = True, total_units: int = 0) -> float:
    """units/second of the whole job: weak scaling counts world * units_per_rank"""
    units = world * units_per_rank if weak else total_units
    return units / seconds


# ----------------------------------------------------------------- b200 arm
def gpu_time_ms(torch, fn, reps, sync):
    """device time of `reps` back-to-back calls of fn (CUDA events on the current stream), per call"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def dump_outputs(out_dir, np, torch, outputs, budget=16 << 20):
    """Write each (batch, N) result of the timed step as <out_dir>/<name>.npy, so that two builds run with the same
    arguments (hence the same seeded inputs) can be compared output for output.  A fixed sample of rows is kept
    (numpy default_rng(0), at most `budget` bytes per output), in float64 of shape (rows, N, 2): the high and the low
    32 bits of every 64-bit word, because float64 alone would round residues above 2^53."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        batch, n = t.shape
        rows = min(batch, max(1, budget // (16 * n)))
        idx = np.sort(np.random.default_rng(0).choice(batch, size=rows, replace=False))
        w = t[torch.from_numpy(idx).to(t.device)].cpu().numpy().view(np.uint64)
        halves = np.stack([w >> np.uint64(32), w & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
        np.save(os.path.join(out_dir, f"{name}.npy"), halves)


def eltwise_sweep(hb, torch, peak, gen, sync):
    """BASELINE configs[2]: N = 2^10..2^17 x q in {40,50,60}-bit x {MultMod, FMAMod, ReduceMod}, batch 4096"""
    out = {"batch": 4096, "bytes_per_element": {"mult_mod": 24, "fma_mod": 24, "reduce_mod": 16}, "points": []}
    fracs = []
    cap = 4096 << 17
    a = torch.empty(cap, dtype=torch.int64, device="cuda")
    b = torch.empty(cap, dtype=torch.int64, device="cuda")
    r = torch.empty(cap, dtype=torch.int64, device="cuda")
    for bits in (40, 50, 60):
        for logn in range(10, 18):
            n = 4096 << logn
            q = hb.GeneratePrimes(1, bits, True, 1 << logn)[0]
            av, bv, rv = a[:n], b[:n], r[:n]
            av.random_(0, q, generator=gen)
            bv.random_(0, q, generator=gen)
            ops = {"mult_mod": (24, lambda: hb.EltwiseMultMod(rv, av, bv, n, q, 1)),
                   "fma_mod": (24, lambda: hb.EltwiseFMAMod(rv, av, 123456789 % q, bv, n, q, 1)),
                   "reduce_mod": (16, lambda: hb.EltwiseReduceMod(rv, av, n, q, q, 1))}
            row = {"logn": logn, "q_bits": bits}
            for name, (bpe, fn) in ops.items():
                fn(); fn()
                reps = 3 if logn >= 15 else 8
                ms = gpu_time_ms(torch, fn, reps, sync)
                gbs = bpe * n / (ms * 1e-3) / 1e9
                row[name] = round(gbs, 1)
                fracs.append(gbs / peak)
            out["points"].append(row)
    out["frac_of_hbm_peak"] = {"min": min(fracs), "median": statistics.median(fracs), "max": max(fracs)}
    # the single largest point, kept under the round-1 key names
    big = out["points"][-1]
    for name in ("mult_mod", "fma_mod", "reduce_mod"):
        out[name] = {"GBps": big[name], "frac_of_hbm_peak": big[name] / peak}
    return out


def c4_leg(args, hb, torch, rank, world, gen, sync, peak, cpu_ok):
    """configs[3]: N = 2^17, 16 x 60-bit moduli split across the ranks, `group` polynomials per modulus"""
    n, nmod, group = 1 << 17, 16, 32
    mods_all = hb.GeneratePrimes(nmod, 60, True, n)
    lo, hi = nmod * rank // world, nmod * (rank + 1) // world
    mods = mods_all[lo:hi]
    ntts = [hb.NTT(n, q) for q in mods]
    sz = n * group
    a = torch.empty(len(mods) * sz, dtype=torch.int64, device="cuda")
    b = torch.empty_like(a)
    for i, q in enumerate(mods):
        a[i * sz:(i + 1) * sz].random_(0, q, generator=gen)
        b[i * sz:(i + 1) * sz].random_(0, q, generator=gen)
    r = torch.empty_like(a)
    fn = lambda: hb.PolyMultiplyMulti(ntts, r, a, b, group)
    fn(); fn()
    ms = max_over_ranks(gpu_time_ms(torch, fn, 5, sync), world)
    fused = os.environ.get("HEXL_B200_NO_PRODUCT_FUSION", "0") in ("", "0")
    bpp = 56 if fused else 72  # bytes per coefficient of one product: 2 x 16 (transforms) + 16 + 8 (inverse, multiplied on load)
    out = {"workload": (f"FwdNTT x2 -> InvNTT multiplying on load (EltwiseMultMod folded in), " if fused else
                        f"FwdNTT x2 -> EltwiseMultMod -> InvNTT, ") + f"N=2^17, {nmod} x 60-bit moduli, {group} polynomials per modulus",
           "value": nmod * group / (ms * 1e-3), "unit": "residue products/s", "ms_per_call": ms, "scaling": "strong",
           "moduli_per_rank": [nmod * (k + 1) // world - nmod * k // world for k in range(world)],
           "algorithmic_bytes_per_product": bpp * n,
           "hbm_GBps_per_gpu": float(bpp) * n * len(mods) * group / (ms * 1e-3) / 1e9,
           "limit": "integer-multiply pipe of the three transforms (no inter-GPU traffic: each rank owns whole moduli)"}
    out["frac_of_hbm_peak"] = out["hbm_GBps_per_gpu"] / peak
    # end to end: pageable-free pinned host buffers through the chunked staging path of the same call
    try:
        ha, hbuf, hr = (hb.pinned_empty(a.numel()) for _ in range(3))
        ha[:] = a.cpu().numpy().view("uint64")
        hbuf[:] = b.cpu().numpy().view("uint64")
        efn = lambda: hb.PolyMultiplyMulti(ntts, hr, ha, hbuf, group)
        efn()
        assert (hr == r.cpu().numpy().view("uint64")).all(), "c4 host path differs from the device path"
        sync()
        t0 = time.perf_counter()
        for _ in range(3):
            efn()
        dt = max_over_ranks((time.perf_counter() - t0) / 3, world)
        out["e2e"] = {"value": nmod * group / dt, "unit": "residue products/s", "h2d_bytes_per_step": 16 * a.numel(),
                      "d2h_bytes_per_step": 8 * a.numel(), "ms_per_call": dt * 1e3,
                      "h2d_GBps_per_gpu": 16 * a.numel() / dt / 1e9}
        for buf in (ha, hbuf, hr):
            hb.pinned_free(buf)
    except hb.HexlB200Error as e:
        out["e2e"] = {"unavailable": str(e)[:120]}
    if cpu_ok:
        import numpy as np
        import oracle
        chk = oracle.best_checker()
        threads = cpu_threads()
        q = mods_all[0]
        polys = max(threads, 8)
        x = np.random.default_rng(1).integers(0, q, size=n * polys, dtype=np.uint64)
        y = np.random.default_rng(2).integers(0, q, size=n * polys, dtype=np.uint64)
        # only the compiled reference splits an element-wise call over threads; the C restatement runs it on one
        split = {"rows": polys, "threads": threads} if chk.kind == "reference" else {}

        def cpu():
            fx = chk.ntt_forward(x, n, q, 1, 4, threads=threads)
            fy = chk.ntt_forward(y, n, q, 1, 4, threads=threads)
            p = chk.mult_mod(fx, fy, q, 4, **split)
            return chk.ntt_inverse(p, n, q, 1, 1, threads=threads)
        cpu()
        t0 = time.perf_counter()
        ref = cpu()
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": polys / dt, "unit": "residue products/s", "cores": threads, "kind": chk.kind,
                               "sample": f"{polys} polynomials of one modulus"}
        # parity of the timed device result against the reference on the first polynomial of the first modulus
        x0 = a[:n].cpu().numpy().view("uint64"); y0 = b[:n].cpu().numpy().view("uint64")
        exp = chk.ntt_inverse(chk.mult_mod(chk.ntt_forward(x0, n, q), chk.ntt_forward(y0, n, q), q), n, q)
        out["parity"] = bool((r[:n].cpu().numpy().view("uint64") == exp).all())
        assert out["parity"], "c4 device result differs from the checker"
    return out


def c5_leg(args, hb, torch, rank, world, gen, sync, cpu_ok):
    """configs[4]: CKKS KeySwitch, N = 2^15, 30 moduli (29 digits + special prime), sharded by ciphertext"""
    import numpy as np
    n, decomp, kcc, cts = 1 << 15, 29, 2, 8
    kms = rns = decomp + 1
    mods = hb.GeneratePrimes(kms, 50, True, n)
    modswitch = [hb.InverseMod(mods[-1] % mods[i], mods[i]) for i in range(decomp)]

    def rand_rows(count_rows, row_mods):  # rows of n values, row i below row_mods[i]
        t = torch.empty(count_rows * n, dtype=torch.int64, device="cuda")
        for i, q in enumerate(row_mods):
            t[i * n:(i + 1) * n].random_(0, q, generator=gen)
        return t
    keys = [rand_rows(kcc * kms, [mods[i] for _ in range(kcc) for i in range(kms)]) for _ in range(decomp)]
    t_all = torch.cat([rand_rows(decomp, mods[:decomp]) for _ in range(cts)])
    r0 = torch.cat([rand_rows(kcc * decomp, [mods[i] for _ in range(kcc) for i in range(decomp)]) for _ in range(cts)])
    handle = hb.KeySwitchKeys(keys, n, decomp, kms, kcc)
    res = r0.clone()
    fn = lambda: hb.KeySwitchResident(res, t_all, n, decomp, kms, rns, kcc, mods, handle, modswitch, cts)
    fn(); fn()
    ms = max_over_ranks(gpu_time_ms(torch, fn, 3, sync), world)
    out = {"workload": f"CKKS KeySwitch, N=2^15, L={kms} 50-bit moduli ({decomp} digits + special prime), "
                       f"{cts} ciphertexts per GPU per call, keys resident ({decomp * kcc * kms * n * 8 >> 20} MiB)",
           "value": world * cts / (ms * 1e-3), "unit": "key switches/s", "ms_per_key_switch": ms / cts, "scaling": "weak",
           "sharding": "by ciphertext (every rank holds the keys; no exchange on the data path). Sharding one key switch "
                       "by modulus would need the all-gather of the decomposed digits (key-switch-internal.cpp:60-131)"}
    # end to end: host buffers in and out, keys stay on the GPU
    try:
        ht, hr = hb.pinned_empty(t_all.numel()), hb.pinned_empty(r0.numel())
        ht[:] = t_all.cpu().numpy().view("uint64")
        r0h = r0.cpu().numpy().view("uint64")
        hr[:] = r0h
        efn = lambda: hb.KeySwitchResident(hr, ht, n, decomp, kms, rns, kcc, mods, handle, modswitch, cts)
        efn()
        res.copy_(r0); fn(); torch.cuda.synchronize()
        assert (hr == res.cpu().numpy().view("uint64")).all(), "c5 host path differs from the device path"
        sync()
        t0 = time.perf_counter()
        for _ in range(3):
            efn()
        dt = max_over_ranks((time.perf_counter() - t0) / 3, world)
        out["e2e"] = {"value": world * cts / dt, "unit": "key switches/s", "ms_per_key_switch": dt * 1e3 / cts,
                      "h2d_bytes_per_step": 8 * (t_all.numel() + r0.numel()), "d2h_bytes_per_step": 8 * r0.numel()}
        # latency of ONE switch from host buffers (what a reference-shaped caller sees): keys resident on one GPU, and --
        # when this single process sees several GPUs -- the moduli of the switch sharded over all of them (digit
        # all-gather + special-prime broadcast over NVLink peer copies)
        if world == 1:
            one = lambda h: hb.KeySwitchResident(hr[:r0.numel() // cts], ht[:t_all.numel() // cts], n, decomp, kms, rns, kcc,
                                                 mods, h, modswitch, 1)
            one(handle); one(handle)
            t0 = time.perf_counter()
            for _ in range(10):
                one(handle)
            lat = {"one_gpu_ms": (time.perf_counter() - t0) * 100.0}
            ndev = hb.device_count()
            if ndev >= 2:
                hkeys = [k.cpu().numpy().view("uint64") for k in keys]
                try:
                    hb.set_host_devices(list(range(ndev)))
                    sh = hb.KeySwitchKeys(hkeys, n, decomp, kms, kcc, sharded_by_modulus=True)
                finally:
                    hb.set_host_devices([])
                hr[:] = r0h
                one(sh)
                ref1 = res[:r0.numel() // cts].cpu().numpy().view("uint64")   # device result of ciphertext 0 (computed above)
                assert (hr[:r0.numel() // cts] == ref1).all(), "sharded key switch differs from the single-GPU result"
                one(sh)
                t0 = time.perf_counter()
                for _ in range(10):
                    one(sh)
                lat["sharded_by_modulus_ms"] = (time.perf_counter() - t0) * 100.0
                lat["shards"] = ndev
                del sh
            out["latency_one_switch_host_buffers"] = lat
        hb.pinned_free(ht); hb.pinned_free(hr)
    except hb.HexlB200Error as e:
        out["e2e"] = {"unavailable": str(e)[:120]}
    if cpu_ok:
        import oracle
        chk = oracle.best_checker()
        if getattr(chk, "has_seal", True):
            hk = [k.cpu().numpy().view("uint64") for k in keys]
            t1 = t_all[:decomp * n].cpu().numpy().view("uint64")
            r1 = r0[:kcc * decomp * n].cpu().numpy().view("uint64")
            threads = cpu_threads()
            results = [None] * threads

            def work(i):
                results[i] = chk.key_switch(r1.copy(), t1, n, decomp, kms, rns, kcc, mods, hk, modswitch)
            t0 = time.perf_counter()
            th = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
            [t.start() for t in th]; [t.join() for t in th]
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": threads / dt, "unit": "key switches/s", "cores": threads, "kind": chk.kind,
                                   "sample": f"{threads} independent key switches, one per thread (the reference's KeySwitch is single-threaded)"}
            res.copy_(r0); fn(); torch.cuda.synchronize()
            out["parity"] = bool((res[:kcc * decomp * n].cpu().numpy().view("uint64") == results[0]).all())
            assert out["parity"], "c5 device result differs from the checker"
    return out


def run_b200_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import hexl_b200 as hb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU fallback)")
    torch.cuda.set_device(local)
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local)
    # stdout is reserved for the one JSON line: libraries that print there (NCCL's version banner
    # does) are sent to stderr at the file-descriptor level, the line goes to the saved descriptor
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = 1 << args.logn
    q = hb.GeneratePrimes(1, args.bits, True, n)[0]
    ntt = hb.NTT(n, q)
    batch = args.batch
    g = torch.Generator(device="cuda").manual_seed(42 + rank)
    x = torch.randint(0, q, (batch, n), dtype=torch.int64, device="cuda", generator=g)
    y = torch.empty_like(x)
    z = torch.empty_like(x)

    def step():
        ntt.ComputeForward(y, x, 1, 1)
        ntt.ComputeInverse(z, y, 1, 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    assert torch.equal(z, x), "round trip Inv(Fwd(x)) != x"

    # ---- device-resident throughput
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first(lambda: (step(), torch.cuda.synchronize()))
    launches0 = hb.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = hb.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np, torch, {"ntt_forward": y, "ntt_inverse": z})
    ms_total = max_over_ranks(ms_total, world)
    ms_step = ms_total / args.steps
    value = whole_job_value(2 * batch, world, ms_step * 1e-3)

    # ---- roofline of the forward transform (its kernels, events on the launch stream)
    fe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ie = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        fe[k][0].record(); ntt.ComputeForward(y, x, 1, 1); fe[k][1].record()
        ie[k][0].record(); ntt.ComputeInverse(z, y, 1, 1); ie[k][1].record()
    barrier()
    fwd_ms = statistics.mean(a.elapsed_time(b) for a, b in fe)
    inv_ms = statistics.mean(a.elapsed_time(b) for a, b in ie)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
    alg_bytes = 16.0 * n * batch
    achieved = alg_bytes / (fwd_ms * 1e-3) / 1e9
    # DRAM traffic of the same call from the committed ncu capture -- believed only if it was taken on this code
    traffic, traffic_note = None, "no profiles/traffic.json"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("source_hash") == source_hash():
            per_poly = tj.get("ntt_forward_bytes_per_polynomial")
            traffic = per_poly * batch if per_poly else tj.get("ntt_forward_bytes_per_launch")
            traffic_note = f"ncu capture {tj.get('tag')} on this source ({tj.get('source_hash')}), scaled to the batch"
        else:
            traffic_note = (f"profiles/traffic.json ({tj.get('tag')}) was captured on other kernel sources "
                            f"({tj.get('source_hash')} != {source_hash()}): not reported")
    except (OSError, ValueError):
        pass
    roofline = {"bound": "hbm", "kernel": "hexl_b200_ntt_forward (all kernels of one call)", "achieved": achieved,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_note,
                "algorithmic_bytes_per_launch": alg_bytes, "fwd_ms": fwd_ms, "inv_ms": inv_ms,
                "inv_achieved": alg_bytes / (inv_ms * 1e-3) / 1e9,
                "butterflies_per_ntt": (n // 2) * args.logn}
    # The bound that actually binds 64-bit moduli (DESIGN.md 4.1/6): the FMA-heavy integer pipe.
    # A Shoup butterfly is >= 5 IMAD.WIDE + 4 IMAD = 31 pipe cycles per warp (measured issue
    # intervals 4.6 / 2 cycles, tools/pipe_bench.cu), one such pipe per SM sub-partition.
    if q >= (1 << 30):
        sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        peak_bf = sms * 4 * 32 * sm_mhz * 1e6 / 31.0
        ach_bf = batch * (n // 2) * args.logn / (fwd_ms * 1e-3)
        roofline["secondary"] = {"bound": "int-multiply pipe (IMAD/IMAD.WIDE)", "achieved": ach_bf / 1e9,
                                 "peak": peak_bf / 1e9, "unit": "G butterflies/s", "frac": ach_bf / peak_bf,
                                 "model": f"{sms} SMs x 4 sub-partitions x 32 lanes x {sm_mhz:.0f} MHz (sampled under load) "
                                          "/ 31 pipe cycles per warp-butterfly"}

    # ---- eltwise kernels (BASELINE configs[2])
    elt = None
    if not args.no_eltwise and rank == 0:
        elt = eltwise_sweep(hb, torch, peak, g, torch.cuda.synchronize)
    barrier()

    # ---- end to end through the host-pointer path of the C ABI: the same per-GPU batch at every N
    e2e = None
    if not args.no_e2e:
        eb = args.e2e_batch or min(batch, 2048)   # 1 GiB per pinned buffer per rank
        hx = hy = hz = None
        while eb >= 64:
            try:
                hx, hy, hz = (hb.pinned_empty(n * eb) for _ in range(3))
                break
            except hb.HexlB200Error:
                hx = hy = hz = None
                eb //= 2
        # every rank must run the same number of units (and the same barriers): agree on the minimum
        agreed = int(-max_over_ranks(-float(eb if hx is not None else 0), world))
        if agreed < 64:
            hx = None
        elif agreed < eb:
            eb = agreed
            hx, hy, hz = hx[:n * eb], hy[:n * eb], hz[:n * eb]
        if hx is not None:
            rng = np.random.default_rng(7 + rank)
            hx[:] = rng.integers(0, q, size=n * eb, dtype=np.uint64)

            def estep():
                ntt.ComputeForward(hy, hx, 1, 1)   # H2D, kernels, D2H inside the call
                ntt.ComputeInverse(hz, hy, 1, 1)

            estep()
            assert (hz == hx).all(), "e2e round trip failed"
            esteps = args.e2e_steps or max(3, min(args.steps, 10))
            esampler = ClockSampler(local)
            if rank == 0:
                esampler.start()
                esampler.wait_first()
            barrier()
            t0 = time.perf_counter()
            for _ in range(esteps):
                estep()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            dt = max_over_ranks(dt, world)
            eclk = esampler.stop() if rank == 0 else None
            link = 2 * 8 * n * eb * esteps / dt / 1e9
            e2e = {"value": whole_job_value(2 * eb * esteps, world, dt), "unit": "NTT/s",
                   "h2d_bytes_per_step": 2 * 8 * n * eb, "d2h_bytes_per_step": 2 * 8 * n * eb,
                   "batch_per_gpu": eb, "steps": esteps, "ms_per_step": 1e3 * dt / esteps,
                   "link_GBps_each_way_per_gpu": link, "clocks": eclk, "numa": numa,
                   "path": "hexl_b200_ntt_forward/inverse with pinned HOST pointers (library stages H2D/kernel/D2H in 32 MiB chunks on 3 streams)",
                   "bound": "PCIe: every transform moves 8N bytes in and 8N bytes out over the host link"}
            # What the host memory system gives this rank while every other rank asks for the same: 4 threads per rank
            # copy pinned buffer to pinned buffer at once (numpy releases the GIL).  A staged transform reads 8N host bytes
            # and writes 8N host bytes per polynomial: `host_traffic_GBps_per_gpu` (the DMA's reads + writes) against
            # `host_copy_GBps_per_gpu` (the CPUs' reads + writes under the same contention) says whether the e2e rate at
            # N GPUs is limited by the host's DRAM / fabric rather than by the PCIe link of one GPU.
            try:
                nth = 4
                seg = (n * eb) // nth
                barrier()
                t0 = time.perf_counter()
                th = [threading.Thread(target=lambda i=i: hy.__setitem__(slice(i * seg, (i + 1) * seg), hx[i * seg:(i + 1) * seg]))
                      for i in range(nth)]
                [t.start() for t in th]; [t.join() for t in th]
                dt_copy = max_over_ranks(time.perf_counter() - t0, world)
                e2e["host_copy_GBps_per_gpu"] = 2 * 8 * seg * nth / dt_copy / 1e9
                e2e["host_traffic_GBps_per_gpu"] = 2 * link
            except (RuntimeError, ValueError):
                pass
            for buf in (hx, hy, hz):
                hb.pinned_free(buf)

    # ---- the composite configurations
    os.sched_setaffinity(0, affinity0)  # the CPU legs use every host core this process owns
    cpu_ok = rank == 0 and world == 1 and not args.no_cpu
    c4 = c5 = None
    if not args.no_composites:
        del z
        torch.cuda.empty_cache()
        c4 = c4_leg(args, hb, torch, rank, world, g, barrier, peak, cpu_ok)
        barrier()
        c5 = c5_leg(args, hb, torch, rank, world, g, barrier, cpu_ok)
        barrier()
        z = torch.empty_like(x)
        ntt.ComputeInverse(z, y, 1, 1)
        torch.cuda.synchronize()

    # ---- CPU baseline (rank 0, single-GPU runs only)
    cpu = None
    if cpu_ok:
        threads = cpu_threads()
        polys = max(threads * 32, 128)
        # a bounded sample: at least 3 passes and about one second of wall clock on all host threads (~10-30 core-seconds)
        v, kind, tier = cpu_leg(n, q, threads, polys, 3, 1.0)
        cpu = {"value": v, "unit": "NTT/s", "cores": threads, "kind": kind,
               "sample": f"{polys} polynomials x (forward + inverse), best of {cpu_leg.last['reps']} passes "
                         f"({cpu_leg.last['seconds']:.1f} s on {threads} threads), tier {tier}"}
        # The checker also looks at what the timed kernels produced: 256 polynomials spread over the batch, the
        # forward output y compared ON THE DEVICE with the reference's output bit for bit, and the round trip z
        # (outside every timed region).
        import oracle
        chk = oracle.best_checker()
        count = min(256, batch)
        idx = torch.arange(count, device="cuda") * (batch // count)
        hx = x[idx].cpu().numpy().view(np.uint64).reshape(-1)
        exp = torch.from_numpy(chk.ntt_forward(hx, n, q, 1, 1, threads=threads).view(np.int64)).cuda().view(count, n)
        ok = bool(torch.equal(y[idx], exp) and torch.equal(z[idx], x[idx]))
        fold = int(torch.bitwise_xor(y[idx].view(-1)[0::2], y[idx].view(-1)[1::2]).sum().item()) & ((1 << 64) - 1)
        cpu["parity"] = {"polynomials_checked": count, "bit_exact": ok, "checker": chk.kind,
                         "compared": "on the device, every coefficient", "fold64_of_forward_output": fold}
        assert ok, "device results differ from the checker"

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "NTT/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": f"batched Fwd+Inv NTT (configs[1]), N=2^{args.logn}, {args.bits}-bit prime q={q}, "
                                   f"batch={batch} polynomials per GPU, out of place",
                       "parallelism": f"{world} x independent shards, no data-path collective",
                       "l2": f"inputs ({8 * n * batch >> 20} MiB per buffer per GPU) exceed the 126 MB L2; no flush needed"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "eltwise": elt, "c4": c4, "c5": c5,
        }
        print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
