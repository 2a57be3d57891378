#!/usr/bin/env python
"""bench.py -- contract benchmark of the B200-native RNS ring engine.

Metric (BASELINE.json): CKKS ciphertext x ciphertext MulRelin (+ Rescale) per second at N = 2^16, L = 44
(44 Q-limbs + 4 P-limbs: the synthetic literal LogQ = [56] + [45]*43, LogP = [55]*4 of SURVEY 8), plus the
NTT's achieved HBM roofline fraction.

  python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the CPU arm: the oracle ("port" of the reference's
                                                           pure-Go path; Go is not installed) on all host cores
  python bench.py ... --dump-outputs DIR                   also writes a seeded sample of the last timed step's output
                                                           (write_dump) for output-for-output comparison of two builds

A "step" = one pass of MulRelinNew + Rescale over a batch of `--batch` synthetic ciphertext pairs per GPU
(uniform residues, random evaluation key: SURVEY 8(d)). `value` times the device-resident path (inputs already
in HBM; the batch is > L2 so no flush is needed), `e2e` the same op through the C ABI's host-buffer entry point
with H2D / D2H inside the timed region. Ciphertexts shard one batch per GPU, evaluation key broadcast once over
NCCL at setup, no collective on the hot path (weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "CKKS ct x ct mul+relin(+rescale)/s at N=2^16 L=44"
UNIT = "ct/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default="CKKS_L44")
    ap.add_argument("--batch", type=int, default=64, help="ciphertext pairs per GPU per step")
    ap.add_argument("--cpu-sample-pairs", type=int, default=0, help="(reference arm) pairs per step; 0 = one per core")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunk", type=int, default=2, help="ciphertext pairs per pipeline chunk of the host entry point (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="mulrelin", choices=["mulrelin", "bootstrap"],
                    help="bootstrap: BASELINE config 5 -- replay of the op trace of one CKKS bootstrapping (use --preset BOOT_N16QP1767)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's output ciphertexts (rank 0) to DIR as .npy files")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "mulrelin"):
        ap.error("--dump-outputs needs --impl ours --workload mulrelin")
    return args


# Output sample of --dump-outputs: DUMP_SAMPLES flat positions drawn with a fixed seed, so that two builds given the same
# arguments (hence the same seeded inputs) can be compared output for output. Residues reach 2^56, past float64's 53-bit
# mantissa, so each one is stored exactly as its high and low 32-bit halves. 3 float64 arrays x 2^21 entries = 50 MB.
DUMP_SAMPLES = 1 << 21
DUMP_SEED = 20261017


def dump_sample_index(numel):
    """Sorted, distinct flat positions into an output of `numel` residues (all of them when it is small)."""
    import numpy as np
    if numel <= DUMP_SAMPLES:
        return np.arange(numel, dtype=np.int64)
    return np.unique(np.random.default_rng(DUMP_SEED).integers(0, numel, DUMP_SAMPLES, dtype=np.int64))


def write_dump(dirname, out_shape, idx, vals):
    """Writes the sampled residues `vals` (uint64, at flat positions `idx` of an output of shape `out_shape`)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    vals = np.asarray(vals, dtype=np.uint64)
    arrays = {"ct_out_hi32": vals >> np.uint64(32), "ct_out_lo32": vals & np.uint64(0xFFFFFFFF), "ct_out_index": idx,
              "ct_out_shape": np.asarray(out_shape)}
    for name, arr in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), arr.astype(np.float64))


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path restated in C (oracle/lattigo_cpu_batch.c; Go is not installed), run the way the
# reference runs its own parallel benchmark: one thread per ciphertext pair sharing read-only inputs and keys
# (b.RunParallel, schemes/ckks/ckks_benchmarks_test.go:218-229), per-thread scratch reused like sync.Pool
# (ring/pool.go:10-61), built -O3 -march=native on the box it runs on. Threads = the CPUs this process may really use
# (affinity mask capped by the cgroup quota: the pool's GPU boxes show 128 logical CPUs but grant a 16-CPU quota, which
# is what made the round-1 fork pool of os.cpu_count() workers irreproducible).
# ----------------------------------------------------------------------------------------------------------
def _mem_available_bytes():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                return int(ln.split()[1]) * 1024
    except OSError:
        pass
    return None


def run_cpu_arm(args, steps, warmup, pairs_per_step=0, curve=True):
    """Times `steps` steps of `pairs_per_step` ciphertext pairs (default: one per usable CPU) in ONE process with a native
    thread per pair slot. Returns the throughput, the usable-CPU report and a 1/8/32/all-thread scaling curve."""
    import numpy as np
    from lattigo_b200 import params as presets      # pure-Python parameter literals (does not load the CUDA library)
    from oracle import cpu_batch as CB
    from oracle import oracle as O
    CB.lib()                                        # dlopen before any timing (and visible to the driver's loader hook)
    cpus = CB.usable_cpus()
    s = presets.PRESETS[args.preset]
    params = O.Parameters(s["logN"], s["Q"], s["P"])
    N = params.N()
    rng = np.random.default_rng(1234)
    level, levelP = len(s["Q"]) - 1, len(s["P"]) - 1
    nd = params.BaseRNSDecompositionVectorSize(level, levelP)

    def rand_rows(ms, lead):
        out = np.empty(tuple(lead) + (len(ms), N), dtype=np.uint64)
        for i, m in enumerate(ms):
            out[..., i, :] = rng.integers(0, m, tuple(lead) + (N,), dtype=np.uint64)
        return out

    evk = O.GadgetCiphertext(rand_rows(s["Q"] + s["P"], (nd, 1, 2)), level + 1, levelP + 1)
    a = rand_rows(s["Q"], (1, 2)); b = rand_rows(s["Q"], (1, 2))
    plan = CB.CKKSBatchPlan(params, evk)
    threads = cpus["usable"]
    ws_bytes = (9 * (level + 1) + 4 * (levelP + 1) + 2) * N * 8
    avail = _mem_available_bytes()
    if avail is not None and threads * ws_bytes > 0.6 * avail:
        threads = max(1, int(0.6 * avail // ws_bytes))
    pairs = pairs_per_step or threads
    threads = min(threads, pairs)
    per_pair = []
    for _ in range(warmup):                         # also first-touches every thread's workspace
        plan.run(a, b, pairs, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        _, per, _, _ = plan.run(a, b, pairs, threads)
        per_pair += list(per)
    dt = time.perf_counter() - t0
    out = {"value": pairs * steps / dt, "cores": threads, "pairs_per_step": pairs, "steps": steps, "warmup_steps_run": warmup,
           "seconds": dt, "single_pair_seconds_median": sorted(per_pair)[len(per_pair) // 2],
           "cpus": {k: cpus[k] for k in ("affinity", "cgroup_quota", "os_cpu_count", "usable")}}
    if curve:
        pts = []
        for nt in sorted({1, 8, 32, threads}):
            if nt > threads:
                continue
            plan.run(a, b, nt, nt)
            t, per, _, _ = plan.run(a, b, nt, nt)
            pts.append({"threads": nt, "ct_per_s": nt / t, "ct_per_s_per_thread": 1.0 / t, "pair_seconds_median": float(sorted(per)[len(per) // 2])})
        out["curve"] = pts
        out["per_core_efficiency_at_all_threads"] = (out["value"] / threads) / pts[0]["ct_per_s"] if pts else None
    CB.lib().lo_batch_release()
    return out


def _cpu_baseline_record(r):
    return {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
            "sample": "%d warm-up + %d timed steps x %d ciphertext pairs (one per usable CPU), C restatement of the reference CPU path "
                      "(oracle/lattigo_cpu_batch.c, gcc -O3 -march=native, one thread per pair)" % (r["warmup_steps_run"], r["steps"], r["pairs_per_step"]),
            "cpus": r["cpus"], "single_pair_seconds_median": r["single_pair_seconds_median"], "curve": r.get("curve"),
            "per_core_efficiency_at_all_threads": r.get("per_core_efficiency_at_all_threads")}


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    r = run_cpu_arm(args, args.steps, args.warmup, args.cpu_sample_pairs)
    from lattigo_b200 import params as presets
    P = presets.PRESETS[args.preset]
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        # same workload description (same keys) as the product arm; each step is a bounded sample of it: one ciphertext pair
        # per usable host CPU instead of the 64 pairs per GPU (see cpu_baseline.sample)
        "config": _config(args, P, args.gpus),
        "cpu_baseline": _cpu_baseline_record(r),
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def _config(args, P, world):
    """Workload description shared verbatim by both arms (the driver compares the two `config` objects)."""
    nbytes = 2 * args.batch * 2 * len(P["Q"]) * (1 << P["logN"]) * 8
    return {"workload": "ckks_mulrelin_rescale", "preset": args.preset, "logN": P["logN"], "q_limbs": len(P["Q"]), "p_limbs": len(P["P"]),
            "batch_per_gpu": args.batch, "global_batch": args.batch * world,
            "parallelism": "dp%d (one batch per GPU, evk broadcast once)" % world,
            "l2_policy": "inputs (%.1f GB per GPU) exceed L2; no flush" % (nbytes / 1e9),
            "timing": "CUDA events on the launching stream, max over ranks (GPU arm); wall clock around the native batch loop (CPU arm)"}


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(gpu_index):
    """Pins this process (and therefore the pinned host buffers it first-touches afterwards) to the CPUs of the NUMA node the GPU hangs off:
    the e2e path moves 8.8 GB per step over PCIe, and host memory on the far socket costs a third of the H2D bandwidth (round-1 SCALE run:
    0.69 efficiency at 8 GPUs with unbound ranks). Returns a description for the JSON line; never fails the benchmark."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=20).stdout.strip().lower()
        if not bus:
            return {"bound": False, "why": "no pci.bus_id"}
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"bound": False, "why": "numa_node = -1 (single node or not reported)", "pci": bus}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus |= set(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"bound": False, "why": "no allowed CPU on node %d" % node, "pci": bus}
        os.sched_setaffinity(0, allowed)
        return {"bound": True, "numa_node": node, "cpus": len(allowed), "pci": bus}
    except Exception as ex:  # noqa: BLE001
        return {"bound": False, "why": repr(ex)[:120]}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t_end = time.time() + 5.0                      # first line = NVML is up and polling
            while not self.lines and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0=None, t1=None):
        """Samples that arrived inside [t0, t1] (host wall clock of the timed region; the poller itself is started BEFORE the warm-up so that its
        start-up -- NVML initialisation takes driver locks for a few hundred ms -- never overlaps a timed step). A region shorter than the 100 ms
        polling period keeps the samples nearest to it."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()          # exact PID, never by pattern
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = list(self.lines)
        if t0 is not None and t1 is not None:
            inside = [r for r in rows if t0 <= r[0] <= t1 + 0.12]
            if len(inside) < 2:
                inside = sorted(rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:3]
            rows = inside
        sm, smax, reasons = [], None, set()
        for _, ln in rows:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "samples": len(sm), "reasons": sorted(reasons)}


def gpu_main(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import lattigo_b200 as lb
    from lattigo_b200 import params as presets, _lib, dist as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)

    s = presets.PRESETS[args.preset]
    logN, Q, P = s["logN"], s["Q"], s["P"]
    N = 1 << logN
    level, levelP = len(Q) - 1, len(P) - 1
    nd = (level + levelP + 1) // (levelP + 1)
    ctx = lb.Context(logN, Q, P, device=local)
    g = torch.Generator(device=dev); g.manual_seed(1000 + rank)

    def rand_rows(mods, lead):
        out = torch.empty(tuple(lead) + (len(mods), N), dtype=torch.int64, device=dev)
        for i, m in enumerate(mods):
            out[..., i, :] = torch.randint(0, m, tuple(lead) + (N,), generator=g, device=dev, dtype=torch.int64)
        return out

    # evaluation key: generated on rank 0, broadcast once over NCCL (SURVEY 8(e)); never touched again on the hot path
    evk_t = rand_rows(Q + P, (nd, 1, 2)) if rank == 0 else torch.empty((nd, 1, 2, len(Q) + len(P), N), dtype=torch.int64, device=dev)
    D.broadcast_key(evk_t, src=0)                     # lattigo_b200/dist.py: the plumbing tests/test_multiprocess_cpu.py exercises with gloo
    rlk = lb.GadgetCiphertext(ctx, evk_t, level, levelP)
    ev = lb.CKKSEvaluator(ctx, rlk)
    B = args.batch
    a = rand_rows(Q, (B, 2)); b = rand_rows(Q, (B, 2))
    out = None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return ev.MulRelinRescaleNew(a, b)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        out = step()
    barrier()
    l0 = _lib.lib().lgpu_launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    barrier()
    w1 = time.time()
    launches = _lib.lib().lgpu_launch_count() - l0
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    t_dev = e0.elapsed_time(e1) * 1e-3
    t_max = D.max_over_ranks(t_dev, dev)
    value = D.job_throughput(B * args.steps, t_dev, dev)
    dump = None
    if args.dump_outputs and rank == 0:
        idx = dump_sample_index(out.numel())
        dump = (tuple(out.shape), idx, out.reshape(-1)[torch.from_numpy(idx).to(dev)].cpu().numpy().view(np.uint64))

    # ---- roofline of the dominant kernel class (NTT): same K steps with the event profiler on --------------------
    roof = None
    if rank == 0:
        import ctypes
        L = _lib.lib()
        nk = 9
        ms = (ctypes.c_double * nk)(); by = (ctypes.c_double * nk)()
        sc = (ctypes.c_ulonglong * nk)(); kn = (ctypes.c_ulonglong * nk)()
        L.lgpu_profile_enable(1)
        for _ in range(args.steps):
            out = step()
        torch.cuda.synchronize()
        L.lgpu_profile_enable(0)
        L.lgpu_profile_read(ms, by, sc, kn)
        names = ["ntt_fwd", "ntt_inv", "vecop", "modup", "mac", "tensor", "automorphism", "fused", "epilogue"]
        classes = {names[i]: {"ms": ms[i], "alg_GB": by[i] / 1e9, "scopes": int(sc[i]), "kernels": int(kn[i]),
                              "alg_GBs": (by[i] / 1e9) / (ms[i] * 1e-3) if ms[i] > 0 else None} for i in range(nk) if sc[i]}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
        tot = sum(ms[i] for i in range(nk)) or 1.0
        # dominant kernel class of the step (by summed CUDA-event time of its launch scopes)
        dom = max(range(nk), key=lambda i: ms[i])
        kernel_names = {
            "mac": "ks_chunk_mac_fp8r_kernel (K3: chunk-pass NTT, 12 stages on the FP64 pipe, + key-switch MAC over all digits from registers)",
            "fused": "ks_strided_j4_kernel (K2: basis extension folded into the strided NTT pass, y/v tile shared by 8 target rows)",
            "epilogue": "fz_chunk_epi_fp8_kernel (chunk-pass NTT + ModDown / Rescale epilogue from registers)",
            "ntt_fwd": "ntt strided + chunk pass kernels (forward)", "ntt_inv": "ntt chunk + strided pass kernels (inverse)",
            "modup": "ks_prepare_kernel / modup_kernel", "vecop": "vecop_kernel", "tensor": "ckks_tensor_kernel",
            "automorphism": "auto_ntt_kernel"}
        ach = (by[dom] / 1e9) / (ms[dom] * 1e-3) if ms[dom] > 0 else 0.0
        traffic = None
        try:
            # ncu dram bytes of the class's launches per ciphertext pair (one --set full capture, see the file), scaled to
            # the average launch scope of this run: per_ct x pairs per step / scopes per step
            import glob
            tr = json.load(open(sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]))   # newest round's capture
            ent = tr.get(names[dom])
            if ent and ent.get("preset") == args.preset:
                traffic = ent["dram_bytes_per_ct"] * B * args.steps / max(1, int(sc[dom]))
        except Exception:
            pass
        # standalone transform rate (BASELINE metric "NTT GB/s vs roofline"): Ring.NTT on all Q limbs of the preset,
        # 16 polynomials per launch (369 MB in + 369 MB out > L2), CUDA events around `iters` launches
        xs = rand_rows(Q, (16,)); ys = torch.empty_like(xs)
        rq = ctx.ringQ
        for _ in range(3):
            rq.NTT(xs, ys)
        torch.cuda.synchronize()
        ea = torch.cuda.Event(enable_timing=True); eb = torch.cuda.Event(enable_timing=True)
        iters = 20
        ea.record()
        for _ in range(iters):
            rq.NTT(xs, ys)
        eb.record(); torch.cuda.synchronize()
        t_ntt = ea.elapsed_time(eb) * 1e-3 / iters
        ntt_bytes = 16.0 * N * len(Q) * 16
        ntt_standalone = {"op": "Ring.NTT, %d limbs x 16 polynomials, N=2^%d" % (len(Q), logN), "us_per_launch": t_ntt * 1e6,
                          "us_per_limb_transform": t_ntt * 1e6 / (len(Q) * 16), "alg_bytes_per_launch": ntt_bytes,
                          "achieved": ntt_bytes / t_ntt / 1e9, "unit": "GB/s", "frac": ntt_bytes / t_ntt / 1e9 / peak}
        del xs, ys
        roof = {"bound": "hbm", "kernel": kernel_names.get(names[dom], names[dom]), "kernel_class": names[dom],
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                "traffic": traffic, "avg_launch_ms": ms[dom] / max(1, int(sc[dom])), "alg_bytes_per_launch": by[dom] / max(1, int(sc[dom])),
                "share_of_step": ms[dom] / tot, "ntt_standalone": ntt_standalone, "classes": classes,
                "note": "classes: summed CUDA-event time of launch scopes over the same K steps re-run with the event profiler on; "
                        "all chains run on the caller's stream, so class times do not overlap and add up to the step"}
    barrier()

    # ---- e2e through the host-buffer C-ABI entry point (pinned host memory, copies inside the timed region) ------
    e2e = None
    if not args.no_e2e:
        nq = level + 1
        ha = torch.empty((B, 2, nq, N), dtype=torch.int64).pin_memory()
        hb = torch.empty((B, 2, nq, N), dtype=torch.int64).pin_memory()
        ho = torch.empty((B, 2, nq - 1, N), dtype=torch.int64).pin_memory()
        ha.copy_(a); hb.copy_(b)
        torch.cuda.synchronize()
        na, nb_, no = ha.numpy().view(np.uint64), hb.numpy().view(np.uint64), ho.numpy().view(np.uint64)
        ev.MulRelinRescaleHost(na, nb_, no, chunk=args.e2e_chunk)     # warm-up (allocators, page touching)
        barrier()
        t0 = time.perf_counter()
        e2e_steps = max(1, min(args.steps, 3))
        for _ in range(e2e_steps):
            ev.MulRelinRescaleHost(na, nb_, no, chunk=args.e2e_chunk)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        td = torch.tensor([D.max_over_ranks(dt, dev)], dtype=torch.float64)
        e2e_ok = bool(torch.equal(ho.to(dev), out)) if out is not None else None
        e2e = {"value": B * world * e2e_steps / float(td.item()), "unit": UNIT, "h2d_bytes_per_step": int(2 * ha.numel() * 8),
               "d2h_bytes_per_step": int(ho.numel() * 8), "steps": e2e_steps, "matches_device_path": e2e_ok,
               "entry_point": "lgpu_ckks_mulrelin_rescale_batch_host (pinned host buffers, 2-stream chunked pipeline)", "chunk": args.e2e_chunk,
               "numa": numa, "h2d_GBs": 2 * ha.numel() * 8 * e2e_steps / float(td.item()) / 1e9}
        del ha, hb, ho
    barrier()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # bounded CPU sample in a separate process (native thread pool there; this process holds a CUDA context)
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                    "--preset", args.preset], capture_output=True, text=True, timeout=900)
                ref = json.loads(r.stdout.strip().splitlines()[-1])
                cpu = ref["cpu_baseline"]
            except Exception as ex:  # noqa: BLE001
                cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": "failed: %r" % (ex,)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": _config(args, s, world),
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "roofline": roof, "cpu_baseline": cpu,
        }
        if dump is not None:
            write_dump(args.dump_outputs, *dump)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------------------------------------
# BASELINE config 5: CKKS bootstrapping throughput by op-trace replay (lattigo_b200/boottrace.py + bootreplay.py)
# ----------------------------------------------------------------------------------------------------------
def bootstrap_main(args):
    import torch
    import torch.distributed as dist
    import lattigo_b200 as lb
    from lattigo_b200 import params as presets, _lib, boottrace
    from lattigo_b200.bootreplay import BootstrapReplay
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "no CPU restatement of circuits/ckks/bootstrapping exists in oracle/ (Go is not installed); "
                              "the bootstrap workload is an op-trace replay of the device path only"}))
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    s = presets.PRESETS[args.preset]
    ctx = lb.Context(s["logN"], s["Q"], s["P"], device=local)
    g = torch.Generator(device=dev); g.manual_seed(2000 + rank)
    n_res = 14 if args.preset == "BOOT_N16QP1767" else max(1, len(s["Q"]) - 16)
    trace = boottrace.bootstrap_trace(logN=s["logN"], residual_limbs=n_res)
    rep = BootstrapReplay(ctx, args.batch, g, trace)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        rep.run()
    barrier()
    l0 = _lib.lib().lgpu_launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    phases = {}
    barrier()
    w0 = time.time()
    e0.record()
    for _ in range(args.steps):
        ms, nops = rep.run()
        for k, v in ms.items():
            phases[k] = phases.get(k, 0.0) + v
    e1.record()
    barrier()
    w1 = time.time()
    launches = _lib.lib().lgpu_launch_count() - l0
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    from lattigo_b200 import dist as D
    t_max = D.max_over_ranks(e0.elapsed_time(e1) * 1e-3, dev)
    alg = None
    if rank == 0:
        import ctypes
        L = _lib.lib()
        nk = 9
        msa = (ctypes.c_double * nk)(); by = (ctypes.c_double * nk)(); sc = (ctypes.c_ulonglong * nk)(); kn = (ctypes.c_ulonglong * nk)()
        L.lgpu_profile_enable(1)
        rep.run()
        torch.cuda.synchronize()
        L.lgpu_profile_enable(0)
        L.lgpu_profile_read(msa, by, sc, kn)
        names = ["ntt_fwd", "ntt_inv", "vecop", "modup", "mac", "tensor", "automorphism", "fused", "epilogue"]
        alg = {"sum_alg_GB_per_step": sum(by) / 1e9, "classes": {names[i]: {"ms": msa[i], "alg_GB": by[i] / 1e9, "kernels": int(kn[i])} for i in range(nk) if sc[i]}}
    barrier()
    if rank == 0:
        line = {"metric": "CKKS bootstraps/s (op-trace replay of circuits/ckks/bootstrapping, N16QP1767H32768H32 shapes)", "value": args.batch * world * args.steps / t_max,
                "unit": "bootstraps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_max / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": "ckks_bootstrap_replay", "preset": args.preset, "logN": s["logN"], "q_limbs": len(s["Q"]), "p_limbs": len(s["P"]),
                           "batch_per_gpu": args.batch, "global_batch": args.batch * world, "ops_per_bootstrap": len(trace), "galois_keys": rep.n_galois_keys,
                           "trace": boottrace.summarize(trace),
                           "l2_policy": "working set (keys, diagonals, batch) far exceeds L2; no flush", "timing": "CUDA events, max over ranks"},
                "clocks": clocks, "gpu_launches": int(launches), "phase_ms_per_step": {k: v / args.steps for k, v in phases.items()},
                "algorithmic_bytes": alg, "e2e": None, "cpu_baseline": None}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.workload == "bootstrap":
        return bootstrap_main(args)
    if args.impl == "reference":
        return reference_main(args)
    return gpu_main(args)


if __name__ == "__main__":
    sys.exit(main())
