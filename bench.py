#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native `bcftools call -m` hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     (also writes the last timed step's results, see dump_outputs)

Metric (BASELINE.json): sample-genotype calls per second (one call = one (sample, site) genotype call).
Workload at N=1 (config.workload): BASELINE.json configs[2] "C3" -- 2,504 samples (1000G-shaped), 2-5 alleles per
site (70/20/7/3 %), allele trimming on, FORMAT/GQ requested.  This is the config the north-star target is quoted on
and it fits one GPU.  A STEP is one pass of the hot path over one batch of `--sites` sites (default 16,384 unique
synthetic sites replicated x4 in HBM = 65,536 sites, 2.9 GB of PL; the 1M-site job is 15.3 such steps).

  value     device-resident throughput: inputs already in HBM, CUDA events on the launching stream, max over ranks
  e2e       the same metric through the C-ABI host entry point mcb_call_host with pinned HOST buffers:
            H2D of the PL slab + kernels + D2H of GT/GQ/PL/site records inside the timed region
  roofline  dominant kernel (mcall_biallelic_warp_kernel, the two-allele class): algorithmic bytes of its sites / its own device time;
            roofline.per_class has the same figures for every allele-count class, roofline.all_kernels for the whole step
  sustained the same step repeated for >= --sustain seconds with its own clock samples (the headline region lasts ~50 ms)
  secondary BASELINE config 5 (mixed ploidy) pooled and with 5 -G groups, device-resident
  job       N > 1 only: ONE C4-shaped job over all N GPUs through mcb_job_call_host (strong scaling; rank 0 drives it)
  cpu_baseline  the CPU oracle on this box's host cores on a bounded sample of the same workload (rank 0, N=1)

The reference arm times the reference's own CPU implementation of the path (oracle/_ref = the unmodified mcall.c
compiled against the htslib stub; falls back to the plain-C port when that library was not built) with one process
per host core over contiguous site shards.  Rank 0 alone runs it.
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
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)

METRIC = "sample_genotype_calls_per_s"
UNIT = "calls/s"
WORKLOAD = "C3"
# --dump-outputs: at most 65,536 sites (every site of the default step) with their per-site fields, 128 of them with their
# per-sample outputs (GT, GQ, PL); at 2,504 samples that is at most ~56 MB of float64 whatever --sites / --replicate are
DUMP_SITES = 65536
DUMP_SAMPLE_SITES = 128
DUMP_SEED = 0xB200D


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clocks and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML every ~5 ms,
    falling back to the nvidia-smi query of the recipe when pynvml is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx, self.stop_flag = gpu_index, False
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)))
        try:
            self.power.append(n.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
        except Exception:
            pass
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        if len(r) >= 9:
            self.sm.append(float(r[1])); self.mx.append(float(r[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            time.sleep(0.005 if self.nvml else 0.1)

    def summary(self):
        return dict(sm_mhz=float(np.median(self.sm)) if self.sm else None, sm_max_mhz=max(self.mx) if self.mx else None,
                    reasons=sorted(self.reasons), samples=len(self.sm), power_w_max=max(self.power) if self.power else None,
                    source="nvml" if self.nvml else "nvidia-smi")


def shard_batch(batch, nproc):
    """Contiguous site shards, one per process (built before the timed region)."""
    R = batch.nsites
    return [batch.subset(range(R * i // nproc, R * (i + 1) // nproc)) for i in range(nproc) if R * (i + 1) // nproc > R * i // nproc]


class OraclePool:
    """One forked worker per shard, started once; every step() runs the CPU oracle over all shards in parallel
    and returns the wall seconds between the start and the end barrier (fork cost stays outside the timing)."""

    def __init__(self, params, shards, tab, kind, nsteps):
        import multiprocessing as mp
        from oracle import pyoracle
        pyoracle._load(kind)
        ctx = mp.get_context("fork")
        n = len(shards)
        self.start, self.done = ctx.Barrier(n + 1), ctx.Barrier(n + 1)

        def work(shard):
            from bcftools_b200 import abi
            res = abi.HostResult(shard)         # allocated once, outside the timed steps
            for _ in range(nsteps):
                self.start.wait()
                pyoracle.call(kind, params, shard, tab, result=res)
                self.done.wait()

        self.procs = [ctx.Process(target=work, args=(sh,), daemon=True) for sh in shards]
        for p in self.procs:
            p.start()

    def step(self):
        self.start.wait()
        t0 = time.perf_counter()
        self.done.wait()
        return time.perf_counter() - t0

    def close(self):
        for p in self.procs:
            p.join(timeout=10)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    import platform
    return platform.processor() or platform.machine()


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from bcftools_b200 import synth
    from oracle import pyoracle
    pyoracle.build(want_ref=True)
    kind = "reference" if pyoracle.have_ref() else "port"
    ncores = os.cpu_count() or 1
    sites = args.ref_sites
    params, batch, tab = synth.make_batch(WORKLOAD, sites, with_groups=0)
    shards = shard_batch(batch, ncores)
    pool = OraclePool(params, shards, tab, kind, args.warmup + args.steps)
    for _ in range(args.warmup):
        pool.step()
    dt = 0.0
    for _ in range(args.steps):
        dt += pool.step()
    pool.close()
    value = args.steps * sites * params.nsmpl / dt
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=dict(workload=WORKLOAD, nsmpl=params.nsmpl, sites_per_step=sites,
                                              note="bounded sample of the same synthetic workload; reference arithmetic is single-threaded "
                                                   "(--threads n/a, vcfcall.c:692), parallelised as one process per core over site shards"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=ncores, cpu_model=cpu_model(), threads_flag="--threads n/a (output compression only, vcfcall.c:692)",
                                  kind=kind, sample=f"{sites} sites x {params.nsmpl} samples per step"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(gpu_index):
    """Multi-GPU runs: keep this rank's threads (and therefore its first-touched pinned buffers) on the CPUs NVML reports
    as local to the GPU, so that N ranks do not push their PCIe traffic through one socket.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def kernel_source_hash():
    """sha256 over the CUDA sources: the committed ncu capture is only quoted when it was taken from these very kernels."""
    import glob
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "bcftools_b200", "csrc")
    for f in sorted(glob.glob(os.path.join(csrc, "*.cu")) + glob.glob(os.path.join(csrc, "*.cuh"))):
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(sites_per_step):
    """DRAM bytes (read + write) per launch of every class kernel, from the committed `ncu --set full` capture of this same
    command (profiles/r02_ncu_kernels.json, written by scripts/ncu_kernels_json.py).  The capture is refused -- loudly --
    when it was taken from other kernel sources or another step size."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_kernels.json")
    try:
        d = json.load(open(path))
    except (OSError, ValueError):
        return {}, "no ncu capture committed"
    if d.get("sites_per_step") != sites_per_step:
        return {}, "ncu capture is for %s sites per step" % d.get("sites_per_step")
    if d.get("kernel_source_hash") != kernel_source_hash():
        sys.stderr.write("bench.py: profiles/r02_ncu_kernels.json was captured from other kernel sources (%s, now %s): traffic not quoted\n"
                         % (d.get("kernel_source_hash"), kernel_source_hash()))
        return {}, "STALE: the ncu capture predates the current kernel sources"
    return {int(k): int(v["dram_bytes_read"] + v["dram_bytes_write"]) for k, v in d.get("classes", {}).items()}, d.get("source", path)


def dump_outputs(out_dir, db, dr):
    """--dump-outputs DIR: the mcb_result arrays of the last timed step as DIR/<name>.npy, so that two builds can be compared
    output for output (the inputs are seeded: the same arguments give the same step).  Site indices are step-wide.
      sites [n]: every site of the step, or a fixed seeded sample of DUMP_SITES of them in a larger step; for these sites
        ret, als_new, site_flags, an, qual [n]; als_map, ac [n, max_nals]; diag [n, 4]
      sample_sites [k]: a fixed seeded sample of DUMP_SAMPLE_SITES of them; for these sites gt [k, nsmpl, 2], gq [k, nsmpl],
        and their trimmed PL blocks concatenated in pl, the block of sample site j at pl[pl_site_offsets[j]:pl_site_offsets[j+1]]
        ([nsmpl][G'] row-major; empty where ret <= 0 or the PLs were dropped)
    qual is float32 as computed; every integer array is widened to float64, exact (the INT32 missing / vector-end sentinels
    stay distinct)."""
    import torch
    from bcftools_b200 import abi
    t, R, S = dr.t, db.nsites, db.nsmpl
    rng = np.random.default_rng(DUMP_SEED)
    sites = np.arange(R) if R <= DUMP_SITES else np.sort(rng.choice(R, size=DUMP_SITES, replace=False))
    smp = np.sort(rng.choice(sites, size=min(DUMP_SAMPLE_SITES, sites.size), replace=False))
    dev = t["gt"].device
    out = dict(sites=sites, sample_sites=smp)
    for name in ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "diag"):
        out[name] = t[name].index_select(0, torch.from_numpy(sites).to(dev)).cpu().numpy().view(abi.RESULT_FIELDS[name])
    for name in ("gt", "gq"):
        if t[name] is not None:
            out[name] = t[name].index_select(0, torch.from_numpy(smp).to(dev)).cpu().numpy()
    ret = t["ret"].cpu().numpy()
    flags = t["site_flags"].cpu().numpy().view(np.uint32)
    blocks, offs = [], [0]
    for i in smp:
        n = int(ret[i])
        g = S * n * (n + 1) // 2 if n > 0 and not (flags[i] & abi.SITE_PL_DROPPED) else 0
        o = int(db.pl_off_host[i])
        blocks.append(t["pl"][o:o + g].cpu().numpy())
        offs.append(offs[-1] + g)
    out["pl"] = np.concatenate(blocks)
    out["pl_site_offsets"] = np.array(offs)
    out = {name: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for name, a in out.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= 64_000_000, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sites", type=int, default=16384, help="unique synthetic sites generated per rank")
    ap.add_argument("--replicate", type=int, default=4, help="HBM copies of the unique sites forming one step")
    ap.add_argument("--e2e-sites", type=int, default=16384, help="sites per mcb_call_host step of the e2e leg (default: every unique site of the synthetic batch)")
    ap.add_argument("--ref-sites", type=int, default=8192)
    ap.add_argument("--cpu-sites", type=int, default=2048)
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of a second, long timed region (clocks under sustained load); 0 = off")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C5 (mixed ploidy, -G groups) secondary workload")
    ap.add_argument("--secondary-sites", type=int, default=2048)
    ap.add_argument("--job-sites-per-gpu", type=int, default=192, help="N>1: C4-shaped sites per GPU of the one-job strong-scaling leg (rank 0 drives all N GPUs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step of rank 0 as DIR/<name>.npy "
                                                          "(the CUDA path only: not with --impl reference)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the CUDA path: not with --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from bcftools_b200 import abi, device, mcall, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 else 0
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # a host-side group: ranks that only WAIT (the one-job leg below) must not park an NCCL kernel on their GPU -- rank 0 drives
    # that GPU from its own context and would be time-sliced against the spinning barrier kernel
    host_group = dist.new_group(backend="gloo") if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload: each rank owns a contiguous range of sites (its own seed offset): weak scaling, no collective
    params, hb, tab = synth.make_batch(WORKLOAD, args.sites, seed_offset=rank, with_groups=0)
    params.device = local_rank
    mc = mcall.MCaller(params, ploidy_tab=tab)
    db = device.DeviceBatch(hb, device=f"cuda:{local_rank}", replicate=args.replicate)
    dr = device.DeviceResult(db)
    b, r = db.c_struct(), dr.c_struct()
    stream = torch.cuda.current_stream().cuda_stream
    calls_per_step = db.nsites * params.nsmpl

    for _ in range(max(3, args.warmup)):
        mc.call_device(b, r, stream)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ktimes = np.zeros(6)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        mc.call_device(b, r, stream)
    e1.record()
    barrier()
    dev_s = e0.elapsed_time(e1) * 1e-3
    launches = int(mc.stats()[0]) * args.steps
    # the legs below reuse the result buffers: the outputs of the timed steps are taken now
    dumped_bytes = dump_outputs(args.dump_outputs, db, dr) if args.dump_outputs and rank == 0 else None
    # ---- sustained leg: the timed region above lasts ~50 ms at boost clocks; these kernels are issue-bound, so a long job
    # runs at whatever clock the power limit settles on.  Same step, >= --sustain seconds, its own clock samples.
    sustained = None
    if args.sustain > 0:
        nsteps_s = max(args.steps, int(args.sustain / max(dev_s / args.steps, 1e-6)) + 1)
        s_samp = ClockSampler(local_rank)
        s_samp.start()
        barrier()
        e0.record()
        for _ in range(nsteps_s):
            mc.call_device(b, r, stream)
        e1.record()
        barrier()
        s_samp.stop_flag = True
        s_samp.join(timeout=2)
        sus_s = e0.elapsed_time(e1) * 1e-3
        if world > 1:
            t = torch.tensor([sus_s], device=f"cuda:{local_rank}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sus_s = float(t.item())
        sustained = dict(value=world * nsteps_s * calls_per_step / sus_s, unit=UNIT, steps=nsteps_s, seconds=sus_s,
                         ms_per_step=1e3 * sus_s / nsteps_s, clocks=s_samp.summary())
    # per-class kernel times of untimed extra steps for the roofline of the dominant kernel: the library serialises the
    # class kernels on the caller's stream and brackets each with events (in the timed region they run on their own
    # streams and overlap at the tails of their persistent grids)
    mc.set_option("time_kernels", 1)
    per_class = []
    for _ in range(5):
        mc.call_device(b, r, stream)
        per_class.append(mc.kernel_times_ms())
    ktimes = np.median(np.array(per_class), axis=0)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- parity spot check of this very run (rank 0): CUDA result of the first sites against the CPU oracle
    res = dr.to_host()
    rd_all, wr_all = synth.algorithmic_bytes(hb, res, params.output_tags)
    parity = None
    cpu = None
    if rank == 0 and not args.no_cpu:
        from oracle import pyoracle
        from tests import parity as par
        pyoracle.build(want_ref=True)
        kind = "reference" if pyoracle.have_ref() else "port"
        n = min(args.cpu_sites, hb.nsites)
        sub = hb.subset(range(n))
        t0 = time.perf_counter()
        exp, secs = pyoracle.call(kind, params, sub, tab)
        got = abi.HostResult(sub)
        for name in abi.RESULT_FIELDS:
            a = getattr(res, name)
            if a is None or getattr(got, name) is None:
                continue
            if name in ("pl", "gp"):
                getattr(got, name)[...] = a[:sub.pl.size]
            else:
                getattr(got, name)[...] = a[:n]
        st = par.compare(got, exp, params)
        parity = dict(sites=n, compared=st["compared"], near_ties=len(st["near_ties"]), qual_max_rel=st["qual_max_rel"], oracle=kind)
        if world == 1:
            cpu = dict(value=n * params.nsmpl / secs, unit=UNIT, cores=1, kind=kind,
                       sample=f"first {n} sites x {params.nsmpl} samples of the step, time inside the per-record calls only")

    # ---- end to end through the host entry point (pinned host buffers, copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        ne = min(args.e2e_sites, hb.nsites)
        sub = mcall.pin_batch(hb.subset(range(ne)))
        hres = mcall.pin_result(abi.HostResult(sub, compact=True))      # trimmed PLs leave the device compacted
        for _ in range(2):
            mc.call_host(sub, hres)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            mc.call_host(sub, hres)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=f"cuda:{local_rank}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        h2d = sum(getattr(sub, k).nbytes for k in ("pl", "pl_off", "nals", "unseen", "qs") if getattr(sub, k) is not None)
        d2h = sum(getattr(hres, k).nbytes for k in ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "diag", "gt", "gq", "pl_off_out")
                  if getattr(hres, k) is not None) + 4 * int(mc.stats()[2])        # + the used (compacted) part of the PL buffer
        e2e = dict(value=world * args.steps * ne * params.nsmpl / dt, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                   host_cpus_bound_per_rank=numa_cpus,
                   sites_per_step=ne, ms_per_step=1e3 * dt / args.steps, pl_transport="int32 (bcf_get_format_int32 layout)")
        # secondary: the same call with the PL slab shipped as BCF int16 typed vectors (mcb_batch.pl_type=2)
        sub16 = mcall.pin_batch(hb.subset(range(ne)).to_int16())
        hres16 = mcall.pin_result(abi.HostResult(sub16, compact=True))
        for _ in range(2):
            mc.call_host(sub16, hres16)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            mc.call_host(sub16, hres16)
        torch.cuda.synchronize()
        dt16 = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt16], device=f"cuda:{local_rank}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt16 = float(t.item())
        e2e["int16_pl_transport"] = dict(value=world * args.steps * ne * params.nsmpl / dt16, h2d_bytes_per_step=int(sub16.pl.nbytes + h2d - sub.pl.nbytes),
                                         ms_per_step=1e3 * dt16 / args.steps)
        # secondary: BCF typed vectors both ways -- int16 PL in, int8 GT / int8 GQ / int16 PL out (mcb_result.gt8/gq8/pl16)
        hrest = mcall.pin_result(abi.HostResult(sub16, compact=True, typed=True))
        for _ in range(2):
            mc.call_host(sub16, hrest)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            mc.call_host(sub16, hrest)
        torch.cuda.synchronize()
        dtt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dtt], device=f"cuda:{local_rank}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtt = float(t.item())
        d2ht = sum(getattr(hrest, k).nbytes for k in ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "diag", "gt8", "gq8", "pl_off_out")
                   if getattr(hrest, k) is not None) + 2 * int(mc.stats()[2])
        e2e["bcf_typed_transport"] = dict(value=world * args.steps * ne * params.nsmpl / dtt, ms_per_step=1e3 * dtt / args.steps,
                                          h2d_bytes_per_step=int(sub16.pl.nbytes + h2d - sub.pl.nbytes), d2h_bytes_per_step=int(d2ht),
                                          types="in: PL int16 (BCF_BT_INT16 as stored in the record); out: GT int8, GQ int8, PL int16, narrowed on the device")

    # ---- secondary workloads (rank 0), device-resident: BASELINE config 5 -- every 2nd sample haploid -- pooled and with 5 -G
    # groups; BASELINE config 2 -- 1,000 diploid samples, two-allele sites only
    secondary = None
    if rank == 0 and not args.no_secondary:
        secondary = {}
        for name, cfg5, nsites5, groups in (("C5_pooled", "C5", args.secondary_sites, 0), ("C5_groups5", "C5", args.secondary_sites, 5),
                                            ("C2", "C2", 4 * args.secondary_sites, 0)):
            p5, h5, t5 = synth.make_batch(cfg5, nsites5, with_groups=groups)
            p5.device = local_rank
            with mcall.MCaller(p5, ploidy_tab=t5) as m5:
                d5 = device.DeviceBatch(h5, device=f"cuda:{local_rank}", replicate=args.replicate)
                r5 = device.DeviceResult(d5)
                b5, rr5 = d5.c_struct(), r5.c_struct()
                for _ in range(3):
                    m5.call_device(b5, rr5, stream)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(5):
                    m5.call_device(b5, rr5, stream)
                e1.record()
                torch.cuda.synchronize()
                s5 = e0.elapsed_time(e1) * 1e-3 / 5
                secondary[name] = dict(value=d5.nsites * p5.nsmpl / s5, unit=UNIT, ms_per_step=1e3 * s5, sites_per_step=d5.nsites, nsmpl=p5.nsmpl,
                                       groups=groups, ploidy="every 2nd sample haploid" if cfg5 == "C5" else "diploid")
            del d5, r5

    # ---- N > 1: ONE job over the N GPUs of the box (mcall_job.h): BASELINE config 4 shape (100,000 samples), contiguous site
    # ranges, host buffers, results concatenated in input order.  Rank 0 drives all devices while the other ranks wait.
    job = None
    if world > 1:
        barrier()
        dist.barrier(group=host_group)
        if rank == 0:
            pj, hj, tj = synth.make_batch("C4", args.job_sites_per_gpu * world)
            hj = mcall.pin_batch(hj)
            rj = mcall.pin_result(abi.HostResult(hj, compact=True))
            job = dict(workload="C4", nsmpl=pj.nsmpl, sites=hj.nsites, scaling="strong: one job, contiguous site ranges balanced by PL volume, ordered concatenation",
                       h2d_bytes=int(hj.pl.nbytes))
            for ndev in sorted({1, world}):
                with mcall.MJob(pj, list(range(ndev))) as jb:
                    jb.call_host(hj, rj)
                    t0 = time.perf_counter()
                    for _ in range(3):
                        jb.call_host(hj, rj)
                    dtj = (time.perf_counter() - t0) / 3
                job["devices_%d" % ndev] = dict(value=hj.nsites * pj.nsmpl / dtj, unit=UNIT, ms_per_call=1e3 * dtj)
            job["speedup"] = job["devices_%d" % world]["value"] / job["devices_1"]["value"]
        dist.barrier(group=host_group)      # the other ranks wait on the host, their GPUs idle
        barrier()

    # ---- max over ranks of the device time
    if world > 1:
        t = torch.tensor([dev_s], device=f"cuda:{local_rank}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_s = float(t.item())
    if rank == 0:
        peak, peak_src = measured_peak()
        # per allele-count class: its sites' algorithmic bytes / its own device time; the dominant kernel is the two-allele one
        traffic, traffic_src = ncu_traffic(db.nsites)
        kernel_names = {2: "mcall_biallelic_warp_kernel", 3: "mcall_multi_kernel<3>", 4: "mcall_multi_kernel<4>", 5: "mcall_multi_kernel<5>"}
        per_class = {}
        for k in range(2, 6):
            isk = hb.nals == k
            if not isk.any() or ktimes[k] <= 0:
                continue
            idx = np.where(isk)[0]
            subk = hb.subset(idx)
            resk = abi.HostResult(subk)
            resk.ret[...] = res.ret[idx]
            resk.site_flags[...] = res.site_flags[idx]
            rdk, wrk = synth.algorithmic_bytes(subk, resk, params.output_tags)
            bk = (rdk + wrk) * args.replicate
            achk = bk / (ktimes[k] * 1e-3) / 1e9
            per_class[str(k)] = dict(kernel=kernel_names[k], sites=int(isk.sum()) * args.replicate, algorithmic_bytes_per_launch=int(bk), kernel_ms=float(ktimes[k]),
                                     achieved=achk, frac=achk / peak, calls_per_s=float(isk.sum() * args.replicate * params.nsmpl / (ktimes[k] * 1e-3)),
                                     traffic=traffic.get(k), traffic_over_algorithmic=(traffic[k] / bk if k in traffic else None))
        roof = None
        if "2" in per_class:
            c2 = per_class["2"]
            roof = dict(bound="hbm", kernel="mcall_biallelic_warp_kernel (the two-allele class: 70 % of the sites of a step)", achieved=c2["achieved"], peak=peak,
                        unit="GB/s", frac=c2["frac"], traffic=c2["traffic"], traffic_source=traffic_src, peak_source=peak_src,
                        algorithmic_bytes_per_launch=c2["algorithmic_bytes_per_launch"],
                        kernel_ms=float(ktimes[2]), kernel_share_of_step=float(ktimes[2] / ktimes[0]),
                        per_class=per_class,
                        all_kernels=dict(achieved=(rd_all + wr_all) * args.replicate / (ktimes[0] * 1e-3) / 1e9,
                                         frac=(rd_all + wr_all) * args.replicate / (ktimes[0] * 1e-3) / 1e9 / peak,
                                         frac_timed_region=(rd_all + wr_all) * args.replicate / (dev_s / args.steps) / 1e9 / peak,
                                         ms_per_class={str(k): float(ktimes[k]) for k in range(1, 6)}))
        value = world * args.steps * calls_per_step / dev_s
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(3, args.warmup),
                    ms_per_step=1e3 * dev_s / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                    data="synthetic",
                    config=dict(workload=WORKLOAD, nsmpl=params.nsmpl, sites_per_step_per_gpu=db.nsites, unique_sites=hb.nsites,
                                replicate=args.replicate, allele_mix="2:70%,3:20%,4:7%,5:3%", flags="call -m -a GQ",
                                l2_policy="inputs larger than L2 (%.2f GB of PL per step)" % (db.pl_bytes() / 1e9),
                                bytes_per_call=(rd_all + wr_all) / (hb.nsites * params.nsmpl), generator_version=synth.GENERATOR_VERSION),
                    gpu_launches=launches, clocks=sampler.summary(), roofline=roof, cpu_baseline=cpu, e2e=e2e, parity=parity,
                    sustained=sustained, secondary=secondary, job=job,
                    dumped_outputs=None if dumped_bytes is None else dict(dir=args.dump_outputs, bytes=dumped_bytes))
        print(json.dumps(line, default=lambda o: o.item() if hasattr(o, 'item') else str(o)), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
