"""A/B of the 4-allele class kernels on the bench step (C3: 16,384 unique sites x 4 replicas in HBM, 2,504 samples):
option warp4=0 (CTA-per-site kernel, mcall_multi.cu) against the default (warp-per-site kernel, mcall_multi_warp.cu),
alternating in one process.  Per round and arm: --steps full steps timed with device events (classes on their own streams, as
bench.py times them), then 5 steps with time_kernels=1 (classes serialised, one event pair per class; median).  At the end
the outputs of the last step of each arm are compared with the first arm's: every integer array must be identical, QUAL and
the per-site diagnostics within 1e-6 relative.  Prints the card, its power limit and SM clock, one JSON line per round and
arm and a summary line.

--sweep adds arms that cap the warps per CTA of the warp kernel (warp4=n): the head of the packed copy that stays in shared
memory grows as the warps per CTA shrink, so this also sweeps the head/tail split (at 2,504 samples on a B200, 228 KB of
shared memory per SM: 8 warps 1,280 samples in shared memory, 7: 1,472, 6: 1,728, 5: 2,112, 4: all)."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from bcftools_b200 import abi, synth, mcall, device

ap = argparse.ArgumentParser()
ap.add_argument("--sites", type=int, default=16384)
ap.add_argument("--replicate", type=int, default=4)
ap.add_argument("--rounds", type=int, default=4)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--sweep", action="store_true")
args = ap.parse_args()

params, hb, tab = synth.make_batch("C3", args.sites, with_groups=0)
db = device.DeviceBatch(hb, replicate=args.replicate)
dr = device.DeviceResult(db)
b, r = db.c_struct(), dr.c_struct()
stream = torch.cuda.current_stream().cuda_stream
arms = {"cta": {"warp4": 0}, "auto": {}}
if args.sweep:
    for w in (8, 7, 6, 5, 4):
        arms[f"warp4={w}"] = {"warp4": w}
callers = {k: mcall.MCaller(params, ploidy_tab=tab, options=o) for k, o in arms.items()}
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
except OSError:
    smi = "nvidia-smi not available"
print(json.dumps(dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=smi, sites=db.nsites, nsmpl=params.nsmpl,
                      class_sites={c: int((hb.nals == c).sum()) * args.replicate for c in (4, 5)})), flush=True)
res = {k: dict(step_ms=[], class_ms=[]) for k in arms}
for rnd in range(args.rounds):
    for k, mc in callers.items():
        for _ in range(3):
            mc.call_device(b, r, stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            mc.call_device(b, r, stream)
        e1.record()
        torch.cuda.synchronize()
        step_ms = e0.elapsed_time(e1) / args.steps
        mc.set_option("time_kernels", 1)
        kt = []
        for _ in range(5):
            mc.call_device(b, r, stream)
            kt.append(mc.kernel_times_ms())
        mc.set_option("time_kernels", 0)
        kt = np.median(np.array(kt), axis=0)
        res[k]["step_ms"].append(step_ms)
        res[k]["class_ms"].append([float(x) for x in kt])
        print(json.dumps(dict(round=rnd, arm=k, step_ms=round(step_ms, 4), class_ms={str(c): round(float(kt[c]), 4) for c in range(1, 6)},
                              class45_ms=round(float(kt[4] + kt[5]), 4))), flush=True)

# outputs of one step of each arm, compared on the device with the first arm's
snap = {}
for k, mc in callers.items():
    for t in dr.t.values():             # nothing left over from another arm can pass for this arm's output
        if t is not None:
            t.fill_(-7)
    mc.call_device(b, r, stream)
    torch.cuda.synchronize()
    snap[k] = {n: t.clone() for n, t in dr.t.items() if t is not None}
ref = snap["cta"]
cmp = {}
for k in arms:
    if k == "cta":
        continue
    c = {}
    for n in ref:
        x, y = snap[k][n], ref[n]
        if x.dtype in (torch.float32, torch.float64):
            xf, yf = x.double(), y.double()
            both_nan = torch.isnan(xf) & torch.isnan(yf)
            rel = ((xf - yf).abs() / yf.abs().clamp_min(1e-300)).masked_fill(both_nan | (xf == yf), 0)
            c[n] = dict(max_rel=float(rel.max()), n_diff=int((rel > 1e-6).sum()))
        else:
            c[n] = dict(n_diff=int((x != y).sum()))
    cmp[k] = c
flags = {k: int(((s["site_flags"] & abi.SITE_NEAR_TIE) != 0).sum()) for k, s in snap.items()} if "site_flags" in ref else {}
summary = {}
for k in arms:
    st = np.array(res[k]["step_ms"]); c45 = np.array([c[4] + c[5] for c in res[k]["class_ms"]])
    c4 = np.array([c[4] for c in res[k]["class_ms"]]); c5 = np.array([c[5] for c in res[k]["class_ms"]])
    summary[k] = dict(step_ms_mean=float(st.mean()), step_ms_min=float(st.min()), step_ms_max=float(st.max()),
                      class4_ms_mean=float(c4.mean()), class5_ms_mean=float(c5.mean()),
                      class45_ms_mean=float(c45.mean()), class45_ms_min=float(c45.min()), class45_ms_max=float(c45.max()))
o, n = summary["cta"], summary["auto"]
print(json.dumps(dict(summary=summary, step_gain=o["step_ms_mean"] / n["step_ms_mean"] - 1,
                      class45_gain=o["class45_ms_mean"] / n["class45_ms_mean"] - 1, outputs=cmp, near_tie_sites=flags)), flush=True)
for mc in callers.values():
    mc.close()
ok = all(v["n_diff"] == 0 for c in cmp.values() for v in c.values())
sys.exit(0 if ok else 1)
