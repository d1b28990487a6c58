"""A/B of the 3-allele class kernels on the bench step (C3: 16,384 unique sites x 4 replicas in HBM, 2,504 samples):
option warp3=0 (CTA-per-site kernel, mcall_multi.cu) against the default (warp-per-site kernel, mcall_triallelic.cu),
alternating in one process.  Per round and arm: --steps full steps timed with device events (classes on their own
streams, as bench.py times them), then 5 steps with time_kernels=1 (classes serialised, one event pair per class; median).
At the end the outputs of the last step of each arm are compared: every integer array must be identical, QUAL and the
per-site diagnostics within 1e-6 relative.  Prints one JSON line per round and arm and a summary line."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from bcftools_b200 import abi, synth, mcall, device

ap = argparse.ArgumentParser()
ap.add_argument("--sites", type=int, default=16384)
ap.add_argument("--replicate", type=int, default=4)
ap.add_argument("--rounds", type=int, default=4)
ap.add_argument("--steps", type=int, default=20)
args = ap.parse_args()

params, hb, tab = synth.make_batch("C3", args.sites, with_groups=0)
db = device.DeviceBatch(hb, replicate=args.replicate)
dr = device.DeviceResult(db)
b, r = db.c_struct(), dr.c_struct()
stream = torch.cuda.current_stream().cuda_stream
arms = {"warp3=0": {"warp3": 0}, "warp3=auto": {}}
callers = {k: mcall.MCaller(params, ploidy_tab=tab, options=o) for k, o in arms.items()}
print(json.dumps(dict(gpu=torch.cuda.get_device_name(0), sites=db.nsites, nsmpl=params.nsmpl,
                      class3_sites=int((hb.nals == 3).sum()) * args.replicate)), flush=True)
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
        print(json.dumps(dict(round=rnd, arm=k, step_ms=round(step_ms, 4), class_ms={str(c): round(float(kt[c]), 4) for c in range(1, 6)})), flush=True)

# outputs of one step of each arm, compared on the device
snap = {}
for k, mc in callers.items():
    for t in dr.t.values():             # nothing left over from the other arm can pass for this arm's output
        if t is not None:
            t.fill_(-7)
    mc.call_device(b, r, stream)
    torch.cuda.synchronize()
    snap[k] = {n: t.clone() for n, t in dr.t.items() if t is not None}
A, B = snap["warp3=0"], snap["warp3=auto"]
cmp = {}
for n in A:
    x, y = A[n], B[n]
    if x.dtype in (torch.float32, torch.float64):
        xf, yf = x.double(), y.double()
        both_nan = torch.isnan(xf) & torch.isnan(yf)
        rel = ((xf - yf).abs() / yf.abs().clamp_min(1e-300)).masked_fill(both_nan | (xf == yf), 0)
        cmp[n] = dict(max_rel=float(rel.max()), n_diff=int((rel > 1e-6).sum()))
    else:
        cmp[n] = dict(n_diff=int((x != y).sum()))
flags = {k: int(((s["site_flags"] & abi.SITE_NEAR_TIE) != 0).sum()) for k, s in snap.items()} if "site_flags" in A else {}
summary = {}
for k in arms:
    st = np.array(res[k]["step_ms"]); c3 = np.array([c[3] for c in res[k]["class_ms"]])
    summary[k] = dict(step_ms_mean=float(st.mean()), step_ms_min=float(st.min()), step_ms_max=float(st.max()),
                      class3_ms_mean=float(c3.mean()), class3_ms_min=float(c3.min()), class3_ms_max=float(c3.max()))
o, n = summary["warp3=0"], summary["warp3=auto"]
print(json.dumps(dict(summary=summary, step_gain=o["step_ms_mean"] / n["step_ms_mean"] - 1,
                      class3_gain=o["class3_ms_mean"] / n["class3_ms_mean"] - 1, outputs=cmp, near_tie_sites=flags)), flush=True)
for mc in callers.values():
    mc.close()
ok = all(v["n_diff"] == 0 for v in cmp.values())
sys.exit(0 if ok else 1)
