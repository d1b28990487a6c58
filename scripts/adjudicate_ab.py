"""Cost of in-call near-tie adjudication (mcb_set_option "adjudicate") on the bench step (C3: 16,384 unique sites x 4
replicas in HBM, 2,504 samples, device-resident), adjudicate 0 against 1, alternating in one process over several rounds.

  * default tie_eps (1e-6): nothing is flagged, so the difference is the scan of site_flags and the empty launches.
  * tie_eps raised to the 0.1 % and 1 % quantiles of diag[3] (the gap between the best and the runner-up allele set) of a
    first run, so that about 0.1 % / 1 % of the sites are flagged and evaluated again with the literal phase 1.  The
    difference of the two arms over the number of flagged sites is the device cost per adjudicated site.

Per round and arm: --steps steps timed with device events.  Prints one JSON line per round and arm and a summary line."""
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


def caller(tie_eps, adjudicate):
    p = abi.CallParams(params.nsmpl, params.max_nals, theta=params.theta, init_ploidy=params.init_ploidy, flag=params.flag,
                       output_tags=params.output_tags, tie_eps=tie_eps)
    return mcall.MCaller(p, ploidy_tab=tab, options={"adjudicate": adjudicate})


# first run: the gaps between the two best allele sets
with caller(0.0, 0) as mc:
    mc.call_device(b, r, stream)
    torch.cuda.synchronize()
gap = dr.t["diag"][:, 3].double().cpu().numpy()
gap = np.sort(gap[np.isfinite(gap)])
eps = {"default": 0.0, "0.1%": float(gap[int(0.001 * db.nsites)]), "1%": float(gap[int(0.01 * db.nsites)])}
callers = {(k, a): caller(e, a) for k, e in eps.items() for a in (0, 1)}
print(json.dumps(dict(gpu=torch.cuda.get_device_name(0), sites=db.nsites, nsmpl=params.nsmpl, tie_eps=eps)), flush=True)

flagged, times = {}, {k: [] for k in callers}
for rnd in range(args.rounds):
    for k, mc in callers.items():
        for _ in range(3):
            mc.call_device(b, r, stream)
        torch.cuda.synchronize()
        if rnd == 0:
            f = dr.t["site_flags"].cpu().numpy().view(np.uint32)
            flagged[k] = dict(near_tie=int(((f & abi.SITE_NEAR_TIE) != 0).sum()), adjudicated=int(((f & abi.SITE_ADJUDICATED) != 0).sum()))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            mc.call_device(b, r, stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        times[k].append(ms)
        print(json.dumps(dict(round=rnd, tie_eps=k, adjudicate=k[1], step_ms=round(ms, 4))), flush=True)

summary = {}
for k in eps:
    off, on = np.array(times[(k, 0)]), np.array(times[(k, 1)])
    n = flagged[(k, 1)]["adjudicated"]
    summary[k] = dict(tie_eps=eps[k], flagged=flagged[(k, 0)]["near_tie"], adjudicated=n,
                      off_ms_mean=float(off.mean()), off_ms_min=float(off.min()), off_ms_max=float(off.max()),
                      on_ms_mean=float(on.mean()), on_ms_min=float(on.min()), on_ms_max=float(on.max()),
                      added_ms=float(on.mean() - off.mean()),
                      us_per_adjudicated_site=float((on.mean() - off.mean()) * 1e3 / n) if n else None)
print(json.dumps(dict(summary=summary)), flush=True)
for mc in callers.values():
    mc.close()
