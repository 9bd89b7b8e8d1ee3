"""Scoring rate at peak depths n_top > 10 (K2d, the deep score table and the deep Ascore kernels) next to n_top = 10.

    python tools/deep_ntop_rates.py [--psms 1000000] [--steps 5] [--n-tops 10,12,20,40]

For config 2 (lowres_phospho) and config 3 (hires_phospho_nl): one batch of synthetic PSMs, resident in HBM, scored at
every n_top of the list on one GPU (the batch comes from bench.py's generator).  Each (workload, n_top) gets two warm-up calls and `--steps` timed calls; the rate is
PSMs over the library's CUDA-event time of the whole call (ms_total), and the stage split is the library's counters
averaged over the timed calls.  Prints one JSON line with the GPU's name and power limit, read in the same run.
Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = ("lowres_phospho", "hires_phospho_nl")
STAGES = ("ms_bin", "ms_plan", "ms_count", "ms_deep", "ms_select", "ms_ascore", "ms_total")


def gpu_info(index):
    """name and power limit of the GPU, from nvidia-smi (None when it cannot be read)"""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return dict(name=name, power_limit_w=float(power), sm_max_mhz=float(clock))
    except Exception as e:                                    # noqa: BLE001 -- reported, not hidden
        return dict(name=None, power_limit_w=None, error="nvidia-smi: %s" % e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--psms", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--n-tops", default="10,12,20,40")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    import bench                                              # its seeded, multi-process batch generator
    from pyascore_b200 import Scorer, synth
    if not torch.cuda.is_available():
        raise SystemExit("deep_ntop_rates.py needs a CUDA device")
    n_tops = [int(x) for x in args.n_tops.split(",")]
    dev = "cuda:%d" % args.device
    out = dict(tool="deep_ntop_rates", gpu=gpu_info(args.device), torch_device_name=torch.cuda.get_device_name(args.device),
               psms=args.psms, steps=args.steps, timing="CUDA events of the library (ms_total per call), batch resident in HBM",
               results=[])
    for wl in WORKLOADS:
        t0 = time.time()
        batch = bench.generate(wl, args.psms, 20261021, os.cpu_count() or 1)
        inputs = {k: torch.from_numpy(v.view(np.int32) if v.dtype == np.uint32 else v).to(dev) for k, v in batch.items()}
        gen_s = time.time() - t0
        w = synth.WORKLOADS[wl]
        for nt in n_tops:
            s = Scorer(**dict(w["scorer"], n_top=nt), device=args.device)
            for g, m in w["neutral_losses"]:
                s.add_neutral_loss(g, m)
            for _ in range(2):
                res = s.score_batch(inputs)
            torch.cuda.synchronize()
            acc = {k: 0.0 for k in STAGES}
            ctr = None
            for _ in range(args.steps):
                res = s.score_batch(inputs, out=res)
                ctr = s.counters()
                for k in STAGES:
                    acc[k] += ctr[k]
            ms = {k: acc[k] / args.steps for k in STAGES}
            n = int(batch["n_mod"].size)
            out["results"].append(dict(
                workload=wl, n_top=nt, psms=n, psm_per_s=n / (ms["ms_total"] * 1e-3), stage_ms=ms,
                n_chunks=ctr["n_chunks"], kernel_launches=ctr["kernel_launches"], launches_deep=ctr["launches_deep"],
                n_isoforms=ctr["n_isoforms"], psms_not_scored=int((res["psm_status"] != 0).sum().item())))
            s.close()
        out.setdefault("generate_s", {})[wl] = gen_s
        del inputs
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
