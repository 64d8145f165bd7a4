"""Device time of every kernel of pynqs_eloc_sample_space, from torch.profiler, on one rank's share of the 10^6-sample Fe2S2
set (the first N / W samples of the beta-grouped copy against the full table, as in eloc_slice.py).

    python profiles/micro/eloc_kernels_profile.py [W ...]       # default 1 8
Per W: 3 warm-up calls, then 10 profiled ones, each after an L2 flush and a table rebuild (the rebuild's kernels are not
listed).  Prints the mean device time per call of every E_loc kernel."""
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE
CALLS = 10


def main():
    worlds = [int(a) for a in sys.argv[1:]] or [1, 8]
    keys = bench.make_table("uniform", 1_000_000)
    psi = bench.make_psi(keys.shape[0], False)
    h1e_np, h2e_np, _ = bench.load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    d_keys, d_psi = torch.from_numpy(keys).to(dev), torch.from_numpy(psi).to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    n = keys.shape[0]
    print(torch.cuda.get_device_name(0), flush=True)
    for w in worlds:
        def call(lut):
            gi = lut.group_index
            return ops.eloc_sample_space(gi.keys(0)[: n // w], h1e, h2e, SORB, NELE, NOA, NOB, lut.bra_key, lut.wf_value, gi)

        lut = WavefunctionLUT(d_keys, d_psi, SORB, dev, rank=0, world_size=1)
        for _ in range(3):
            call(lut)
        torch.cuda.synchronize()
        luts = []
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(CALLS):
                flush.fill_(1)
                luts.append(WavefunctionLUT(d_keys, d_psi, SORB, dev, rank=0, world_size=1))
                luts[-1].group_index
                call(luts[-1])
            torch.cuda.synchronize()
        totals = {}
        for e in prof.events():
            if e.device_type == torch.autograd.DeviceType.CUDA and ("eloc" in e.name or "sample_" in e.name or "diag" in e.name):
                name = e.name.split("(")[0].replace("void ", "")
                totals[name] = totals.get(name, 0.0) + e.device_time
        print(f"W = {w}: {n // w} samples, mean device time per call over {CALLS} calls", flush=True)
        for name, t in sorted(totals.items(), key=lambda kv: -kv[1]):
            print(f"  {t / CALLS / 1e3:8.3f} ms  {name}", flush=True)


if __name__ == "__main__":
    main()
