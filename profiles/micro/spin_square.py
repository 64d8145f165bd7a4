"""S^2 over the sample space (C_extension.spin_square_matmul, energy.local_spin_square) next to one one-pass E_loc call, on the
benchmarked 10^6-sample Fe2S2 set and its Zipf-0.8 variant, each its own table (samples = keys, as the bench runs them).

    python profiles/micro/spin_square.py [out.json]      # profiles/r05/spin_square.json

Reports the GPU and its power limit; per table the spin exchanges per sample (the lookups the kernel does: |A| |B| plus the
sample itself) and how many of them are in the table; spin_square_matmul for k = 1 and 8, local_spin_square and
eloc_sample_space on the same inputs (CUDA events, median (min, max) of 20 calls after 3 warm-up calls)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200 import synthetic as S  # noqa: E402
from pynqs_b200.energy import local_spin_square  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402
from sample_space_diag import gpu_name_and_power, timed  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE


def open_shells(keys):
    """(|A|, |B|) of every key (uint8 [n, 8]): the numbers of alpha-only and beta-only orbitals"""
    w = keys.view(torch.int64).view(-1)
    a, b = w & 0x5555555555555555, (w >> 1) & 0x5555555555555555
    bits = torch.arange(0, 64, 2, device=keys.device)
    return (((a & ~b).unsqueeze(1) >> bits) & 1).sum(1), (((b & ~a).unsqueeze(1) >> bits) & 1).sum(1)


def main():
    h1e_np, h2e_np, _ = bench.load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    out = {"gpu": gpu_name_and_power(), "config": "Fe2S2 40 sorb 15a15b, 10^6 samples = the table (bench.make_table), float64 psi",
           "timing": "CUDA events, median (min, max) of 20 calls after 3 warm-up calls; table, group index and X stay resident "
                     "between calls (no cache flush); local_spin_square includes its table lookup of psi(x), whose hash "
                     "index is built in the warm-up"}
    for table in ("uniform", "zipf0.8"):
        keys = bench.make_table(table, 1_000_000)
        lut = WavefunctionLUT(torch.from_numpy(keys).to(dev), torch.from_numpy(S.random_psi(keys.shape[0], seed=1235)).to(dev), SORB, dev,
                              rank=0, world_size=1)
        x, N = lut.bra_key, lut.bra_key.size(0)
        gidx = lut.group_index
        nA, nB = open_shells(x)
        pairs = nA * nB
        # exchanges found in the table: S^2 applied to ones minus the diagonal |B| (Sz = 0; every sample is in the table)
        found = ops.spin_square_matmul(x, SORB, x, torch.ones(N, dtype=torch.float64, device=dev), gidx) - nB
        res = {"n": N, "spin_exchanges_per_sample": {"mean": float(pairs.double().mean()), "max": int(pairs.max())},
               "lookups_per_sample_mean": 1.0 + float(pairs.double().mean()),
               "spin_exchanges_in_table": {"total": int(found.sum()), "samples_with_any": int((found > 0).sum())}}
        g = torch.Generator(device=dev).manual_seed(5)
        for k in (1, 8):
            X = torch.randn(N, k, dtype=torch.float64, device=dev, generator=g)
            res[f"spin_square_matmul_k{k}_ms"] = timed(lambda: ops.spin_square_matmul(x, SORB, x, X, gidx))
            del X
        res["local_spin_square_ms"] = timed(lambda: local_spin_square(x, lut, SORB))
        res["eloc_sample_space_ms"] = timed(lambda: ops.eloc_sample_space(x, h1e, h2e, SORB, NELE, NOA, NOB, x, lut.wf_value, gidx))
        res["spin_square_k1_over_eloc"] = res["spin_square_matmul_k1_ms"][0] / res["eloc_sample_space_ms"][0]
        out[table] = res
        del lut, x, found
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
