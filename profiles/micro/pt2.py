"""Epstein-Nesbet PT2 correction (energy.sample_space_pt2) on the benchmarked 10^6-sample Fe2S2 set, its Zipf-0.8 variant
(root 0 of sample_space_ground_state each) and the 18 496-determinant Fe2S2 CI space (3 roots).

    python profiles/micro/pt2.py [out.json]      # profiles/r09/pt2.json

Reports the GPU and its power limit; per table the (row, external) pairs, the externals, the passes of the default 16 GiB
budget, E_var, E_PT2 and E_var + E_PT2 per root, and the time of each phase (count, emit, sort, reduce; CUDA events around
each call, summed over the passes) and of the whole call (host clock around it, ending in a device synchronise).  The
timed call follows one warm-up call of sample_space_pt2 on the same table and repeats its pass loop on the ABI with events
between the calls; its result is checked to have the warm-up's bits."""
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200 import _lib  # noqa: E402
from pynqs_b200 import synthetic as S  # noqa: E402
from pynqs_b200.energy import sample_space_ground_state, sample_space_pt2  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402
from sample_space_diag import gpu_name_and_power  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE
MAX_BYTES = 16 << 30
vp, i64 = _lib.vp, _lib.i64


def timed_pass_loop(lut, C, E, h1e, h2e, lg):
    """pt2_sums' pass loop for a known log2(passes), with CUDA events around each phase; (acc, ms per phase, total ms)"""
    lib, keys = _lib.load(), lut.bra_key
    N, k = keys.size(0), C.size(1)
    gw = lut.group_index.workspace
    prep = ops._cached_prep(h2e, SORB)

    def scratch_bytes(pairs):
        nb = _lib.ctypes.c_int64()
        _lib.check(lib.pynqs_pt2_scratch_bytes(i64(N), i64(pairs), SORB, _lib.ctypes.byref(nb)))
        return nb.value

    stream = vp(torch.cuda.current_stream(dev).cuda_stream)
    events = {p: [] for p in ("count", "emit", "sort", "reduce")}

    def phase(name, call):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(call())
        b.record()
        events[name].append((a, b))

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    cs = torch.empty(scratch_bytes(0), dtype=torch.uint8, device=dev)
    acc = torch.zeros(k, dtype=torch.float64, device=dev)
    ext = torch.zeros(1, dtype=torch.int64, device=dev)
    key = (vp(keys.data_ptr()), i64(N))
    for part in range(1 << lg):
        sel = (vp(gw.data_ptr()), part, lg)
        phase("count", lambda: lib.pynqs_pt2_count(*key, SORB, NOA, NOB, *sel, vp(cs.data_ptr()), i64(cs.numel()), vp(offsets.data_ptr()), stream))
        pairs = int(offsets[N].item())
        if pairs == 0:
            continue
        sc = torch.empty(scratch_bytes(pairs), dtype=torch.uint8, device=dev)
        s = (vp(sc.data_ptr()), i64(sc.numel()))
        phase("emit", lambda: lib.pynqs_pt2_emit(*key, vp(h1e.data_ptr()), vp(prep.workspace.data_ptr()), SORB, NOA, NOB, *sel,
                                                 vp(offsets.data_ptr()), i64(pairs), *s, stream))
        phase("sort", lambda: lib.pynqs_pt2_sort(i64(N), i64(pairs), SORB, *s, stream))
        phase("reduce", lambda: lib.pynqs_pt2_reduce(i64(N), i64(pairs), vp(h1e.data_ptr()), vp(h2e.data_ptr()), SORB, NELE, vp(C.data_ptr()),
                                                     i64(k), k, vp(E.data_ptr()), *s, vp(acc.data_ptr()), vp(ext.data_ptr()), stream))
        del sc
    torch.cuda.synchronize()
    total = (time.perf_counter() - t0) * 1e3
    ms = {p: sum(a.elapsed_time(b) for a, b in ev) for p, ev in events.items()}
    return acc, ms, total


def main():
    h1e_np, h2e_np, _ = bench.load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    out = {"gpu": gpu_name_and_power(), "config": f"Fe2S2 40 sorb 15a15b, max_bytes = {MAX_BYTES}",
           "timing": "one warm-up call of sample_space_pt2, then its pass loop on the ABI: CUDA events around each phase call "
                     "(summed over the passes), host clock around the whole loop (ends in a device synchronise)"}
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import fe2s2

    cases = {"uniform": (lambda: bench.make_table("uniform", 1_000_000), 1), "zipf0.8": (lambda: bench.make_table("zipf0.8", 1_000_000), 1),
             "fe2s2_ci": (lambda: fe2s2()["ci"], 3)}
    for name, (make, nroots) in cases.items():
        keys = make()
        lut = WavefunctionLUT(torch.from_numpy(keys).to(dev), torch.from_numpy(S.random_psi(keys.shape[0], seed=1235)).to(dev), SORB, dev,
                              rank=0, world_size=1)
        e, C, dinfo = sample_space_ground_state(lut, h1e, h2e, SORB, NELE, NOA, NOB, nroots)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e_pt2, info = sample_space_pt2(lut, C, e, h1e, h2e, SORB, NELE, NOA, NOB, max_bytes=MAX_BYTES)
        torch.cuda.synchronize()
        warm = (time.perf_counter() - t0) * 1e3
        lg = info["passes"].bit_length() - 1
        acc, ms, total = timed_pass_loop(lut, C.contiguous(), e.contiguous(), h1e, h2e, lg)
        assert (acc / (C * C).sum(0)).cpu().numpy().tobytes() == e_pt2.cpu().numpy().tobytes()
        res = {"n": keys.shape[0], "roots": nroots, "davidson_converged": dinfo["converged"], **info,
               "e_var": e.tolist(), "e_pt2": e_pt2.tolist(), "e_var_plus_pt2": (e + e_pt2).tolist(),
               "ms": {**{p: round(v, 2) for p, v in ms.items()}, "total": round(total, 2), "warm_up_call": round(warm, 2)}}
        out[name] = res
        print(name, json.dumps(res), flush=True)
        del lut, C
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
