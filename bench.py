#!/usr/bin/env python
"""bench.py -- E_loc samples/sec on the Fe2S2 workload (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                          # reference CPU build (oracle/_ref)
    python bench.py --impl reference_cuda [...]                     # reference CUDA build (oracle/_ref, GPU-vs-GPU)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload: Fe2S2 CAS(30e,20o): 40 spin orbitals, 15 alpha + 15 beta electrons (M = 7876 connected determinants
per sample), the reference's own Fe2S2 integrals (example/Fe2S2/fe2s2-OO.pth, shipped here as the data file
tests/golden/fe2s2_integrals.npz), 10^6 unique seeded random ONVs that are both the evaluated samples and the
lookup table, psi = randn (seed 1235), FP64.

One step = one pass of the hot path over the whole sample set:
  [N > 1: NCCL all-gather of every rank's unique ONVs + psi] -> sorted table + string-grouped copies ->
  one-pass sample-space E_loc on this rank's slice -> fused energy statistics (one collective).
Strong scaling: the 10^6 samples are sharded over the ranks.  `value` = samples / step time with everything
resident in HBM; `e2e` repeats the step from pinned HOST buffers (H2D of ONVs + psi, D2H of E_loc + statistics
inside the timed region).  L2 is flushed between timed steps.

Parity is part of the line: the E_loc values the `cpu_baseline` leg computes with the unmodified reference
extension (>= 10^5 samples of the same 10^6-key run) are compared with the GPU values of the same samples
(`parity`); the run exits non-zero when they differ by more than 1e-12 relative / 1e-10 Ha on the mean.  The same
is done for a complex128 psi and for a skewed (Zipf) table (`variants`).  Prints ONE JSON line on rank 0.
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

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SORB, NOA, NOB = 40, 15, 15
NELE = NOA + NOB
M_FE2S2 = 7876
METRIC = "E_loc samples/sec (Fe2S2 40 sorb)"
UNIT = "samples/s"
TOL_REL, TOL_MEAN_HA = 1e-12, 1e-10


def algorithmic_bytes_per_sample(M: int, L: int, psi_bytes: int = 8) -> int:
    """SURVEY.md section 8(d): API path (fused + lut) B = 8L + M (16L + 17) + P_psi."""
    return 8 * L + M * (16 * L + 17) + psi_bytes


def hbm_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---- inputs ------------------------------------------------------------------------------------------------------
def load_integrals():
    """The config-2 Hamiltonian: the reference's Fe2S2 integrals (data file made by tests/golden/make_golden.py)."""
    from pynqs_b200 import synthetic as S

    path = os.path.join(ROOT, "tests", "golden", "fe2s2_integrals.npz")
    if os.path.exists(path):
        g = np.load(path)
        assert int(g["sorb"]) == SORB and int(g["noA"]) == NOA and int(g["noB"]) == NOB
        return np.ascontiguousarray(g["h1e"]), np.ascontiguousarray(g["h2e"]), "fe2s2-OO.pth of the reference (tests/golden/fe2s2_integrals.npz)"
    h1e, h2e = S.random_packed_integrals(SORB, seed=7, symmetric=True)
    return h1e, h2e, "random 8-fold symmetric, seed 7 (Fe2S2 data file missing)"


def _strings(n, rng, shift=0):
    occ = np.argsort(rng.random((n, SORB // 2)), axis=1)[:, :NOA]
    out = np.zeros(n, dtype=np.uint64)
    for c in range(NOA):
        out |= np.uint64(1) << (2 * occ[:, c] + shift).astype(np.uint64)
    return out


def make_table(kind: str, n: int) -> np.ndarray:
    """uint8 [n, 8] unique ONVs.  uniform: every determinant equally likely.  zipf0.8: the beta strings are drawn
    with Zipf(0.8) weights over all C(20,15) strings, so the table is dominated by a few heavy strings (groups of
    thousands of keys next to groups of a handful) like a VMC sample set."""
    from pynqs_b200 import synthetic as S

    if kind == "uniform":
        return S.random_onvs(n, SORB, NOA, NOB, seed=1234)
    if kind.startswith("zipf"):
        beta_exp = float(kind[4:])
        rng = np.random.default_rng(3)
        # all 15504 strings (with overwhelming probability) in ascending order: the heavy strings are numerically
        # adjacent, i.e. mostly single excitations of each other, so heavy groups are connected to heavy groups
        # (the construction of profiles/skew_check.py, round 1: 35 M samples/s)
        beta = np.unique(_strings(400_000, rng)) << np.uint64(1)
        w = 1.0 / np.arange(1, beta.size + 1) ** beta_exp
        keys = np.unique(_strings(3 * n, rng) | beta[rng.choice(beta.size, size=3 * n, p=w / w.sum())])
        keys = keys[rng.permutation(keys.size)[:n]]
        return np.ascontiguousarray(keys.view(np.uint8).reshape(-1, 8))
    raise ValueError(kind)


def make_psi(n: int, cplx: bool) -> np.ndarray:
    from pynqs_b200 import synthetic as S

    return S.random_psi(n, seed=1235, complex_=cplx)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


# ---- the reference arms ---------------------------------------------------------------------------------------------
def reference_ops(cuda: bool = False):
    """(module, kind): the unmodified reference extension if oracle/_ref was built, else the oracle port."""
    from oracle import build_ref

    if cuda:
        return (build_ref.load_ref(1, cuda=True), "reference_cuda") if build_ref.cuda_available(1) else (None, "unavailable")
    if build_ref.available(1):
        return build_ref.load_ref(1), "reference"
    return None, "port"


def reference_eloc_step(ref, x, h1e, h2e, key, val):
    """The reference's op sequence for the sample-space local energy (vmc/energy/eloc.py:369-397) on torch tensors
    of either device, through the reference extension `ref`."""
    import torch

    comb_x, comb_hij = ref.get_comb_hij_fused(x, h1e, h2e, SORB, NELE, NOA, NOB)
    x1 = comb_x.reshape(-1, comb_x.size(2))
    psi_x1 = torch.zeros(x.size(0), comb_x.size(1), dtype=val.dtype, device=x.device)
    idx_array, mask = ref.wavefunction_lut(key, x1, SORB)
    baseline = torch.arange(x1.size(0), dtype=torch.int64, device=x.device)
    psi_x1.view(-1)[baseline[mask]] = val[idx_array.masked_select(mask)]
    return ((psi_x1.T / psi_x1[..., 0]).T * comb_hij).sum(-1)


def cpu_eloc_step(ref, kind, x_np, h1e_np, h2e_np, skeys_np, spsi_np):
    import torch

    if kind == "reference":
        t = torch.from_numpy
        return reference_eloc_step(ref, t(x_np), t(h1e_np), t(h2e_np), t(skeys_np), t(spsi_np)).numpy()
    from oracle import oracle as O

    return O.eloc_sample_space(x_np, h1e_np, h2e_np, skeys_np, spsi_np, SORB, NELE, NOA, NOB)


def cpu_reference_eloc(keys, psi, h1e, h2e, budget_s=12.0, chunk=512, max_samples=None):
    """Bounded sample of the same workload on the host cores: E_loc of the first `done` samples (original order)
    against the full table.  Returns (eloc[done], record)."""
    import torch

    from oracle import oracle as O

    ref, kind = reference_ops()
    cores = os.cpu_count() if kind == "reference" else 1
    torch.set_num_threads(cores)
    order = O.sort_onv(keys)
    skeys, spsi = np.ascontiguousarray(keys[order]), np.ascontiguousarray(psi[order])
    if kind == "port":
        chunk = 32
    cpu_eloc_step(ref, kind, keys[:chunk], h1e, h2e, skeys, spsi)  # warm-up
    out, done, t0 = [], 0, time.perf_counter()
    while True:
        out.append(cpu_eloc_step(ref, kind, keys[done : done + chunk], h1e, h2e, skeys, spsi))
        done += chunk
        el = time.perf_counter() - t0
        if el > budget_s or done + chunk > keys.shape[0] or (max_samples is not None and done >= max_samples):
            break
    rec = {"value": done / el, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"{done} of {keys.shape[0]} samples in {chunk}-sample chunks against the full {keys.shape[0]}-key table "
                     f"(get_comb_hij_fused + wavefunction_lut + torch reduce), {el:.1f} s"}
    return np.concatenate(out), rec


def parity_block(eloc_gpu_orig: np.ndarray, eloc_ref: np.ndarray, psi: np.ndarray, against: str) -> dict:
    """GPU E_loc vs reference E_loc of the same samples: per-element relative error and the |psi|^2-weighted mean."""
    n = eloc_ref.shape[0]
    a, b = eloc_gpu_orig[:n], eloc_ref
    rel = np.abs(a - b) / np.abs(b)
    w = np.abs(psi[:n]) ** 2
    w = w / w.sum()
    mean_a, mean_b = complex(np.sum(w * a)), complex(np.sum(w * b))
    diff = abs(mean_a - mean_b)
    ok = bool(np.all(np.isfinite(a)) and rel.max() <= TOL_REL and diff <= TOL_MEAN_HA)
    return {"n": int(n), "against": against, "max_rel_err": float(rel.max()), "mean_energy_abs_diff_ha": float(diff),
            "mean_energy_ha": mean_b.real, "tol_rel": TOL_REL, "tol_mean_ha": TOL_MEAN_HA, "ok": ok}


def base_config(n_total: int, integrals: str, table: str = "uniform") -> dict:
    return {"workload": "fe2s2_cas30e20o_40sorb_15a15b", "sorb": SORB, "noA": NOA, "noB": NOB, "M": M_FE2S2, "n_samples": int(n_total),
            "lut_keys": int(n_total), "integrals": integrals, "table": table}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    from oracle import oracle as O

    cuda = args.impl == "reference_cuda"
    keys = make_table("uniform", args.samples)
    psi = make_psi(keys.shape[0], False)
    h1e, h2e, integrals = load_integrals()
    ref, kind = reference_ops(cuda)
    if cuda and (ref is None or not torch.cuda.is_available()):
        print(json.dumps({"impl": "reference_cuda", "unavailable": "oracle/_ref/C_extension_cuda_L1.so missing or no CUDA device"}), flush=True)
        return
    cores = os.cpu_count() if kind == "reference" else 1
    torch.set_num_threads(os.cpu_count())
    order = O.sort_onv(keys)
    skeys, spsi = np.ascontiguousarray(keys[order]), np.ascontiguousarray(psi[order])
    if cuda:
        per_step, chunk = 32768, 8192
        dev = torch.device("cuda", 0)
        d = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
        d_keys, d_h1e, d_h2e, d_skeys, d_spsi = d(keys), d(h1e), d(h2e), d(skeys), d(spsi)

        def step(i):
            lo = (i * per_step) % (keys.shape[0] - per_step)
            for b in range(lo, lo + per_step, chunk):
                reference_eloc_step(ref, d_keys[b : b + chunk], d_h1e, d_h2e, d_skeys, d_spsi)
            torch.cuda.synchronize()
    else:
        per_step = args.ref_samples if kind == "reference" else 64
        chunk = 512 if kind == "reference" else 32

        def step(i):
            lo = (i * per_step) % (keys.shape[0] - per_step)
            for b in range(lo, lo + per_step, chunk):
                cpu_eloc_step(ref, kind, keys[b : min(b + chunk, lo + per_step)], h1e, h2e, skeys, spsi)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    el = time.perf_counter() - t0
    value = per_step * args.steps / el
    sample = (f"each step = E_loc of {per_step} samples ({chunk}-sample chunks) against the prebuilt sorted "
              f"{keys.shape[0]}-key table; table sort not timed")
    line = {
        "impl": args.impl, "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(keys.shape[0], integrals),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from pynqs_b200 import _lib
    from pynqs_b200 import C_extension as ops
    from pynqs_b200.distributed import energy_statistics_amplitudes, exchange_unique_samples, sample_space_energy_sharded
    from pynqs_b200.lut import WavefunctionLUT, split_length_idx
    from pynqs_b200.step import SampleSpaceStep

    _lib.load()
    from pynqs_b200 import peer

    if args.no_peer:
        peer.set_enabled(False)
    h1e_np, h2e_np, integrals = load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    M = ops.get_Num_SinglesDoubles(SORB, NOA, NOB) + 1
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def measure(keys_np, psi_np, steps, warmup, want_e2e=True):
        """Times `steps` steps of the hot path over the sample set (keys_np, psi_np).  The timed step is the library's
        SampleSpaceStep (pynqs_b200/step.py): exchange -> table -> E_loc -> statistics captured in ONE CUDA graph after the
        warm-up steps and replayed per step (--no-graph: launched kernel by kernel).  A few extra EAGER steps with CUDA events
        between the phases give `phases_ms_rank0` (not part of `value`)."""
        n_total = keys_np.shape[0]
        cplx = np.iscomplexobj(psi_np)
        # every rank "samples" a contiguous piece of the unique set (disjoint pieces, like use_same_tree)
        cuts = [0] + split_length_idx(n_total, world)
        lo, hi = cuts[rank], cuts[rank + 1]
        host_keys = torch.from_numpy(keys_np[lo:hi]).pin_memory()
        host_psi = torch.from_numpy(psi_np[lo:hi]).pin_memory()
        d_keys, d_psi = host_keys.to(dev), host_psi.to(dev)
        host_eloc = torch.empty(hi - lo, dtype=d_psi.dtype).pin_memory()
        step_obj = SampleSpaceStep(hi - lo, d_keys.size(1), d_psi.dtype, h1e, h2e, SORB, NELE, NOA, NOB, device=dev,
                                   use_graph=not args.no_graph, warmup=max(2, warmup - 1))
        step_obj.load(d_keys, d_psi)

        def step(from_host: bool):
            if from_host:
                step_obj.load(host_keys, host_psi)  # H2D of this step's inputs (pinned memory)
            eloc, psi0, st = step_obj.run()
            if from_host:
                host_eloc.copy_(eloc, non_blocking=True)  # D2H of the step's result
                st = st.result()
            return eloc, psi0, st

        def timed(n_steps: int, from_host: bool):
            total_ms = 0.0
            eloc = psi0 = st = None
            for _ in range(n_steps):
                flush.fill_(1)  # write > L2 (126 MB) between timed steps
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                eloc, psi0, st = step(from_host)
                t.record()
                torch.cuda.synchronize()
                total_ms += s.elapsed_time(t)
            tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()), (eloc, psi0, st)

        for _ in range(max(warmup, 4)):  # eager steps, then the capture, then replays
            step(False)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        total_ms, (eloc, psi0, st) = timed(steps, False)
        launches = _lib.launch_count() - l0
        stats = st.result()
        last = None
        if args.dump_outputs:  # copied now: the steps that follow reuse the step's output buffers
            last = {"eloc": eloc.cpu().numpy(), "psi0": psi0.cpu().numpy(), "stats": stats}
        if step_obj.graph is not None:  # replays do not pass through the library's launch counter: count one eager step
            l0 = _lib.launch_count()
            step_obj._body()
            launches = (_lib.launch_count() - l0) * steps
        out = {"n_total": n_total, "ms_per_step": total_ms / steps, "value": n_total / (total_ms / steps * 1e-3), "launches": int(launches),
               "stats": stats, "last_step": last, "cplx": cplx, "graph": step_obj.graph is not None, "why_eager": step_obj.why_eager}
        if want_e2e:
            for _ in range(2):  # the end-to-end path has first-use costs of its own (pinned copies both ways)
                step(True)
            torch.cuda.synchronize()
            e2e_ms, (_, _, st2) = timed(steps, True)
            out["e2e"] = {"value": n_total / (e2e_ms / steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(n_total * (8 + d_psi.element_size())),
                          "d2h_bytes_per_step": int(n_total * d_psi.element_size() + 56 * world), "ms_per_step": e2e_ms / steps}
            out["mean_e2e"] = st2["mean"]
        # the phases of the step, from eager launches with events in between (kernel by kernel, so launch-latency bound at
        # small per-rank sizes; the timed value above is the captured step)
        names = ["exchange", "table_sort_and_index", "eloc_kernels", "probabilities_and_statistics"]
        acc, nphase = [0.0] * 4, 3
        for it in range(nphase + 1):  # the first pass warms the eager allocations up again (the graph has a pool of its own)
            flush.fill_(1)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
            uniq, wf, _ = exchange_unique_samples(d_keys, d_psi, None, disjoint=True, sizes=step_obj.sizes)
            ev[1].record()
            lut = WavefunctionLUT(uniq, wf, SORB, dev, rank=rank, world_size=world)
            lut.group_index  # built here, inside the table phase
            ev[2].record()
            eloc, psi0 = sample_space_energy_sharded(lut, h1e, h2e, SORB, NELE, NOA, NOB)
            ev[3].record()
            energy_statistics_amplitudes(eloc, psi0, lazy=True)
            ev[4].record()
            torch.cuda.synchronize()
            for i in range(4):
                acc[i] += ev[i].elapsed_time(ev[i + 1]) / nphase if it else 0.0
        out["phases"] = dict(zip(names, acc))
        out["kernel_ms"], out["kernel_samples"] = acc[2], hi - lo
        # E_loc of the whole sample set back in the ORIGINAL sample order (one rank only: parity legs).  The step returns the
        # rows of the sorted table; row j of it is original row sort_perm[j]
        if world == 1:
            eloc_sorted, _, _ = step_obj.run()
            eloc_orig = torch.empty_like(eloc_sorted)
            eloc_orig[step_obj.lut._sort_perm] = eloc_sorted
            out["eloc_orig"] = eloc_orig.cpu().numpy()
        out["d_keys"], out["d_psi"] = d_keys, d_psi
        return out

    keys_np = make_table(args.table, args.samples)
    psi_np = make_psi(keys_np.shape[0], False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    main = measure(keys_np, psi_np, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main["last_step"], rank, world)
    n_total = main["n_total"]

    # variants (the same step, --steps timed steps each): complex128 psi (config 2 is complex, Fe2S2-OO-dcut-20.py:39) and a skewed table
    variants = {}
    vsteps, vwarm = args.steps, 3
    if not args.no_variants and world == 1:
        psi_c = make_psi(n_total, True)
        variants["complex128"] = (measure(keys_np, psi_c, vsteps, vwarm, want_e2e=False), keys_np, psi_c)
        keys_z = make_table("zipf0.8", args.samples)
        variants["zipf0.8"] = (measure(keys_z, psi_np[: keys_z.shape[0]], vsteps, vwarm, want_e2e=False), keys_z, psi_np[: keys_z.shape[0]])

    B = algorithmic_bytes_per_sample(M, 1)
    peak, peak_src = hbm_peak_gbs()
    prof = load_profile_numbers()
    k_ms, k_n = main["kernel_ms"], main["kernel_samples"]
    equiv = B * k_n / (k_ms * 1e-3) / 1e9
    inst = prof.get("eloc_warp_instructions_per_sample")
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = 148 * 4 * sm_mhz * 1e6  # warp-instructions / s: 4 schedulers per SM, one instruction per cycle each
    issue_rate = inst * k_n / (k_ms * 1e-3) if inst else None
    roof = {"bound": "issue",
            "kernel": "one-pass sample-space E_loc: eloc scan kernels (+ eloc_eval_kernel, diag_table_kernel)",
            "launch": "one pynqs_eloc_sample_space call on this rank's samples",
            "achieved": issue_rate, "peak": issue_peak, "unit": "warp-instructions/s", "frac": issue_rate / issue_peak if issue_rate else None,
            "achieved_note": "warp-instructions per sample from the committed ncu capture (profiles/%s) x samples per call / live CUDA-event time of the call; "
                             "peak = 592 warp schedulers x sampled SM clock" % prof.get("tag", "?"),
            "traffic": prof.get("eloc_dram_bytes_per_sample") and prof["eloc_dram_bytes_per_sample"] * k_n,
            "traffic_note": "DRAM bytes per call from ncu (profiles/%s/traffic.json): the table copies stay in L2" % prof.get("tag", "?"),
            "samples_per_launch": k_n, "kernel_ms": k_ms,
            "equivalent_hbm": {"achieved": equiv, "peak": peak, "unit": "GB/s", "frac": equiv / peak, "peak_source": peak_src,
                               "algorithmic_bytes_per_sample": B,
                               "note": "SURVEY.md 8(d) equivalent-bytes figure: API-path bytes (fused + lut, 259.9 KB/sample) / time. NOT a physical HBM "
                                       "fraction -- the one-pass kernels never write comb/Hmat/idx; the kernels that really move those bytes are in "
                                       "'roofline_hbm_kernels'"}}
    if rank != 0:
        leave(world)
        return
    cfg = base_config(n_total, integrals, args.table)
    cfg.update({"method": "sample-space, one-pass kernels", "l2": "flushed between timed steps (512 MiB write)",
                "collectives": peer.route() if world > 1 else "none (one rank)",
                "launch": "one CUDA graph per step (captured after the warm-up steps)" if main["graph"] else "kernel by kernel: " + main["why_eager"],
                "parallelism": f"samples sharded over {world} rank(s)", "step": "exchange + table sort + grouped table + E_loc + statistics"})
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg, "roofline": roof, "e2e": main["e2e"], "gpu_launches": main["launches"],
        "phases_ms_rank0": main["phases"],
        "phases_note": "measured in extra EAGER steps with CUDA events between the phases (kernel by kernel, launch latency included); "
                       "ms_per_step / value are the captured step",
        "clocks": clocks,
        "energy": {"mean": main["stats"]["mean"], "var": main["stats"]["var"], "mean_e2e": main["mean_e2e"]},
    }
    ok = True
    if world == 1 and not args.no_cpu_baseline:
        eloc_ref, rec = cpu_reference_eloc(keys_np, psi_np, h1e_np, h2e_np, budget_s=args.cpu_budget)
        line["cpu_baseline"] = rec
        line["parity"] = parity_block(main["eloc_orig"], eloc_ref, psi_np, f"unmodified reference extension ({rec['kind']}), same inputs")
        ok &= line["parity"]["ok"]
    else:
        line["cpu_baseline"] = None
    vout = {}
    for name, (m, k_np, p_np) in variants.items():
        ent = {"value": m["value"], "unit": UNIT, "ms_per_step": m["ms_per_step"], "steps": vsteps, "phases_ms_rank0": m["phases"],
               "energy_mean": str(m["stats"]["mean"])}
        if world == 1 and not args.no_cpu_baseline:
            eloc_ref, rec = cpu_reference_eloc(k_np, p_np, h1e_np, h2e_np, budget_s=3.0, max_samples=args.variant_parity_samples)
            ent["parity"] = parity_block(m["eloc_orig"], eloc_ref, p_np, f"unmodified reference extension ({rec['kind']}), same inputs")
            ok &= ent["parity"]["ok"]
        vout[name] = ent
    if vout:
        line["variants"] = vout
    if world == 1 and not args.no_api_path:
        line["roofline_hbm_kernels"] = time_api_path(ops, dev, main["d_keys"], main["d_psi"], h1e, h2e, M, peak, prof)
    print(json.dumps(line), flush=True)
    if not ok:
        sys.stderr.write("bench.py: PARITY FAILURE against the reference extension (see 'parity' in the JSON line)\n")
        sys.stderr.flush()
        if world > 1:
            os._exit(3)
        sys.exit(3)
    leave(world)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, last: dict, rank: int, world: int) -> None:
    """Write what the last timed step returned to its caller, as float64 .npy files in out_dir:
      eloc.npy, psi0.npy     this rank's rows of the sorted table ([n] real, or [n, 2] = (re, im) for complex psi);
      energy_statistics.npy  [mean.real, mean.imag, var, sd, se, n].
    Above DUMP_BYTES in all, a fixed seeded sample of rows is written instead, with its row numbers in rows.npy.
    With more than one rank, every rank writes its own files with a _rank<r> suffix."""
    os.makedirs(out_dir, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    arrays = {k: np.ascontiguousarray(last[k]) for k in ("eloc", "psi0")}
    arrays = {k: (a.view(np.float64).reshape(-1, 2) if np.iscomplexobj(a) else a).astype(np.float64) for k, a in arrays.items()}
    n = arrays["eloc"].shape[0]
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(n, 1)
    budget = DUMP_BYTES // world - 4096
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, size=budget // (row_bytes + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    st = last["stats"]
    mean = complex(st["mean"])
    arrays["energy_statistics"] = np.array([mean.real, mean.imag, st["var"], st["sd"], st["se"], st["n"]], dtype=np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}{sfx}.npy"), a)


def leave(world: int) -> None:
    """End of a multi-rank run: synchronise, then exit WITHOUT destroy_process_group() -- the teardown was seen to block for
    minutes after the symmetric-memory rendezvous of the peer-memory collectives (every rank had finished its work), and a
    rank that never exits keeps torchrun, and whoever launched it, waiting."""
    if world <= 1:
        return
    import torch
    import torch.distributed as dist

    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    time.sleep(0.5)  # the peers may still be completing their side of the barrier: do not pull the memory from under them
    os._exit(0)


def load_profile_numbers():
    """ncu-derived numbers of the latest committed profile (profiles/rNN/traffic.json): per-launch DRAM traffic and
    warp-instructions per sample of the one-pass kernels."""
    for tag in ("r02", "r01"):
        try:
            out = json.load(open(os.path.join(ROOT, "profiles", tag, "traffic.json")))
            out["tag"] = tag
            out.setdefault("eloc_warp_instructions_per_sample", 5685 if tag == "r01" else None)
            return out
        except Exception:
            continue
    return {}


def time_api_path(ops, dev, d_keys, d_psi, h1e, h2e, M, peak, prof, chunk=32768, reps=7):
    """The materialising reference-API kernels on one chunk: the real HBM movers of the hot path, with the
    UNMODIFIED reference CUDA extension (oracle/_ref/C_extension_cuda_L1.so) timed on the same tensors beside them.
    Outputs are allocated by torch inside the call (caching allocator, no cudaMalloc after warm-up);
    2.06 GB comb + 2.06 GB Hmat per call exceed L2, so no flush is needed between repetitions."""
    import torch

    from pynqs_b200.lut import WavefunctionLUT

    lut = WavefunctionLUT(d_keys, d_psi, SORB, dev, rank=0, world_size=1)
    x = lut.bra_key[:chunk]
    prep = ops.PreparedIntegrals(h2e, SORB)

    def t(fn, reps=reps):
        for _ in range(3):
            out = fn()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts), out

    f_ms, (comb, hmat) = t(lambda: ops.get_comb_hij_fused(x, h1e, h2e, SORB, NELE, NOA, NOB, prepared=prep))
    flat = comb.view(-1, 8)
    l_ms, (idx, mask) = t(lambda: ops.wavefunction_lut(lut.bra_key, flat, SORB, hash_index=lut.hash_index))
    fb, lb = (16 * M + 8) * chunk, 17 * M * chunk
    ref_cuda = {}
    try:
        ref, kind = reference_ops(cuda=True)
        if ref is not None:
            rf_ms, (rcomb, rhmat) = t(lambda: ref.get_comb_hij_fused(x, h1e, h2e, SORB, NELE, NOA, NOB), reps=3)
            same_f = bool(torch.equal(rcomb, comb) and torch.equal(rhmat.view(torch.int64), hmat.view(torch.int64)))
            del rcomb, rhmat
            rl_ms, (ridx, rmask) = t(lambda: ref.wavefunction_lut(lut.bra_key, flat, SORB), reps=3)
            same_l = bool(torch.equal(ridx, idx) and torch.equal(rmask, mask))
            del ridx, rmask
            ref_cuda = {"fused": {"ms": rf_ms, "speedup": rf_ms / f_ms, "bit_identical_outputs": same_f},
                        "lut": {"ms": rl_ms, "speedup": rl_ms / l_ms, "bit_identical_outputs": same_l}}
            sub = 8192
            re_ms, _ = t(lambda: reference_eloc_step(ref, x[:sub], h1e, h2e, lut.bra_key, lut.wf_value), reps=3)
            ref_cuda["eloc_three_call"] = {"ms": re_ms, "samples": sub, "samples_per_s": sub / re_ms * 1e3,
                                           "what": "reference CUDA extension: get_comb_hij_fused + wavefunction_lut + torch scatter/divide/sum"}
    except Exception as e:  # the comparator is optional: never fail the bench on it
        ref_cuda = {"unavailable": repr(e)[:200]}
    # REDUCE method (SURVEY.md 8f-2): kept rows only; eps at the 90th percentile of |H| of the first samples
    eps = float(torch.quantile(hmat[:64].abs().flatten()[:: 7], 0.9))
    del comb, hmat, flat, idx, mask
    r_ms, (xk, hk, ik, off) = t(lambda: ops.get_comb_hij_reduced(x, h1e, h2e, SORB, NELE, NOA, NOB, eps, prepared=prep))
    kept = int(ik.numel())
    rb = kept * (8 + 8 + 8) + 8 * (chunk + 1)
    reduce_entry = {"bound": "issue", "kernel": "reduce_kernel<1,double> count + emit (+ diag, scan) = get_comb_hij_reduced, eps = %.3g" % eps,
                    "ms": r_ms, "samples_per_s": chunk / r_ms * 1e3, "rows_per_s": chunk * M / r_ms * 1e3, "kept_fraction": kept / (chunk * M),
                    "output_bytes_per_launch": rb, "samples_per_launch": chunk,
                    "note": "two passes over the rows (count, emit) instead of writing and re-reading [n, M] arrays; includes the "
                            "host read of K between them"}
    return [
        {"bound": "hbm", "kernel": "enumerate_kernel<1,double,true> (+diag_kernel) = get_comb_hij_fused", "achieved": fb / f_ms / 1e6,
         "peak": peak, "unit": "GB/s", "frac": fb / f_ms / 1e6 / peak, "traffic": prof.get("enumerate_dram_bytes_per_launch"),
         "algorithmic_bytes_per_launch": fb, "samples_per_launch": chunk, "ms": f_ms, "samples_per_s": chunk / f_ms * 1e3,
         "vs_reference_cuda": ref_cuda.get("fused", ref_cuda)},
        {"bound": "hbm", "kernel": "lut_batched_kernel (four consecutive queries per thread) = wavefunction_lut", "achieved": lb / l_ms / 1e6, "peak": peak,
         "unit": "GB/s", "frac": lb / l_ms / 1e6 / peak, "traffic": prof.get("lut_dram_bytes_per_launch"),
         "algorithmic_bytes_per_launch": lb, "samples_per_launch": chunk, "ms": l_ms, "samples_per_s": chunk / l_ms * 1e3,
         "vs_reference_cuda": ref_cuda.get("lut", ref_cuda)},
        reduce_entry,
        {"kernel": "reference CUDA three-call E_loc (GPU-vs-GPU comparator of the headline value)", **ref_cuda.get("eloc_three_call", ref_cuda)},
    ]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference_cuda"])
    ap.add_argument("--samples", type=int, default=1_000_000)
    ap.add_argument("--ref-samples", type=int, default=4096, help="samples per step of the reference CPU arm")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of reference CPU work behind cpu_baseline / parity")
    ap.add_argument("--variant-parity-samples", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api-path", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--table", default="uniform", help="sample set of the main measurement: uniform (the headline) or zipf0.8")
    ap.add_argument("--no-graph", action="store_true", help="launch the step kernel by kernel instead of replaying its CUDA graph")
    ap.add_argument("--no-peer", action="store_true", help="NCCL collectives only (no NVLink peer-memory pull kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the E_loc, psi0 and energy statistics of the last timed step "
                                                          "as .npy files in DIR (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl != "ours":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
