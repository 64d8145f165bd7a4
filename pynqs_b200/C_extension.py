"""Host mirror of the reference operator API `libs.C_extension` (stubs: libs/C_extension.pyi;
bindings: cpp_src/tensor/bind.cpp:317-391) on top of libpynqs_b200.so.

Same function names, keyword names, tensor layouts, dtypes and exception types.  Differences,
all deliberate (SURVEY.md section 8b):
  * CUDA only -- CPU tensors raise RuntimeError (the product has no CPU fallback);
  * MAX_SORB_LEN is dispatched at run time from the tensor width (1, 2 or 3 words);
  * shape problems raise ValueError instead of tripping an assert / exit(1);
  * kernels run on torch's current stream of the tensor's device.
Outputs are allocated with torch (caching allocator); the C side never allocates.
"""
from __future__ import annotations

import weakref
from typing import Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib
from ._lib import i64, vp

MAX_SORB_LEN: int = 3
MAX_SORB: int = 192
MAX_NELE: int = 120

# queries >= this (and >= N / 8) switch wavefunction_lut from the classic search to the hash index
_HASH_MIN_QUERIES = 1 << 15


# ------------------------------------------------------------------------------------------------
def _need_cuda(*tensors: Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if not isinstance(t, Tensor):
            raise TypeError(f"expected torch.Tensor, got {type(t)}")
        if not t.is_cuda:
            raise NotImplementedError(
                "pynqs_b200 operators are CUDA-only (no CPU fallback, by design): move the tensors to a B200 device, or keep "
                "the reference's CPU build of libs.C_extension for host-side callers (CI matrices, gloo runs) -- INTEGRATION.md section 4"
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors on different devices: {dev} vs {t.device}")
    return dev


def _contig(t: Tensor, name: str) -> None:
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")  # CHECK_CONTIGUOUS, bind.cpp:45-48,72


def _onv_words(t: Tensor, name: str) -> int:
    if t.dtype != torch.uint8:
        raise ValueError(f"{name} must be torch.uint8, got {t.dtype}")
    w = t.size(-1)
    if w % 8 or not 1 <= w // 8 <= MAX_SORB_LEN:
        raise ValueError(f"{name}: last dim {w} must be 8, 16 or 24 bytes")
    return w // 8


def _check_width(t: Tensor, sorb: int, name: str) -> int:
    L = _onv_words(t, name)
    if L != (sorb - 1) // 64 + 1:
        raise ValueError(f"{name}: width {8 * L} bytes does not match sorb = {sorb}")  # bind.cpp:73-75
    return L


def _stream(dev: torch.device):
    return vp(torch.cuda.current_stream(dev).cuda_stream)


def _fdtype(h1e: Tensor, h2e: Tensor) -> int:
    if h1e.dtype != h2e.dtype:
        raise ValueError(f"h1e ({h1e.dtype}) and h2e ({h2e.dtype}) must have the same dtype")
    if h1e.dtype == torch.float64:
        return _lib.F64
    if h1e.dtype == torch.float32:
        return _lib.F32
    raise ValueError(f"h1e/h2e must be float32 or float64, got {h1e.dtype}")  # AT_DISPATCH_FLOATING_TYPES


def _check_integrals(h1e: Tensor, h2e: Tensor, sorb: int) -> None:
    pair = sorb * (sorb - 1) // 2
    if h1e.numel() != sorb * sorb or h2e.numel() != pair * (pair + 1) // 2:
        raise ValueError(
            f"packed integrals have {h1e.numel()} / {h2e.numel()} elements, expected "
            f"{sorb * sorb} / {pair * (pair + 1) // 2} for sorb = {sorb}"
        )


# ------------------------------------------------------------------------------------------------
def check_sorb(sorb: int, nele: int) -> None:
    """check_sorb (bind.cpp:282-301): ValueError for an unsupported sorb, OverflowError for too many electrons."""
    _lib.check(_lib.load().pynqs_check_sorb(int(sorb), int(nele)))


def get_Num_SinglesDoubles(sorb: int, noA: int, noB: int) -> int:
    """number of singles + doubles (cpp_src/cpu/excitation.cpp:8-16; utils/public_function.py:132-144)."""
    out = _lib.ctypes.c_int64()
    _lib.check(_lib.load().pynqs_num_sd(int(sorb), int(noA), int(noB), _lib.ctypes.byref(out)))
    return int(out.value)


def tensor_to_onv(bra: Tensor, sorb: int) -> Tensor:
    """0/1 uint8 states [n, sorb] (or [sorb]) -> packed ONV uint8 [n, 8L]   (C_extension.pyi:5-24)."""
    dev = _need_cuda(bra)
    _contig(bra, "bra")
    if bra.dtype != torch.uint8 or bra.dim() not in (1, 2):
        raise ValueError("bra must be a 1-D or 2-D torch.uint8 tensor")
    L = (sorb - 1) // 64 + 1
    if bra.numel() == 0:
        return torch.empty((0, 8 * L), dtype=torch.uint8, device=dev)
    if bra.numel() % sorb:
        raise ValueError(f"bra has {bra.numel()} elements, not a multiple of sorb = {sorb}")
    n = bra.numel() // sorb
    out = torch.empty((n, 8 * L), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().pynqs_tensor_to_onv(vp(bra.data_ptr()), i64(n), int(sorb), vp(out.data_ptr()), _stream(dev)))
    return out


def onv_to_tensor(bra: Tensor, sorb: int) -> Tensor:
    """packed ONV uint8 [n, 8L] (or [8L]) -> +-1 tensor [n, sorb] in torch.get_default_dtype()
    (C_extension.pyi:26-45, cpu_tensor.cpp:55)."""
    dev = _need_cuda(bra)
    _contig(bra, "bra")
    if bra.dim() not in (1, 2):
        raise ValueError("bra must be 1-D or 2-D")
    L = _check_width(bra, sorb, "bra")  # the kernel strides by ceil(sorb / 64) words
    bra2 = bra.view(-1, 8 * L)
    dtype = torch.get_default_dtype()
    if dtype not in (torch.float32, torch.float64):
        raise ValueError(f"default dtype {dtype} unsupported")
    n = bra2.size(0)
    out = torch.empty((n, sorb), dtype=dtype, device=dev)
    if n == 0:
        return out
    code = _lib.F64 if dtype == torch.float64 else _lib.F32
    with torch.cuda.device(dev):
        _lib.check(_lib.load().pynqs_onv_to_tensor(vp(bra2.data_ptr()), i64(n), int(sorb), vp(out.data_ptr()), code, _stream(dev)))
    return out


def get_comb_tensor(bra: Tensor, sorb: int, nele: int, noA: int, noB: int, flag_bit: bool = False) -> Tuple[Tensor, Tensor]:
    """All singles and doubles of every bra (C_extension.pyi:47-90): comb uint8 [n, M, 8L], row 0 = bra.
    Second value: +-1 states double [n, M, sorb] if flag_bit else ones(1) on the CPU, exactly as the
    reference returns it (cpu_tensor.cpp:191, cuda_tensor.cpp:247)."""
    dev = _need_cuda(bra)
    _contig(bra, "bra")
    if bra.dim() == 1:
        bra = bra.view(1, -1)
    L = _check_width(bra, sorb, "bra")
    M = get_Num_SinglesDoubles(sorb, noA, noB) + 1
    n = bra.size(0)
    comb = torch.empty((n, M, 8 * L), dtype=torch.uint8, device=dev)
    states = torch.empty((n, M, sorb), dtype=torch.float64, device=dev) if flag_bit else None
    if n:
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_comb(
                    vp(bra.data_ptr()), i64(n), int(sorb), int(noA), int(noB), vp(comb.data_ptr()),
                    vp(states.data_ptr() if flag_bit else None), _stream(dev),
                )
            )
    if not flag_bit:
        states = torch.ones(1, dtype=torch.float64)
    return comb, states


class PreparedIntegrals:
    """Gather-friendly device copy of the packed h2e (csrc/prepare.cu): same numbers, bit for bit."""

    def __init__(self, h2e: Tensor, sorb: int):
        dev = _need_cuda(h2e)
        _contig(h2e, "h2e")
        code = _fdtype(h2e, h2e)
        nbytes = _lib.ctypes.c_int64()
        _lib.check(_lib.load().pynqs_prepared_bytes(int(sorb), code, _lib.ctypes.byref(nbytes)))
        self.sorb, self.dtype = sorb, h2e.dtype
        self.workspace = torch.empty(max(nbytes.value, 16), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_prepare_integrals(vp(h2e.data_ptr()), int(sorb), code, vp(self.workspace.data_ptr()), i64(nbytes.value), _stream(dev))
            )

    @property
    def nbytes(self) -> int:
        return self.workspace.numel()


def pin_in_l2(t: "Tensor | None", hit_ratio: float = 0.0) -> Tuple[int, int]:
    """Keep a tensor (h2e, a PreparedIntegrals workspace, a table copy) resident in a persisting-L2 window for the kernels
    launched afterwards on the current stream; pin_in_l2(None) lifts it.  Returns (bytes set aside, window bytes).
    For Hamiltonians too large to stay in L2 by themselves next to the streaming outputs (H50: 98 MB of h2e)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if t is None else _need_cuda(t)
    granted = (_lib.ctypes.c_int64 * 2)()
    with torch.cuda.device(dev):
        _lib.check(_lib.load().pynqs_l2_persist(vp(None if t is None else t.data_ptr()), i64(0 if t is None else t.numel() * t.element_size()),
                                               _lib.ctypes.c_double(float(hit_ratio)), _stream(dev), granted))
    return int(granted[0]), int(granted[1])


_prep_cache: dict = {}
# preparing costs one pass over ~(sorb/2)^4 elements: only worth it when the call writes more than that
_PREP_MIN_OUTPUT_RATIO = 4
# the prepared copy is O((sorb/2)^4) elements (1.07 GB in FP64 at 192 spin orbitals): get_comb_hij_fused only builds
# one on its own below this size (above it the packed arrays are read directly -- identical results), and at most
# _PREP_CACHE_ENTRIES of them are kept alive (least recently used first out)
PREPARED_AUTO_MAX_BYTES = 2 << 30
_PREP_CACHE_ENTRIES = 4


def prepared_nbytes(sorb: int, dtype: torch.dtype) -> int:
    nbytes = _lib.ctypes.c_int64()
    code = _lib.F64 if dtype == torch.float64 else _lib.F32
    _lib.check(_lib.load().pynqs_prepared_bytes(int(sorb), code, _lib.ctypes.byref(nbytes)))
    return int(nbytes.value)


def _cached_prep(h2e: Tensor, sorb: int) -> PreparedIntegrals:
    """Per-tensor-object cache: valid while the same h2e tensor object is alive and unmodified."""
    k = id(h2e)
    ent = _prep_cache.pop(k, None)
    if ent is not None:
        ref, version, ptr, prep = ent
        if ref() is h2e and version == h2e._version and ptr == h2e.data_ptr() and prep.sorb == sorb:
            _prep_cache[k] = ent  # most recently used last
            return prep
    prep = PreparedIntegrals(h2e, sorb)
    while len(_prep_cache) >= _PREP_CACHE_ENTRIES:
        _prep_cache.pop(next(iter(_prep_cache)))
    _prep_cache[k] = (weakref.ref(h2e, lambda _r, k=k: _prep_cache.pop(k, None)), h2e._version, h2e.data_ptr(), prep)
    return prep


def get_comb_hij_fused(bra: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int,
                       *, prepared: "PreparedIntegrals | None | bool" = None) -> Tuple[Tensor, Tensor]:
    """Fused enumeration + <x|H|x'> (C_extension.pyi:125-137): (comb uint8 [n, M, 8L], Hmat [n, M]).
    `prepared`: a PreparedIntegrals of h2e, None = build/cache one when the call is large enough,
    False = read the packed arrays directly (identical results)."""
    dev = _need_cuda(bra, h1e, h2e)
    for t, nm in ((bra, "bra"), (h1e, "h1e"), (h2e, "h2e")):
        _contig(t, nm)
    if bra.dim() == 1:
        bra = bra.view(1, -1)
    L = _check_width(bra, sorb, "bra")
    code = _fdtype(h1e, h2e)
    _check_integrals(h1e, h2e, sorb)
    M = get_Num_SinglesDoubles(sorb, noA, noB) + 1
    n = bra.size(0)
    comb = torch.empty((n, M, 8 * L), dtype=torch.uint8, device=dev)
    hmat = torch.empty((n, M), dtype=h1e.dtype, device=dev)
    if n:
        if prepared is None:
            na = sorb // 2
            big = n * M >= _PREP_MIN_OUTPUT_RATIO * (na**4 + sorb**3) or id(h2e) in _prep_cache
            if big and id(h2e) not in _prep_cache and prepared_nbytes(sorb, h2e.dtype) > PREPARED_AUTO_MAX_BYTES:
                big = False  # too large to build unasked: pass a PreparedIntegrals explicitly to use the table-driven kernel
            prepared = _cached_prep(h2e, sorb) if big else False
        prep_ptr = prepared.workspace.data_ptr() if prepared else None
        if prepared and (prepared.sorb != sorb or prepared.dtype != h2e.dtype):
            raise ValueError("prepared integrals do not match sorb / dtype")
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_comb_hij_fused(
                    vp(bra.data_ptr()), vp(h1e.data_ptr()), vp(h2e.data_ptr()), vp(prep_ptr), i64(n), int(sorb), int(nele),
                    int(noA), int(noB), vp(comb.data_ptr()), vp(hmat.data_ptr()), code, _stream(dev),
                )
            )
    return comb, hmat


def get_comb_hij_reduced(bra: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int, eps: float,
                         *, prepared: "PreparedIntegrals | None" = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Additive op for the REDUCE method (vmc/energy/eloc.py:257-297): what the reference obtains from
    get_comb_tensor + get_hij_torch + torch.where(|Hmat| >= eps), without materialising [n, M] arrays.
    Returns (x uint8 [K, 8L], hij [K], gt_eps_idx int64 [K], offsets int64 [n + 1]): the kept determinants,
    their matrix elements (bit-identical to get_comb_hij_fused), their flat indices s * M + m in ascending
    order (= torch.where's), and the first kept row of every sample.  One host synchronisation (K)."""
    dev = _need_cuda(bra, h1e, h2e)
    for t, nm in ((bra, "bra"), (h1e, "h1e"), (h2e, "h2e")):
        _contig(t, nm)
    if bra.dim() == 1:
        bra = bra.view(1, -1)
    L = _check_width(bra, sorb, "bra")
    code = _fdtype(h1e, h2e)
    _check_integrals(h1e, h2e, sorb)
    get_Num_SinglesDoubles(sorb, noA, noB)  # geometry / overflow checks
    if not (eps >= 0.0):
        raise ValueError("eps must be >= 0")
    n = bra.size(0)
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    if n == 0:
        return (torch.empty((0, 8 * L), dtype=torch.uint8, device=dev), torch.empty(0, dtype=h1e.dtype, device=dev),
                torch.empty(0, dtype=torch.int64, device=dev), offsets)
    if prepared is None:
        prepared = _cached_prep(h2e, sorb)
    if prepared.sorb != sorb or prepared.dtype != h2e.dtype:
        raise ValueError("prepared integrals do not match sorb / dtype")
    lib = _lib.load()
    nbytes = int(lib.pynqs_reduce_scratch_bytes(i64(n)))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    common = (vp(bra.data_ptr()), vp(h1e.data_ptr()), vp(h2e.data_ptr()), vp(prepared.workspace.data_ptr()), i64(n), int(sorb),
              int(nele), int(noA), int(noB), _lib.ctypes.c_double(float(eps)), code, vp(scratch.data_ptr()), i64(nbytes))
    with torch.cuda.device(dev):
        _lib.check(lib.pynqs_reduce_count(*common, vp(offsets.data_ptr()), _stream(dev)))
        K = int(offsets[n].item())
        x = torch.empty((K, 8 * L), dtype=torch.uint8, device=dev)
        hij = torch.empty(K, dtype=h1e.dtype, device=dev)
        idx = torch.empty(K, dtype=torch.int64, device=dev)
        _lib.check(lib.pynqs_reduce_emit(*common, vp(offsets.data_ptr()), vp(x.data_ptr()), vp(hij.data_ptr()), vp(idx.data_ptr()),
                                         _stream(dev)))
    return x, hij, idx, offsets


def get_comb_hij_sampled(bra: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int, eps: float, eps_sample: int,
                         *, seed: int | None = None, draws: Tensor | None = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Additive op for the stochastic / semi-stochastic REDUCE method (vmc/energy/eloc.py:257-283, eps_sample > 0):
    per sample, eps_sample draws from p(m) ~ |H_m| over the rows with |H_m| < eps (all rows if eps == 0); the element of a
    drawn row becomes (count / eps_sample) * H_m / p(m); rows with |H_m| >= eps (eps > 0) are kept exactly.  eps is compared
    in the integrals' dtype, like torch.where(|Hmat| >= eps) and get_comb_hij_reduced.  A sample whose sub-eps magnitudes
    sum to 0 has nothing drawn (where torch.multinomial would raise); the generator never draws a row with H_m == 0.
    Returns (x uint8 [K, 8L], hij [K], gt_eps_idx int64 [K], offsets int64 [n + 1]) like get_comb_hij_reduced; per sample the
    kept rows (ascending) come first, then the drawn ones (ascending).  Nothing of size [n, M] or [n, eps_sample] is stored.
    seed: Philox key (default: drawn from torch's CPU generator, so torch.manual_seed makes runs reproducible);
    draws: int64 [n, eps_sample] row indices to use instead of the generator (what torch.multinomial returned)."""
    dev = _need_cuda(bra, h1e, h2e)
    for t, nm in ((bra, "bra"), (h1e, "h1e"), (h2e, "h2e")):
        _contig(t, nm)
    if bra.dim() == 1:
        bra = bra.view(1, -1)
    L = _check_width(bra, sorb, "bra")
    code = _fdtype(h1e, h2e)
    _check_integrals(h1e, h2e, sorb)
    M = get_Num_SinglesDoubles(sorb, noA, noB) + 1
    if not (eps >= 0.0) or int(eps_sample) < 1:
        raise ValueError("eps must be >= 0 and eps_sample >= 1")
    n = bra.size(0)
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    if n == 0:
        return (torch.empty((0, 8 * L), dtype=torch.uint8, device=dev), torch.empty(0, dtype=h1e.dtype, device=dev),
                torch.empty(0, dtype=torch.int64, device=dev), offsets)
    draws_ptr = None
    if draws is not None:
        _need_cuda(draws)
        draws = draws.to(torch.int64).contiguous()
        if draws.shape != (n, int(eps_sample)):
            raise ValueError(f"draws must be [n, eps_sample] = [{n}, {eps_sample}]")
        if int(draws.min()) < 0 or int(draws.max()) >= M:
            raise ValueError("draws: row index outside [0, M)")
        draws_ptr = draws.data_ptr()
    if seed is None:
        seed = int(torch.randint(0, 2**62, (1,)).item())
    lib = _lib.load()
    nbytes = int(lib.pynqs_reduce_sample_scratch_bytes(i64(n)))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    common = (vp(bra.data_ptr()), vp(h1e.data_ptr()), vp(h2e.data_ptr()), i64(n), int(sorb), int(nele), int(noA), int(noB),
              _lib.ctypes.c_double(float(eps)), int(eps_sample), _lib.ctypes.c_uint64(int(seed) & (2**64 - 1)), vp(draws_ptr), code,
              vp(scratch.data_ptr()), i64(nbytes))
    with torch.cuda.device(dev):
        _lib.check(lib.pynqs_reduce_sample_count(*common, vp(offsets.data_ptr()), _stream(dev)))
        K = int(offsets[n].item())
        x = torch.empty((K, 8 * L), dtype=torch.uint8, device=dev)
        hij = torch.empty(K, dtype=h1e.dtype, device=dev)
        idx = torch.empty(K, dtype=torch.int64, device=dev)
        _lib.check(lib.pynqs_reduce_sample_emit(*common, vp(offsets.data_ptr()), vp(x.data_ptr()), vp(hij.data_ptr()), vp(idx.data_ptr()),
                                                _stream(dev)))
    return x, hij, idx, offsets


def reduce_eloc(psi: Tensor, hij: Tensor, gt_eps_idx: Tensor, offsets: Tensor, M: int) -> Tuple[Tensor, Tensor]:
    """eloc[s] = sum over the kept rows of sample s of (psi_k / psi0) * hij_k -- the last lines of _reduce_psi
    (eloc.py:283-297) on the compacted rows.  psi0 = psi of the sample's row 0 (0 if it was not kept, as in the
    reference).  Returns (eloc [n], psi0 [n]) in psi's dtype (float64 or complex128)."""
    dev = _need_cuda(psi, hij, gt_eps_idx, offsets)
    if psi.dtype not in (torch.float64, torch.complex128):
        raise ValueError("psi must be float64 or complex128")
    psi = psi.contiguous()
    hij = hij.to(torch.float64).contiguous()
    gt_eps_idx = gt_eps_idx.contiguous()
    offsets = offsets.contiguous()
    if hij.numel() != psi.numel() or gt_eps_idx.numel() != psi.numel() or offsets.dtype != torch.int64 or gt_eps_idx.dtype != torch.int64:
        raise ValueError("psi, hij and gt_eps_idx must have one entry per kept row; offsets / gt_eps_idx int64")
    n = offsets.numel() - 1
    eloc = torch.empty(n, dtype=psi.dtype, device=dev)
    psi0 = torch.empty(n, dtype=psi.dtype, device=dev)
    if n > 0:
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_reduce_eloc(
                    vp(psi.data_ptr()), int(psi.is_complex()), vp(hij.data_ptr()), vp(gt_eps_idx.data_ptr()), vp(offsets.data_ptr()),
                    i64(n), i64(M), vp(eloc.data_ptr()), vp(psi0.data_ptr()), _stream(dev),
                )
            )
    return eloc, psi0


def get_hij_torch(bra: Tensor, ket: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int) -> Tensor:
    """<bra|H|ket> (C_extension.pyi:92-123): ket 3-D [n, m, 8L] -> local-energy layout [n, m];
    ket 2-D [m, 8L] -> matrix [n, m].  dtype/device of h1e."""
    dev = _need_cuda(bra, ket, h1e, h2e)
    for t, nm in ((bra, "bra"), (ket, "ket"), (h1e, "h1e"), (h2e, "h2e")):
        _contig(t, nm)
    if bra.dim() != 2 or ket.dim() not in (2, 3):
        raise ValueError("bra must be 2-D and ket 2-D or 3-D")
    L = _check_width(bra, sorb, "bra")
    if _onv_words(ket, "ket") != L:
        raise ValueError("bra and ket widths differ")
    code = _fdtype(h1e, h2e)
    _check_integrals(h1e, h2e, sorb)
    n = bra.size(0)
    ket3d = ket.dim() == 3
    if ket3d and ket.size(0) != n:
        raise ValueError(f"ket batch {ket.size(0)} != bra batch {n}")
    m = ket.size(1) if ket3d else ket.size(0)
    out = torch.empty((n, m), dtype=h1e.dtype, device=dev)
    if n and m:
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_hij(
                    vp(bra.data_ptr()), vp(ket.data_ptr()), vp(h1e.data_ptr()), vp(h2e.data_ptr()), i64(n), i64(m),
                    int(ket3d), int(sorb), int(nele), vp(out.data_ptr()), code, _stream(dev),
                )
            )
    return out


# ---- hash index over a sorted key table ---------------------------------------------------------
class HashIndex:
    """Device hash index of a sorted unique key table (internal accelerator of the lookups)."""

    def __init__(self, bra_key: Tensor):
        dev = _need_cuda(bra_key)
        _contig(bra_key, "bra_key")
        self.L = _onv_words(bra_key, "bra_key")
        self.N = bra_key.size(0)
        self.key_ptr = bra_key.data_ptr()
        nbytes = _lib.ctypes.c_int64()
        _lib.check(_lib.load().pynqs_hash_bytes(i64(self.N), self.L, _lib.ctypes.byref(nbytes)))
        self.workspace = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_hash_build(
                    vp(bra_key.data_ptr()), i64(self.N), self.L, vp(self.workspace.data_ptr()), i64(nbytes.value), _stream(dev)
                )
            )

    @property
    def nbytes(self) -> int:
        return self.workspace.numel()


_hash_cache: dict = {}


def hash_worthwhile(n_queries: int, n_keys: int) -> bool:
    """The hash index costs ~200 bytes per key to build: only for query batches that amortise it."""
    return n_queries >= _HASH_MIN_QUERIES and 8 * n_queries >= n_keys and n_keys < (1 << 32)


def _cached_hash(bra_key: Tensor) -> HashIndex:
    """Per-tensor-object cache: valid while the same tensor object is alive and unmodified."""
    k = id(bra_key)
    ent = _hash_cache.get(k)
    if ent is not None:
        ref, version, ptr, hidx = ent
        if ref() is bra_key and version == bra_key._version and ptr == bra_key.data_ptr():
            return hidx
    hidx = HashIndex(bra_key)
    _hash_cache[k] = (weakref.ref(bra_key, lambda _r, k=k: _hash_cache.pop(k, None)), bra_key._version, bra_key.data_ptr(), hidx)
    return hidx


# ---- string-grouped copies of a sorted key table (what the local-energy kernels scan) ----------------
class GroupIndex:
    """The key table bucketed by the hash of the beta string and, a second time, of the alpha string
    (csrc/gindex.cuh); internal to eloc_sample_space."""

    def __init__(self, bra_key: Tensor):
        dev = _need_cuda(bra_key)
        _contig(bra_key, "bra_key")
        self.L = _onv_words(bra_key, "bra_key")
        self.N = bra_key.size(0)
        self.key_ptr = bra_key.data_ptr()
        nbytes = _lib.ctypes.c_int64()
        _lib.check(_lib.load().pynqs_group_bytes(i64(self.N), self.L, _lib.ctypes.byref(nbytes)))
        self.workspace = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(
                _lib.load().pynqs_group_build(
                    vp(bra_key.data_ptr()), i64(self.N), self.L, vp(self.workspace.data_ptr()), i64(nbytes.value), _stream(dev)
                )
            )

        lay = (_lib.ctypes.c_int64 * 10)()
        _lib.check(_lib.load().pynqs_group_layout(i64(self.N), self.L, lay))
        self._layout = list(lay)

    @property
    def nbytes(self) -> int:
        return self.workspace.numel()

    def keys(self, grouping: int = 0) -> Tensor:
        """the table's keys in bucket order (uint8 [N, 8L]): grouping 0 = bucketed by beta string, 1 = by alpha string"""
        o = self._layout[3 + grouping]
        return self.workspace[o : o + self.N * 8 * self.L].view(self.N, 8 * self.L)

    def pos(self) -> Tensor:
        """position in keys(0) of every row of the sorted table (int32 [N]): the inverse of rows(0)"""
        o = self._layout[9]
        return self.workspace[o : o + self.N * 4].view(torch.int32)

    def rows(self, grouping: int = 0) -> Tensor:
        """row in the sorted table of every key of keys(grouping) (int32 [N])"""
        o = self._layout[5 + grouping]
        return self.workspace[o : o + self.N * 4].view(torch.int32)


_group_cache: dict = {}


def _cached_group(bra_key: Tensor) -> GroupIndex:
    """Per-tensor-object cache: valid while the same tensor object is alive and unmodified."""
    k = id(bra_key)
    ent = _group_cache.get(k)
    if ent is not None:
        ref, version, ptr, gidx = ent
        if ref() is bra_key and version == bra_key._version and ptr == bra_key.data_ptr():
            return gidx
    gidx = GroupIndex(bra_key)
    _group_cache[k] = (weakref.ref(bra_key, lambda _r, k=k: _group_cache.pop(k, None)), bra_key._version, bra_key.data_ptr(), gidx)
    return gidx


def wavefunction_lut(bra_key: Tensor, onv: Tensor, sorb: int, little_endian: bool = True, *,
                     hash_index: "HashIndex | None | bool" = None) -> Tuple[Tensor, Tensor]:
    """Index of every onv row in the sorted key table (C_extension.pyi:305-357): (idx int64 [n]
    with -1 for absent rows, mask bool [n]).  The ONV width comes from the tensors, not from
    `sorb` (DetLUT passes a prefix length, utils/det_helper/determinant_lut.py:285-291).
    hash_index: a HashIndex of bra_key; None = build / reuse one when the query batch is large enough to pay for it
    (~200 bytes per key); False = always the classic binary search."""
    if not little_endian:
        raise NotImplementedError("little_endian=False is broken in the reference (cpu_tensor.cpp:613) and never used")
    dev = _need_cuda(bra_key, onv)
    _contig(bra_key, "bra_key")
    _contig(onv, "onv")
    L = _onv_words(bra_key, "bra_key")
    if onv.dim() != 2 or _onv_words(onv, "onv") != L:
        raise ValueError("onv must be 2-D with the same width as bra_key")  # exit(1) in cuda_tensor.cpp:445-449
    n, N = onv.size(0), bra_key.size(0)
    idx = torch.empty(n, dtype=torch.int64, device=dev)
    mask = torch.empty(n, dtype=torch.bool, device=dev)
    if n == 0:
        return idx, mask
    lib = _lib.load()
    if hash_index is None and hash_worthwhile(n, N):
        hash_index = _cached_hash(bra_key)
    if hash_index is not None and hash_index is not False and (hash_index.N != N or hash_index.L != L or hash_index.key_ptr != bra_key.data_ptr()):
        raise ValueError("hash_index was built for another key table")
    with torch.cuda.device(dev):
        if hash_index:
            _lib.check(
                lib.pynqs_lut_hashed(
                    vp(bra_key.data_ptr()), i64(N), vp(onv.data_ptr()), i64(n), L, vp(hash_index.workspace.data_ptr()),
                    vp(idx.data_ptr()), vp(mask.data_ptr()), _stream(dev),
                )
            )
        else:
            _lib.check(
                lib.pynqs_lut(vp(bra_key.data_ptr()), i64(N), vp(onv.data_ptr()), i64(n), L, vp(idx.data_ptr()), vp(mask.data_ptr()), _stream(dev))
            )
    return idx, mask


def eloc_sample_space(
    bra: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int,
    bra_key: Tensor, wf_value: Tensor, group_index: GroupIndex | None = None,
) -> Tuple[Tensor, Tensor]:
    """Additive op: the whole sample-space local energy of vmc/energy/eloc.py:326-397 in one pass.
    Returns (eloc [n], psi0 [n]) in wf_value's dtype (float64 or complex128).  bra_key must be the
    sorted unique table and wf_value its values in the same order."""
    dev = _need_cuda(bra, h1e, h2e, bra_key, wf_value)
    for t, nm in ((bra, "bra"), (h1e, "h1e"), (h2e, "h2e"), (bra_key, "bra_key"), (wf_value, "wf_value")):
        _contig(t, nm)
    if bra.dim() != 2 or bra_key.dim() != 2 or wf_value.dim() != 1:
        raise ValueError("bra and bra_key must be 2-D [rows, 8L], wf_value 1-D")
    L = _check_width(bra, sorb, "bra")
    if _onv_words(bra_key, "bra_key") != L:
        raise ValueError("bra and bra_key widths differ")
    if h1e.dtype != torch.float64 or h2e.dtype != torch.float64:
        raise ValueError("eloc_sample_space needs float64 integrals")
    _check_integrals(h1e, h2e, sorb)
    if wf_value.dtype not in (torch.float64, torch.complex128) or wf_value.numel() != bra_key.size(0):
        raise ValueError("wf_value must be float64/complex128 with one value per key")
    cplx = int(wf_value.dtype == torch.complex128)
    n, N = bra.size(0), bra_key.size(0)
    eloc = torch.empty(n, dtype=wf_value.dtype, device=dev)
    psi0 = torch.empty(n, dtype=wf_value.dtype, device=dev)
    if n == 0:
        return eloc, psi0
    if group_index is None:
        group_index = _cached_group(bra_key)
    if group_index.N != N or group_index.L != L or group_index.key_ptr != bra_key.data_ptr():
        raise ValueError("group_index was built for another key table")
    lib = _lib.load()
    nbytes = _lib.ctypes.c_int64()
    _lib.check(lib.pynqs_eloc_scratch_bytes(i64(n), int(sorb), int(noA), int(noB), cplx, _lib.ctypes.byref(nbytes)))
    scratch = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.pynqs_eloc_sample_space(
                vp(bra.data_ptr()), i64(n), vp(h1e.data_ptr()), vp(h2e.data_ptr()), int(sorb), int(nele), int(noA), int(noB),
                vp(bra_key.data_ptr()), vp(wf_value.data_ptr()), cplx, i64(N), vp(group_index.workspace.data_ptr()),
                vp(scratch.data_ptr()), i64(nbytes.value), vp(eloc.data_ptr()), vp(psi0.data_ptr()), _stream(dev),
            )
        )
    return eloc, psi0


def sample_space_hamiltonian(
    bra: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int,
    bra_key: Tensor, group_index: GroupIndex | None = None,
) -> Tuple[Tensor, Tensor, Tensor]:
    """Additive op: H[i, j] = <bra_i|H|bra_key_j> as CSR arrays (crow int64 [n + 1], col int64 [nnz], val float64 [nnz]) --
    the rows of get_hij_torch(bra, bra_key) restricted to the entries eloc_sample_space sums over: bra_i itself (when it is in
    the table) and its single and double excitations that are in the table.  Entries are structural (exact zeros are kept),
    columns ascend within a row, values are bit-identical to get_hij_torch.  One host synchronisation (nnz)."""
    dev = _need_cuda(bra, h1e, h2e, bra_key)
    for t, nm in ((bra, "bra"), (h1e, "h1e"), (h2e, "h2e"), (bra_key, "bra_key")):
        _contig(t, nm)
    if bra.dim() != 2 or bra_key.dim() != 2:
        raise ValueError("bra and bra_key must be 2-D [rows, 8L]")
    L = _check_width(bra, sorb, "bra")
    if _onv_words(bra_key, "bra_key") != L:
        raise ValueError("bra and bra_key widths differ")
    if h1e.dtype != torch.float64 or h2e.dtype != torch.float64:
        raise ValueError("sample_space_hamiltonian needs float64 integrals")
    _check_integrals(h1e, h2e, sorb)
    get_Num_SinglesDoubles(sorb, noA, noB)  # geometry / overflow checks
    n, N = bra.size(0), bra_key.size(0)
    crow = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    if n == 0 or N == 0:
        return crow, torch.empty(0, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.float64, device=dev)
    if group_index is None:
        group_index = _cached_group(bra_key)
    if group_index.N != N or group_index.L != L or group_index.key_ptr != bra_key.data_ptr():
        raise ValueError("group_index was built for another key table")
    lib = _lib.load()

    def scratch_for(nnz: int) -> Tensor:
        nbytes = _lib.ctypes.c_int64()
        _lib.check(lib.pynqs_hamiltonian_scratch_bytes(i64(n), i64(nnz), int(sorb), int(noA), int(noB), _lib.ctypes.byref(nbytes)))
        return torch.empty(nbytes.value, dtype=torch.uint8, device=dev)

    table = (vp(bra_key.data_ptr()), i64(N), vp(group_index.workspace.data_ptr()))
    with torch.cuda.device(dev):
        scratch = scratch_for(0)
        _lib.check(lib.pynqs_hamiltonian_count(vp(bra.data_ptr()), i64(n), int(sorb), int(noA), int(noB), *table, vp(scratch.data_ptr()),
                                               i64(scratch.numel()), vp(crow.data_ptr()), _stream(dev)))
        nnz = int(crow[n].item())
        del scratch
        scratch = scratch_for(nnz)
        col = torch.empty(nnz, dtype=torch.int64, device=dev)
        val = torch.empty(nnz, dtype=torch.float64, device=dev)
        _lib.check(lib.pynqs_hamiltonian_emit(vp(bra.data_ptr()), i64(n), vp(h1e.data_ptr()), vp(h2e.data_ptr()), int(sorb), int(nele),
                                              int(noA), int(noB), *table, vp(scratch.data_ptr()), i64(scratch.numel()), vp(crow.data_ptr()),
                                              i64(nnz), vp(col.data_ptr()), vp(val.data_ptr()), _stream(dev)))
    return crow, col, val


def csr_matmul(crow: Tensor, col: Tensor, val: Tensor, X: Tensor, N: int) -> Tensor:
    """Y = H X for the CSR matrix H [n, N] of sample_space_hamiltonian (crow int64 [n + 1], col int64 [nnz] < N, val float64
    [nnz]).  X: float64 or complex128, [N] or [N, k] of any k (rows may be strided, columns must be adjacent or X is
    copied); Y has X's dtype and shape with n rows.  H is real, so a complex X is multiplied as its torch.view_as_real
    view, real and imaginary parts in one pass.  The kernel takes 8 columns per call; wider blocks go through in column
    slices of X and Y.  Deterministic (identical bits on every call); no host synchronisation."""
    dev = _need_cuda(crow, col, val, X)
    if crow.dtype != torch.int64 or col.dtype != torch.int64 or val.dtype != torch.float64:
        raise ValueError("crow and col must be int64, val float64")
    if crow.dim() != 1 or crow.numel() < 1 or col.dim() != 1 or val.shape != col.shape:
        raise ValueError("crow must be 1-D [n + 1], col and val 1-D of the same length")
    for t, nm in ((crow, "crow"), (col, "col"), (val, "val")):
        _contig(t, nm)
    N = int(N)
    n = crow.numel() - 1
    Xr, ldx = _real_block(X, N)
    kk = Xr.size(1)
    work = n > 0 and N > 0 and col.numel() > 0 and kk > 0
    Y = (torch.empty if work else torch.zeros)((n, kk), dtype=torch.float64, device=dev)
    if work:
        lib = _lib.load()
        with torch.cuda.device(dev):
            for c0 in range(0, kk, 8):
                k = min(8, kk - c0)
                _lib.check(lib.pynqs_csr_spmm(vp(crow.data_ptr()), vp(col.data_ptr()), vp(val.data_ptr()), i64(n), i64(N),
                                              vp(Xr.data_ptr() + 8 * c0), i64(ldx), int(k), vp(Y.data_ptr() + 8 * c0), i64(kk),
                                              _stream(dev)))
    return _from_real_block(Y, X)


def _real_block(X: Tensor, N: int) -> Tuple[Tensor, int]:
    """X float64 / complex128 [N] or [N, k] as the real row-major block the block kernels read: (Xr float64 [N, k'], ldx),
    k' = k for a real X and 2k for a complex one (its torch.view_as_real view, real and imaginary parts as adjacent
    columns).  Rows may be strided; columns that are not adjacent are copied."""
    if X.dtype not in (torch.float64, torch.complex128):
        raise ValueError(f"X must be float64 or complex128, got {X.dtype}")
    if X.dim() not in (1, 2) or X.size(0) != N:
        raise ValueError(f"X must be [N] or [N, k] with N = {N}, got {tuple(X.shape)}")
    Xr = X.unsqueeze(1) if X.dim() == 1 else X
    if (Xr.size(1) > 1 and Xr.stride(1) != 1) or (N > 1 and Xr.stride(0) < Xr.size(1)):
        Xr = Xr.contiguous()  # the kernel reads rows of adjacent columns, rows apart by ldx >= k
    if X.is_complex():
        Xr = torch.view_as_real(Xr.resolve_conj())
        Xr = Xr.as_strided((N, 2 * Xr.size(1)), (Xr.stride(0), 1))  # [N, k, 2] with adjacent columns -> real [N, 2k]
    return Xr, (Xr.stride(0) if N > 1 else Xr.size(1))  # a single row's stride is not meaningful


def _from_real_block(Y: Tensor, X: Tensor) -> Tensor:
    """The real result block Y [n, k'] of a kernel that read _real_block(X) in X's dtype and shape."""
    n = Y.size(0)
    if X.is_complex():
        Y = torch.view_as_complex(Y.view(n, Y.size(1) // 2, 2))
    return Y.view(n) if X.dim() == 1 else Y


def spin_square_matmul(bra: Tensor, sorb: int, bra_key: Tensor, X: Tensor, group_index: GroupIndex | None = None) -> Tensor:
    """Y = S^2 X over the sorted key table: Y[i] = sum over j of <bra_i|S^2|bra_key_j> X[j] (pynqs_spin_square_apply).  The
    diagonal |B| + Sz (Sz + 1) counts when bra_i is in the table; the +1 of each spin exchange of bra_i (an alpha-only and a
    beta-only orbital that swap their spins) counts when that determinant is in the table.  Sz comes from each row's own
    bits.  With bra = bra_key this is S^2 restricted to the sample set, in the table's row order.

    X: float64 or complex128, [N] or [N, k] of any k, handled as csr_matmul handles it; Y has X's dtype and shape with n
    rows.  group_index: the table's GroupIndex (WavefunctionLUT.group_index), built and cached when not given.
    Deterministic (identical bits on every call); no host synchronisation."""
    dev = _need_cuda(bra, bra_key, X)
    for t, nm in ((bra, "bra"), (bra_key, "bra_key")):
        _contig(t, nm)
    if bra.dim() != 2 or bra_key.dim() != 2:
        raise ValueError("bra and bra_key must be 2-D [rows, 8L]")
    L = _check_width(bra, sorb, "bra")
    if _onv_words(bra_key, "bra_key") != L:
        raise ValueError("bra and bra_key widths differ")
    n, N = bra.size(0), bra_key.size(0)
    Xr, ldx = _real_block(X, N)
    kk = Xr.size(1)
    work = n > 0 and N > 0 and kk > 0
    Y = (torch.empty if work else torch.zeros)((n, kk), dtype=torch.float64, device=dev)
    if work:
        if group_index is None:
            group_index = _cached_group(bra_key)
        if group_index.N != N or group_index.L != L or group_index.key_ptr != bra_key.data_ptr():
            raise ValueError("group_index was built for another key table")
        lib = _lib.load()
        with torch.cuda.device(dev):
            for c0 in range(0, kk, 8):
                k = min(8, kk - c0)
                _lib.check(lib.pynqs_spin_square_apply(vp(bra.data_ptr()), i64(n), int(sorb), vp(bra_key.data_ptr()), i64(N),
                                                       vp(group_index.workspace.data_ptr()), vp(Xr.data_ptr() + 8 * c0), i64(ldx),
                                                       int(k), vp(Y.data_ptr() + 8 * c0), i64(kk), _stream(dev)))
    return _from_real_block(Y, X)


def rdm_offdiag(crow: Tensor, col: Tensor, bra_key: Tensor, c: Tensor, sorb: int, two_body: bool = True) -> Tuple[Tensor, "Tensor | None"]:
    """The off-diagonal part of the reduced density matrices of c over the sorted table (pynqs_rdm_offdiag): the sums over
    the entries (i, j != i) of the square CSR structure crow int64 [N + 1] / col int64 [nnz] (sample_space_hamiltonian with
    bra = bra_key) of conj(c_i) c_j <key_i| ... |key_j>, not normalised.  Returns dm1 [2, norb, norb] (alpha, beta) and dm2
    [3, norb, norb, norb, norb] (aa, ab, bb) in PySCF's make_rdm12s layout, or None when not two_body; c's dtype (float64 or
    complex128).  Deterministic (identical bits on every call); one host synchronisation (nnz)."""
    dev = _need_cuda(crow, col, bra_key, c)
    if crow.dtype != torch.int64 or col.dtype != torch.int64:
        raise ValueError("crow and col must be int64")
    if bra_key.dim() != 2 or crow.dim() != 1 or crow.numel() != bra_key.size(0) + 1 or col.dim() != 1:
        raise ValueError("bra_key must be 2-D [N, 8L], crow 1-D [N + 1], col 1-D")
    if c.dtype not in (torch.float64, torch.complex128) or c.shape != (bra_key.size(0),):
        raise ValueError(f"c must be float64 or complex128 [N] with N = {bra_key.size(0)}")
    for t, nm in ((crow, "crow"), (col, "col"), (bra_key, "bra_key"), (c, "c")):
        _contig(t, nm)
    _check_width(bra_key, sorb, "bra_key")
    N, norb = bra_key.size(0), sorb // 2
    nnz = int(crow[N].item())
    if nnz != col.numel():
        raise ValueError(f"crow[N] = {nnz} does not match col's {col.numel()} entries")
    cr = torch.view_as_real(c.resolve_conj()) if c.is_complex() else c
    dm1 = torch.empty((2, norb, norb), dtype=c.dtype, device=dev)
    dm2 = torch.empty((3, norb, norb, norb, norb), dtype=c.dtype, device=dev) if two_body else None
    lib = _lib.load()
    nbytes = _lib.ctypes.c_int64()
    _lib.check(lib.pynqs_rdm_scratch_bytes(i64(N), i64(nnz), int(sorb), _lib.ctypes.byref(nbytes)))
    scratch = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.pynqs_rdm_offdiag(vp(crow.data_ptr()), vp(col.data_ptr()), vp(bra_key.data_ptr()), i64(N), i64(nnz), int(sorb),
                                         vp(cr.data_ptr()), int(c.is_complex()), vp(scratch.data_ptr()), i64(nbytes.value),
                                         vp(dm1.data_ptr()), vp(dm2.data_ptr() if two_body else None), _stream(dev)))
    return dm1, dm2


_PT2_MAX_PAIRS = (1 << 31) - 1  # pairs of one pass: the table sort's limit


def pt2_log2_parts(upper_pairs: int, max_bytes: int, pass_bytes) -> int:
    """log2 of the smallest power of two P for which a pass of ceil(upper_pairs / P) pairs needs at most max_bytes of scratch
    (pass_bytes(pairs) -> bytes) and stays below 2^31 pairs.  ValueError when no P does."""
    lg = 0
    while True:
        pairs = -(-upper_pairs // (1 << lg))
        if pairs <= _PT2_MAX_PAIRS and pass_bytes(pairs) <= max_bytes:
            return lg
        if pairs <= 1 or lg >= 31:
            raise ValueError(f"max_bytes = {max_bytes} cannot hold a pass of the PT2 sum ({pass_bytes(1)} bytes at one pair)")
        lg += 1


def pt2_sums(bra_key: Tensor, C: Tensor, E: Tensor, h1e: Tensor, h2e: Tensor, sorb: int, nele: int, noA: int, noB: int,
             group_index: GroupIndex | None = None, max_bytes: int = 16 << 30) -> Tuple[Tensor, dict]:
    """The unnormalised Epstein-Nesbet sums of the columns of C over the sorted unique table bra_key (pynqs_pt2_*):
    acc[r] = sum over the externals a of (sum_i <key_i|H|a> C[i, r])^2 / (E[r] - <a|H|a>), float64 [k].  C: float64 [N, k]
    (any k: column slices of 8), E: float64 [k].  The externals are split into P = 2^log2 partitions, P the smallest power
    of two for which the scratch of a pass of N * nsd / P pairs fits in max_bytes (pt2_log2_parts); a partition whose exact
    count does not fit doubles P and restarts.  The passes' sums are added in pass order.  Returns (acc, info) with info["externals"],
    info["pairs"] and info["passes"].  Deterministic for a given P; one host synchronisation per pass."""
    dev = _need_cuda(bra_key, C, E, h1e, h2e)
    for t, nm in ((bra_key, "bra_key"), (h1e, "h1e"), (h2e, "h2e")):
        _contig(t, nm)
    if bra_key.dim() != 2 or C.dim() != 2 or C.size(0) != bra_key.size(0) or E.shape != (C.size(1),):
        raise ValueError("bra_key must be [N, 8L], C [N, k] and E [k]")
    if C.dtype != torch.float64 or E.dtype != torch.float64 or h1e.dtype != torch.float64 or h2e.dtype != torch.float64:
        raise ValueError("pt2_sums needs float64 C, E and integrals")
    _check_width(bra_key, sorb, "bra_key")
    _check_integrals(h1e, h2e, sorb)
    nsd = get_Num_SinglesDoubles(sorb, noA, noB)
    N, kk = bra_key.size(0), C.size(1)
    if N == 0:
        raise ValueError("the table is empty")
    if group_index is None:
        group_index = _cached_group(bra_key)
    if group_index.N != N or group_index.L != bra_key.size(1) // 8 or group_index.key_ptr != bra_key.data_ptr():
        raise ValueError("group_index was built for another key table")
    C = C.contiguous()
    E = E.contiguous()
    lib = _lib.load()

    def scratch_bytes(pairs: int) -> int:
        nb = _lib.ctypes.c_int64()
        _lib.check(lib.pynqs_pt2_scratch_bytes(i64(N), i64(pairs), int(sorb), _lib.ctypes.byref(nb)))
        return nb.value

    prep = _cached_prep(h2e, sorb)
    key = (vp(bra_key.data_ptr()), i64(N))
    lg = pt2_log2_parts(N * nsd, max_bytes, scratch_bytes)
    with torch.cuda.device(dev):
        offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
        count_scratch = torch.empty(scratch_bytes(0), dtype=torch.uint8, device=dev)
        while True:
            acc = torch.zeros(kk, dtype=torch.float64, device=dev)
            externals = torch.zeros(1, dtype=torch.int64, device=dev)
            pairs_total, restart = 0, False
            for part in range(1 << lg):
                sel = (vp(group_index.workspace.data_ptr()), int(part), int(lg))
                _lib.check(lib.pynqs_pt2_count(*key, int(sorb), int(noA), int(noB), *sel, vp(count_scratch.data_ptr()),
                                               i64(count_scratch.numel()), vp(offsets.data_ptr()), _stream(dev)))
                pairs = int(offsets[N].item())
                if pairs > _PT2_MAX_PAIRS or scratch_bytes(pairs) > max_bytes:  # a partition larger than planned
                    restart = True
                    break
                if pairs == 0:
                    continue
                pairs_total += pairs
                scratch = torch.empty(scratch_bytes(pairs), dtype=torch.uint8, device=dev)
                sc = (vp(scratch.data_ptr()), i64(scratch.numel()))
                _lib.check(lib.pynqs_pt2_emit(*key, vp(h1e.data_ptr()), vp(prep.workspace.data_ptr()), int(sorb), int(noA), int(noB), *sel,
                                              vp(offsets.data_ptr()), i64(pairs), *sc, _stream(dev)))
                _lib.check(lib.pynqs_pt2_sort(i64(N), i64(pairs), int(sorb), *sc, _stream(dev)))
                for c0 in range(0, kk, 8):
                    k = min(8, kk - c0)
                    _lib.check(lib.pynqs_pt2_reduce(i64(N), i64(pairs), vp(h1e.data_ptr()), vp(h2e.data_ptr()), int(sorb), int(nele),
                                                    vp(C.data_ptr() + 8 * c0), i64(kk), int(k), vp(E.data_ptr() + 8 * c0), *sc,
                                                    vp(acc.data_ptr() + 8 * c0), vp(externals.data_ptr() if c0 == 0 else None),
                                                    _stream(dev)))
                del scratch
            if not restart:
                return acc, {"externals": int(externals.item()), "pairs": pairs_total, "passes": 1 << lg}
            lg += 1


def lookup_compact(idx_array: Tensor, mask: Tensor, wf_value: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """(positions with mask set, positions without, wf_value[idx_array[mask]]) -- the index glue of
    WavefunctionLUT.lookup (utils/public_function.py:825-838: arange, two boolean-mask selections, masked_select, gather)
    in two passes of the library.  One host synchronisation (the number of hits), like the boolean indexing it replaces."""
    dev = _need_cuda(idx_array, mask, wf_value)
    n = idx_array.numel()
    if mask.dtype != torch.bool or mask.numel() != n or idx_array.dtype != torch.int64:
        raise ValueError("idx_array must be int64 and mask bool, of the same length")
    if wf_value.dim() != 1 or wf_value.element_size() not in (8, 16):
        raise ValueError("wf_value must be 1-D with 8- or 16-byte elements")
    _contig(idx_array, "idx_array")
    _contig(mask, "mask")
    _contig(wf_value, "wf_value")
    lib = _lib.load()
    nbytes = int(lib.pynqs_compact_scratch_bytes(i64(n)))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    n_hit = torch.zeros(1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.pynqs_lookup_count(vp(mask.data_ptr()), i64(n), vp(scratch.data_ptr()), i64(nbytes), vp(n_hit.data_ptr()), _stream(dev)))
        k = int(n_hit.item())
        hit = torch.empty(k, dtype=torch.int64, device=dev)
        miss = torch.empty(n - k, dtype=torch.int64, device=dev)
        value = torch.empty(k, dtype=wf_value.dtype, device=dev)
        _lib.check(lib.pynqs_lookup_emit(vp(mask.data_ptr()), vp(idx_array.data_ptr()), i64(n), vp(wf_value.data_ptr()),
                                         int(wf_value.element_size()), vp(scratch.data_ptr()), vp(hit.data_ptr()), vp(miss.data_ptr()),
                                         vp(value.data_ptr()), _stream(dev)))
    return hit, miss, value


def unique_onv(x: Tensor) -> Tuple[Tensor, Tensor]:
    """(distinct rows of x, inverse) with unique[inverse] == x -- what Func (vmc/energy/flip.py:44-61) asks of
    torch.unique(x, dim=0, return_inverse=True), on the library's radix sort instead of a comparison sort of rows.  The
    distinct rows come out ascending as ONV integers (torch.unique orders them byte 0 first); callers that only use
    unique[inverse] -- Func does -- see no difference."""
    dev = _need_cuda(x)
    _contig(x, "x")
    if x.dim() != 2:
        raise ValueError("x must be 2-D [rows, 8L]")
    L = _onv_words(x, "x")
    n = x.size(0)
    inverse = torch.empty(n, dtype=torch.int64, device=dev)
    if n == 0:
        return x.clone(), inverse
    key_sorted, _, perm = sort_table(x, None, 0, want_perm=True)
    lib = _lib.load()
    nbytes = int(lib.pynqs_compact_scratch_bytes(i64(n)))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    n_u = torch.zeros(1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.pynqs_unique_count(vp(key_sorted.data_ptr()), i64(n), L, vp(scratch.data_ptr()), i64(nbytes), vp(n_u.data_ptr()), _stream(dev)))
        k = int(n_u.item())
        uniq = torch.empty((k, 8 * L), dtype=torch.uint8, device=dev)
        _lib.check(lib.pynqs_unique_emit(vp(key_sorted.data_ptr()), vp(perm.data_ptr()), i64(n), L, vp(scratch.data_ptr()), vp(uniq.data_ptr()),
                                         vp(inverse.data_ptr()), _stream(dev)))
    return uniq, inverse


# ---- the steps either side of the kernels: table sort and energy moments ------------------------
def sort_table(bra_key: Tensor, wf_value: Tensor | None = None, sorb: int = 0, want_perm: bool = True):
    """Stable ascending sort of ONV rows as little-endian multi-word integers -- the order of the
    reference's torch_sort_onv (utils/public_function.py:626-689) -- applied to the keys and their
    values in one go.  Returns (sorted keys, sorted values or None, source row of every sorted row
    or None).  sorb > 0 promises that no key has a bit >= sorb set."""
    dev = _need_cuda(bra_key) if wf_value is None else _need_cuda(bra_key, wf_value)
    _contig(bra_key, "bra_key")
    L = _onv_words(bra_key, "bra_key")
    if bra_key.dim() != 2:
        raise ValueError("bra_key must be 2-D")
    N = bra_key.size(0)
    psi_bytes = 0
    if wf_value is not None:
        _contig(wf_value, "wf_value")
        if wf_value.dim() != 1 or wf_value.numel() != N or wf_value.element_size() not in (8, 16):
            raise ValueError("wf_value must hold one 8- or 16-byte value per key")
        psi_bytes = wf_value.element_size()
    key_out = torch.empty_like(bra_key)
    psi_out = torch.empty_like(wf_value) if wf_value is not None else None
    perm = torch.empty(N, dtype=torch.int64, device=dev) if want_perm else None
    if N == 0:
        return key_out, psi_out, perm
    lib = _lib.load()
    nbytes = int(lib.pynqs_sort_bytes(i64(N)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.pynqs_sort_table(
                vp(bra_key.data_ptr()), vp(wf_value.data_ptr() if wf_value is not None else None), i64(N), L, int(sorb), psi_bytes or 8,
                vp(key_out.data_ptr()), vp(psi_out.data_ptr() if psi_out is not None else None),
                vp(perm.data_ptr() if perm is not None else None), vp(ws.data_ptr()), i64(nbytes), _stream(dev),
            )
        )
    return key_out, psi_out, perm


_moment_scratch: dict = {}


def weighted_moments(eloc: Tensor, weight: Tensor, weight_is_amplitude: bool = False) -> Tensor:
    """[sum w, sum w Re d, sum w Im d, sum w |d|^2, Re c, Im c, n] (float64[7] on the device) with
    d = eloc - c, c = eloc[0]; w = weight, or |weight|^2 when weight_is_amplitude.  One kernel,
    deterministic; the building block of utils/stats/dist_stats.py:18-79."""
    dev = _need_cuda(eloc, weight)
    _contig(eloc, "eloc")
    _contig(weight, "weight")
    if eloc.dtype not in (torch.float64, torch.complex128) or eloc.dim() != 1 or weight.shape != eloc.shape:
        raise ValueError("eloc must be 1-D float64/complex128 and weight of the same shape")
    if weight_is_amplitude:
        if weight.dtype not in (torch.float64, torch.complex128):
            raise ValueError("amplitudes must be float64/complex128")
        kind = 2 if weight.dtype == torch.complex128 else 1
    else:
        if weight.dtype != torch.float64:
            raise ValueError("weights must be float64")
        kind = 0
    lib = _lib.load()
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    scratch = _moment_scratch.get(key)
    if scratch is None:
        scratch = torch.zeros(int(lib.pynqs_moments_scratch_bytes()), dtype=torch.uint8, device=dev)
        _moment_scratch[key] = scratch
    out = torch.empty(7, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.pynqs_weighted_moments(
                vp(eloc.data_ptr()), int(eloc.is_complex()), vp(weight.data_ptr()), kind, i64(eloc.numel()), vp(scratch.data_ptr()),
                vp(out.data_ptr()), _stream(dev),
            )
        )
    return out


# ---- names outside the hot path that callers import (SURVEY.md section 8b) -----------------------
def merge_rank_sample(idx: Tensor, counts: Tensor, split_idx: Tensor, length: int) -> Tensor:
    """merge_counts[idx[i]] += counts[i] (C_extension.pyi:256-279; merge_sample_cpu, cpu_tensor.cpp:537-556):
    int64 [length].  Integer atomics, so `split_idx` (which the reference's non-atomic CUDA kernel needs to keep
    equal indices apart, cuda/kernel.cu:520-536) is accepted and ignored."""
    dev = _need_cuda(idx, counts)
    idx = idx.to(torch.int64).contiguous()
    counts = counts.to(torch.int64).contiguous()
    if idx.dim() != 1 or counts.shape != idx.shape:
        raise ValueError("idx and counts must be 1-D of equal length")
    out = torch.empty(int(length), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().pynqs_merge_rank_sample(vp(idx.data_ptr()), vp(counts.data_ptr()), i64(idx.numel()), i64(length),
                                                       vp(out.data_ptr()), _stream(dev)))
    return out


def compress_h1e_h2e(h1e: np.ndarray, h2e: np.ndarray, sorb: int):
    """dense spin-orbital <pq||rs> -> packed 1-D arrays (cpp_src/tensor/integral.cpp:6-60)."""
    h1e = np.asarray(h1e, dtype=np.float64)
    h2e = np.asarray(h2e, dtype=np.float64)
    pair = sorb * (sorb - 1) // 2
    ii, jj = np.tril_indices(sorb, -1)  # i > j, ordered by pair index i(i-1)/2 + j
    block = h2e[ii[:, None], jj[:, None], ii[None, :], jj[None, :]]  # [pair, pair] = <ij||kl>
    r, c = np.tril_indices(pair)
    return h1e.reshape(-1).copy(), block[r, c].copy()


def decompress_h1e_h2e(h1e: np.ndarray, h2e: np.ndarray, sorb: int):
    """packed -> dense with the antisymmetry signs; entries with i == j or k == l are 0
    (the reference leaves them uninitialised, SURVEY.md Q5)."""
    pair = sorb * (sorb - 1) // 2
    sq = np.zeros((pair, pair))
    r, c = np.tril_indices(pair)
    sq[r, c] = h2e
    sq[c, r] = h2e
    ii, jj = np.tril_indices(sorb, -1)
    dense = np.zeros((sorb,) * 4)
    I, J = ii[:, None], jj[:, None]
    K, Lx = ii[None, :], jj[None, :]
    dense[I, J, K, Lx] = sq
    dense[J, I, K, Lx] = -sq
    dense[I, J, Lx, K] = -sq
    dense[J, I, Lx, K] = sq
    return np.asarray(h1e, dtype=np.float64).reshape(sorb, sorb).copy(), dense


def _not_on_path(name: str):
    def f(*_a, **_k):
        raise NotImplementedError(
            f"{name} is outside the local-energy hot path (SURVEY.md section 8) and is not provided by pynqs_b200"
        )

    f.__name__ = name
    return f


spin_flip_rand = _not_on_path("spin_flip_rand")
MCMC_sample = _not_on_path("MCMC_sample")
permute_sgn = _not_on_path("permute_sgn")
constrain_make_charts = _not_on_path("constrain_make_charts")
convert_sites = _not_on_path("convert_sites")
mps_vbatch = _not_on_path("mps_vbatch")
wavefunction_lut_map = _not_on_path("wavefunction_lut_map")
BKDR = _not_on_path("BKDR")
