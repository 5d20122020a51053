"""Shared helpers for the parity tests (CPU side: numpy + oracle; GPU side: torch tensors)."""
from __future__ import annotations

import dataclasses
import enum

import numpy as np

import oracle

MODES = {"f32_wire_bf16": oracle.B2O_F32_WIRE_BF16, "f32": oracle.B2O_F32, "bf16": oracle.B2O_BF16}
WIRE = {"f32_wire_bf16": "bf16", "f32": "f32", "bf16": "bf16"}
GUARD = 64  # canary elements on each side of every tensor a kernel writes

SPECIALS = np.array(
    [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 1.17549435e-38, 3.3895314e38, -3.3895314e38, 1.0, -1.0,
     1.00390625, 1.0078125, 1.01171875, 65504.0, 1e-3, -1e-3, 255.0, 256.0, 257.0],
    dtype=np.float32,
)


def make_inputs(world: int, n: int, seed: int, kind: str = "randn") -> list:
    """Per-rank fp32 buckets. kinds: randn (seed 1234+rank as in SURVEY §8d), special (inf/nan/subnormal/
    cancellation sprinkled in), onehot (the reference's own compute_world_size trick), ints (exact in bf16)."""
    out = []
    for r in range(world):
        rng = np.random.default_rng(seed + 1234 + r)
        if kind == "randn":
            x = rng.standard_normal(n).astype(np.float32)
        elif kind == "special":
            x = rng.standard_normal(n).astype(np.float32)
            if n:
                idx = rng.integers(0, n, size=max(1, n // 7))
                x[idx] = SPECIALS[rng.integers(0, len(SPECIALS), size=idx.size)]
                if n > 4:
                    x[1] = 3.25 if r % 2 == 0 else -3.25  # cancellation across rank pairs
        elif kind == "onehot":
            x = np.zeros(n, dtype=np.float32)
            x[r::world] = 1.0
        elif kind == "ints":
            x = rng.integers(-120, 121, size=n).astype(np.float32)
        else:
            raise ValueError(kind)
        out.append(x)
    return out


def encode(v, subst: dict):
    """JSON form of a value crossing the Runner -> scheduler boundary (tests/golden/reference_dropin.json): dataclasses
    and enums by class name, other objects by type name only, and every ``subst`` key inside a string replaced by its
    token, so that run-specific paths and ids compare equal."""
    if isinstance(v, enum.Enum):
        return {"__enum__": [type(v).__name__, v.name]}
    if dataclasses.is_dataclass(v) and not isinstance(v, type):
        return {"__dataclass__": type(v).__name__, "fields": {f.name: encode(getattr(v, f.name), subst) for f in dataclasses.fields(v)}}
    if isinstance(v, dict):
        return {str(k): encode(x, subst) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [encode(x, subst) for x in v]
    if isinstance(v, str):
        for k, tok in subst.items():
            v = v.replace(k, tok)
        return v
    if v is None or isinstance(v, (bool, int, float)):
        return v
    return {"__object__": type(v).__name__}


def assert_bits_equal(got: np.ndarray, want: np.ndarray, what: str = "") -> None:
    """Bit-exact comparison; NaNs must coincide but their payload may differ (cvt.rn gives 0x7fff,
    torch's CPU path 0x7fc0)."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.dtype == np.uint16:
        gf, wf = oracle.bf16_bits_to_f32(got), oracle.bf16_bits_to_f32(want)
        gi, wi = got, want
    else:
        gf, wf = got.astype(np.float32, copy=False), want.astype(np.float32, copy=False)
        gi, wi = gf.view(np.uint32), wf.view(np.uint32)
    gn, wn = np.isnan(gf), np.isnan(wf)
    assert np.array_equal(gn, wn), f"{what}: NaN positions differ at {np.flatnonzero(gn != wn)[:8]}"
    bad = np.flatnonzero((gi != wi) & ~gn)
    assert bad.size == 0, (
        f"{what}: {bad.size} of {got.size} elements differ; first at {bad[:8]}: got {gf[bad[:8]]} want {wf[bad[:8]]}"
    )


def assert_nvls_result(got: np.ndarray, inputs: list, scale: float, mode: int, what: str = "") -> dict:
    """The NVLS path lets the NVSwitch add the W wire contributions (fp32 accumulation, one rounding to bf16).  The
    switch's summation ORDER is not the rank order of the P2P kernels, so the contract checked here is:
      * wherever the exact sum of the contributions is representable in fp32 along EVERY summation order the result is
        order-independent and must equal the rank-order oracle bit for bit (the overwhelming majority of elements);
      * elsewhere it must equal the correctly rounded bf16 of SOME fp32 summation order: checked as within one bf16 ulp
        of the exact (float64) sum.
    Returns counts for reporting."""
    want = oracle.allreduce(mode, inputs, scale)
    contrib = [oracle.compress(mode, x, scale).astype(np.float64) for x in inputs]  # bf16-representable values
    exact = np.sum(contrib, axis=0)
    if got.dtype == np.uint16:
        gf, wf = oracle.bf16_bits_to_f32(got), oracle.bf16_bits_to_f32(want)
    else:
        gf, wf = got.astype(np.float32), want.astype(np.float32)
    gn, wn = np.isnan(gf), np.isnan(wf)
    assert np.array_equal(gn, wn), f"{what}: NaN positions differ at {np.flatnonzero(gn != wn)[:8]}"
    diff = np.flatnonzero((gf.view(np.uint32) != wf.view(np.uint32)) & ~gn)
    if diff.size:
        # order-independence test: every partial sum of |c_r| spans < 2^24 relative to the smallest contribution bit
        absmax = np.max(np.abs(contrib), axis=0)[diff]
        ulp = np.maximum(np.abs(exact[diff]), np.float64(2.0) ** -126) * 2.0 ** -7  # >= one bf16 ulp of the result
        err = np.abs(gf[diff].astype(np.float64) - exact[diff])
        bad = diff[(err > ulp) & np.isfinite(exact[diff])]
        assert bad.size == 0, (
            f"{what}: {bad.size} elements are more than one bf16 ulp from the exact sum; first at {bad[:8]}: "
            f"got {gf[bad[:8]]} exact {exact[bad[:8]]} rank-order {wf[bad[:8]]}")
        del absmax
    return {"n": int(got.size), "differ_from_rank_order": int(diff.size)}


# ---- GPU side ------------------------------------------------------------------------------------------------------
def devices(world: int, cuda_count: int, spread: bool) -> list:
    """Device of each rank: one rank per GPU (skips the test without enough GPUs) or every rank on cuda:0."""
    import pytest

    if spread:
        if cuda_count < world:
            pytest.skip(f"needs {world} GPUs")
        return list(range(world))
    return [0] * world


class World:
    """An in-process topology (b2_comm_create_local): rank r launches on its own stream of devices[r]."""

    def __init__(self, devices, stage_mb=8, timeout_s=10.0):
        import torch
        from torchx_b200.ddp import Communicator

        self.comms = Communicator.create_local(devices, stage_mb=stage_mb)
        self.streams = [torch.cuda.Stream(device=d) for d in devices]
        same_device = len(set(devices)) == 1
        for c in self.comms:
            c.set_timeout(timeout_s)
            if same_device:  # all kernels must be co-resident on one GPU: W ranks x grid <= #SMs (1 CTA per SM)
                c.set_max_ctas(max(1, 128 // len(devices)))

    def run(self, fn):
        """fn(rank, comm, stream) launches that rank's work; then wait for all and check health.  fn must not allocate
        or synchronise: the ranks launched before it spin until every peer has launched."""
        for r, (c, s) in enumerate(zip(self.comms, self.streams)):
            fn(r, c, s)
        for s in self.streams:
            s.synchronize()
        for c in self.comms:
            c.check()

    def close(self):
        for c in self.comms:
            c.close()


def host_elems(x: np.ndarray, mode: str) -> np.ndarray:
    """fp32 values as the tensor of `mode` holds them: fp32, or bf16 bit patterns (uint16) in bf16 mode."""
    return oracle.f32_to_bf16_bits(x) if mode == "bf16" else x


def _int_view(a: np.ndarray) -> np.ndarray:
    return a.view(np.uint16) if a.dtype.itemsize == 2 else a.view(np.uint32)


def upload(h: np.ndarray, device):
    """Host elements (fp32, or uint16 bf16 bits) -> the same bits in a float32 / bfloat16 tensor, NaN payloads included."""
    import torch

    bits = _int_view(np.ascontiguousarray(h))
    if bits.dtype == np.uint16:
        return torch.from_numpy(bits.view(np.int16).copy()).to(f"cuda:{device}").view(torch.bfloat16)
    return torch.from_numpy(bits.view(np.int32).copy()).to(f"cuda:{device}").view(torch.float32)


def to_dev(x: np.ndarray, mode: str, device):
    h = host_elems(x, mode)
    return upload(h, device), h


def to_host(t, mode: str) -> np.ndarray:
    import torch

    if mode == "bf16":
        return t.view(torch.int16).cpu().numpy().view(np.uint16)
    return t.cpu().numpy()


def garbage(n: int, mode: str, seed: int) -> np.ndarray:
    """Random bit patterns (NaNs and infinities included) in the element type of `mode`."""
    rng = np.random.default_rng(seed)
    if mode == "bf16":
        return rng.integers(0, 1 << 16, size=n, dtype=np.uint16)
    return rng.integers(0, 1 << 32, size=n, dtype=np.uint32).view(np.float32)


class Guarded:
    """A device tensor `t` holding the host elements `h`, placed `offset` elements after GUARD canary elements and
    followed by GUARD more, all in one allocation.  A store past either end of `t` lands in a canary, where the caching
    allocator's slack would have hidden it."""

    def __init__(self, h: np.ndarray, mode: str, device, offset: int = 0, seed: int = 0):
        n = h.size
        self.mode = mode
        self.lo, self.hi = GUARD + offset, GUARD + offset + n
        self.init = garbage(self.hi + GUARD, mode, seed)
        _int_view(self.init)[self.lo:self.hi] = _int_view(np.ascontiguousarray(h))
        self.full = upload(self.init, device)
        self.t = self.full[self.lo:self.hi]

    def check(self, what: str = "") -> None:
        got = _int_view(to_host(self.full, self.mode))
        want = _int_view(self.init)
        for name, sl in (("before", slice(0, self.lo)), ("after", slice(self.hi, None))):
            bad = np.flatnonzero(got[sl] != want[sl])
            assert bad.size == 0, f"{what}: {bad.size} canary elements {name} the tensor were overwritten, first at {bad[:8]}"
