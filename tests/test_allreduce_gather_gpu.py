"""Parity of the zero-copy gather allreduce (b2_allreduce_gather) against the CPU oracle, kernel by kernel.

DistributedDataParallel sends every bucket through this entry point by default: the kernels read their input through a
table of up to B2_MAX_SEGMENTS per-parameter tensors instead of the bucket.  For rank r the expected result is the oracle
applied to r's segments joined in bucket order.  The tables are built by hand so that the lookup meets its edges: vecs
that straddle up to 8 segments, segment pointers at every alignment, pointers that are not monotonic in the bucket order,
segments that are the bucket itself, and messages cut into several launches with the cuts inside segments.  Every call
also checks that no source tensor was written and that the canaries around `out` survive.
"""
import numpy as np
import pytest
import torch

import oracle
from tests._util import (MODES, WIRE, Guarded, World, assert_bits_equal, assert_nvls_result, devices, garbage, host_elems,
                         make_inputs, to_host, upload)
from torchx_b200.ddp import _native as N

pytestmark = pytest.mark.gpu

# Segment lengths, cycled: eight 1-element parameters in a row make one vec straddle 8 segments; the rest are ragged
# around multiples of 8 and 256.
PATTERN = [1] * 8 + [2, 3, 7, 8, 9, 13, 31, 33, 255, 257, 4097]
DEFAULT_N = sum(PATTERN[i % len(PATTERN)] for i in range(N.B2_MAX_SEGMENTS))  # one full table of PATTERN
LAYOUTS = ["one", "ragged", "shared", "mixed"]
# "twoshot_pipe_1k": the pipelined two-shot with 1 KiB chunks, so that K reaches 16
ALGOS = ["oneshot", "twoshot", "twoshot_pipe", "twoshot_pipe_1k", "twoshot_ll", "auto"]
STAGE_N = (3 << 20) + 17  # with stage_mb=1: several launches for every algorithm, world and mode


def _lengths(nseg, n):
    """nseg segment lengths cycling PATTERN, the long ones stretched so that they sum to n (DEFAULT_N: PATTERN itself)."""
    base = [PATTERN[i % len(PATTERN)] for i in range(nseg)]
    small = sum(b for b in base if b < 255)
    m = (n - small) // sum(b for b in base if b >= 255)
    out = [b * m if b >= 255 else b for b in base]
    out[-1] += n - sum(out)
    assert min(out) > 0 and sum(out) == n
    return out


def _places(layout, lens, seed):
    """Where each segment lives: ("src", k) = at element k of the rank's source allocation, ("out", None) = at its own
    place in `out` (the segment is the bucket view, which the ABI allows).  Returns (places, source allocation size)."""
    nseg = len(lens)
    places, at = [None] * nseg, 0
    if layout == "shared":  # one tensor, the segments packed into it in a random order: table pointers not monotonic
        at = 5
        for i in np.random.default_rng(seed).permutation(nseg):
            places[i] = ("src", at)
            at += lens[i]
        return places, at + 16
    for i, ln in enumerate(lens):
        if layout == "mixed" and i % 2 == 0:
            places[i] = ("out", None)
            continue
        k = at + (i * 3 // 2 % 8 if layout != "one" else 0)  # k % 8 != 0: not 32 B (fp32) / 16 B (bf16) aligned
        places[i] = ("src", k)
        at = (k + ln + 16) // 16 * 16  # each source in its own slot, with canary elements behind it
    return places, at + 16


class _Rank:
    """One rank's buffers: the source allocation (data at the places, garbage between) and the guarded `out` (garbage,
    except where a segment is the bucket view), both uploaded, plus the segment table pointing into them."""

    def __init__(self, concat, mode, device, lens, places, src_size, seed):
        self.mode = mode
        self.src_host = garbage(src_size, mode, seed)
        out_host = garbage(concat.size, mode, seed + 1)
        begins = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        for (where, k), b, e in zip(places, begins[:-1], begins[1:]):
            if where == "src":
                self.src_host[k:k + e - b] = concat[b:e]
            else:
                out_host[b:e] = concat[b:e]
        self.src = upload(self.src_host, device)
        self.out = Guarded(out_host, mode, device, seed=seed + 2)
        esize = self.src.element_size()
        self.segs = (N.B2Segment * len(lens))()
        for i, ((where, k), b, e) in enumerate(zip(places, begins[:-1], begins[1:])):
            base = self.src.data_ptr() + k * esize if where == "src" else self.out.t.data_ptr() + int(b) * esize
            self.segs[i].src, self.segs[i].begin, self.segs[i].end = base, int(b), int(e)

    def check_inputs(self, what):
        got = to_host(self.src, self.mode)
        bits = np.uint16 if self.mode == "bf16" else np.uint32
        bad = np.flatnonzero(got.view(bits) != self.src_host.view(bits))
        assert bad.size == 0, f"{what}: {bad.size} elements of the source tensors were written, first at {bad[:8]}"


def _check_gather(w, n, mode, algo, layout, seed, scale=None, kind="special"):
    W = len(w.comms)
    lens = [n] if layout == "one" else _lengths(N.B2_MAX_SEGMENTS, n)
    places, src_size = _places(layout, lens, seed)
    concats = [host_elems(x, mode) for x in make_inputs(W, n, seed, kind)]
    ranks = [_Rank(concats[r], mode, c.device, lens, places, src_size, seed + 10 * r) for r, c in enumerate(w.comms)]
    if scale is None:
        scale = 1.0 / W
    abi_algo = "twoshot_pipe" if algo == "twoshot_pipe_1k" else algo
    w.run(lambda r, c, s: c.allreduce_gather_(ranks[r].out.t, ranks[r].segs, len(lens), scale=scale, wire=WIRE[mode],
                                              algo=abi_algo, stream=s))
    what = f"gather W={W} n={n} mode={mode} algo={algo} layout={layout} nseg={len(lens)} scale={scale!r}"
    for r, rk in enumerate(ranks):
        rk.out.check(f"{what} rank={r}")
        rk.check_inputs(f"{what} rank={r}")
    got = [to_host(rk.out.t, mode) for rk in ranks]
    if W > 1 and w.comms[0].last_algo == "nvls":
        for r in range(W):
            assert_nvls_result(got[r], concats, scale, MODES[mode], f"{what} rank={r}")
            assert_bits_equal(got[r], got[0], f"{what}: rank {r} vs rank 0")
        return
    want = oracle.allreduce(MODES[mode], concats, scale)
    for r in range(W):
        assert_bits_equal(got[r], want, f"{what} rank={r}")


def _world(devs, algo, stage_mb=8):
    w = World(devs, stage_mb=stage_mb)
    if algo == "twoshot_pipe_1k":
        for c in w.comms:
            c.set_param("pipe_chunk_bytes", 1 << 10)
    return w


@pytest.mark.parametrize("world", [2, 3, 5, 7, 8])
@pytest.mark.parametrize("algo", ALGOS)
def test_gather_matches_oracle_one_device(world, algo):
    w = _world([0] * world, algo)
    try:
        for i, mode in enumerate(MODES):
            for j, layout in enumerate(LAYOUTS):
                n = 70001 if layout == "one" else DEFAULT_N
                _check_gather(w, n, mode, algo, layout, seed=10 * i + j, kind="special" if (i + j) % 2 else "randn")
    finally:
        w.close()


@pytest.mark.parametrize("world", [3, 7])
@pytest.mark.parametrize("algo", ALGOS)
def test_gather_several_launches(world, algo):
    """stage_mb=1: the message is cut into launches whose boundaries fall inside segments (Src::off moves the window)."""
    w = _world([0] * world, algo, stage_mb=1)
    try:
        for mode, layout in zip(MODES, ("ragged", "mixed", "shared")):
            before = w.comms[0].launches
            _check_gather(w, STAGE_N, mode, algo, layout, seed=31)
            assert w.comms[0].launches - before >= 3, (mode, algo)
    finally:
        w.close()


class _Solo(World):
    """W = 1: the gather runs through the fused local pass."""

    def __init__(self):
        from torchx_b200.ddp import Communicator

        self.comms = [Communicator.create(0, 1, 0, "/unused")]
        self.streams = [torch.cuda.Stream(device=0)]


@pytest.mark.parametrize("mode", list(MODES))
def test_gather_local_pass(mode):
    """In f32 mode with scale 1 there is nothing to compute, but `out` (garbage here) must still receive the sources."""
    w = _Solo()
    try:
        for i, layout in enumerate(LAYOUTS):
            for scale in (1.0, 0.125, 1.0 / 3.0):
                _check_gather(w, 70001 if layout == "one" else DEFAULT_N, mode, "auto", layout, seed=i, scale=scale)
            # several trips per thread: the segment hint is reused within a parameter and invalidated at its end
            _check_gather(w, (1 << 22) + 3, mode, "auto", layout, seed=40 + i, scale=1.0)
        _check_gather(w, (1 << 24) + 3, mode, "auto", "ragged", seed=50, scale=1.0)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("algo", ALGOS + ["nvls"])
def test_gather_across_devices(world, algo, cuda_count):
    """One rank per GPU over NVLink, in one launch and in several; nvls where the fabric offers multicast (without the
    fp32-wire mode, as in test_allreduce_across_devices)."""
    devs = devices(world, cuda_count, spread=True)
    for stage_mb in (64, 1):
        w = _world(devs, algo, stage_mb=stage_mb)
        try:
            if algo == "nvls" and not w.comms[0].has_multicast:
                pytest.skip("no NVSwitch multicast on this box")
            for mode in MODES:
                if algo == "nvls" and mode == "f32":
                    continue
                if stage_mb == 1:
                    before = w.comms[0].launches
                    _check_gather(w, STAGE_N, mode, algo, "mixed", seed=7)
                    assert w.comms[0].launches - before >= 3, (mode, algo)
                    continue
                for j, layout in enumerate(LAYOUTS):
                    _check_gather(w, 70001 if layout == "one" else DEFAULT_N, mode, algo, layout, seed=j)
        finally:
            w.close()
