"""Parity of the CUDA hot path (through the C ABI) against the CPU oracle.  All ranks of a topology live
in this process on one or more devices (b2_comm_create_local), each launching on its own stream - the same
kernels, flags and staging layout as the multi-process path, minus CUDA IPC (covered in test_ipc_gpu.py).
"""
import numpy as np
import pytest
import torch

import oracle
from tests._util import (MODES, WIRE, Guarded, World, assert_bits_equal, assert_nvls_result, devices, host_elems, make_inputs,
                         to_dev, to_host)

pytestmark = pytest.mark.gpu

SIZES = [1, 7, 8, 9, 1023, 1024, 1025, 4099, 32771, (1 << 18) + 5]


def _check_allreduce(world_obj, n, mode, algo, kind, seed, offset=0, scale=None, poke=None):
    """One allreduce of make_inputs(kind) on every rank of `world_obj`, compared with the oracle.  Each rank's tensor lies
    `offset` elements into its allocation, between canaries that must come through unchanged; `poke(rank, h)` may rewrite
    rank r's elements (raw bits: fp32, or uint16 bf16 patterns) before they are uploaded."""
    W = len(world_obj.comms)
    xs = make_inputs(W, n + offset, seed, kind)
    bufs, host = [], []
    for r, c in enumerate(world_obj.comms):
        h = host_elems(xs[r][offset:], mode).copy()
        if poke is not None:
            poke(r, h)
        bufs.append(Guarded(h, mode, c.device, offset=offset, seed=seed + r))
        host.append(h)
    if scale is None:
        scale = 1.0 / W
    world_obj.run(lambda r, c, s: c.allreduce_(bufs[r].t, scale=scale, wire=WIRE[mode], algo=algo, stream=s))
    what = f"W={W} n={n} mode={mode} algo={algo} kind={kind} scale={scale!r}"
    for r in range(W):
        bufs[r].check(f"{what} rank={r}")
    got = [to_host(b.t, mode) for b in bufs]
    ran_nvls = world_obj.comms[0].last_algo == "nvls"
    if ran_nvls and kind != "onehot":  # onehot: one non-zero term per element - exact on every path
        # the switch's own arithmetic (tools/nvls_probe.py, DESIGN.md 2.4): within one bf16 ulp of the exact sum
        stats = [assert_nvls_result(got[r], host, scale, MODES[mode], f"{what} rank={r}") for r in range(W)]
        for r in range(1, W):  # every rank holds the SAME bits (one reduction per element, replicated by the switch)
            assert_bits_equal(got[r], got[0], f"{what}: rank {r} vs rank 0")
        return stats[0]
    want = oracle.allreduce(MODES[mode], host, scale)
    for r in range(W):
        assert_bits_equal(got[r], want, f"{what} rank={r}")
    return None


@pytest.mark.parametrize("mode", list(MODES))
def test_local_pass_matches_oracle(mode):
    from torchx_b200.ddp import local_pass_

    for n in SIZES + [(1 << 22) + 3]:
        for kind in ("randn", "special"):
            for offset in (0, 1):
                x = make_inputs(1, n + offset, 7, kind)[0]
                t, h = to_dev(x, mode, 0)
                for scale in (1.0, 0.125, 1.0 / 3.0):
                    tt = t.clone()[offset:]
                    local_pass_(tt, scale=scale, wire=WIRE[mode])
                    torch.cuda.synchronize()
                    want = oracle.allreduce(MODES[mode], [h[offset:]], scale)
                    assert_bits_equal(to_host(tt, mode), want, f"local n={n} mode={mode} scale={scale} off={offset}")


@pytest.mark.parametrize("world", [2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("algo", ["oneshot", "twoshot", "twoshot_pipe", "twoshot_ll"])
def test_allreduce_matches_oracle_one_device(world, mode, algo):
    """SIZES 1..9 leave some ranks an empty slice; 768 * W elements end every slice (Ls = ceil(V / W) vecs) exactly on a
    32-vec pipeline unit, one more element starts the next unit."""
    w = World([0] * world)
    try:
        for i, n in enumerate(SIZES + [768 * world, 768 * world + 1]):
            _check_allreduce(w, n, mode, algo, "randn" if i % 2 == 0 else "special", seed=i)
        _check_allreduce(w, 4099, mode, algo, "randn", seed=99, offset=1)  # misaligned base pointer
        _check_allreduce(w, 1 << 12, mode, algo, "onehot", seed=0)
        _check_allreduce(w, 1 << 12, mode, algo, "ints", seed=0)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_allreduce_auto_and_chunking(world):
    """stage_mb=1 forces messages through several chunked launches; AUTO switches algorithm by size."""
    w = World([0] * world, stage_mb=1)
    try:
        for n in (100, 5000, 70001, (1 << 20) + 17):
            _check_allreduce(w, n, "f32_wire_bf16", "auto", "randn", seed=n)
        _check_allreduce(w, (1 << 19) + 3, "f32", "twoshot", "randn", seed=5)
        _check_allreduce(w, (1 << 20) + 9, "f32_wire_bf16", "twoshot_pipe", "special", seed=6)
        _check_allreduce(w, (1 << 20) + 11, "f32_wire_bf16", "twoshot_ll", "special", seed=7)
        _check_allreduce(w, (1 << 19) + 7, "bf16", "twoshot_ll", "randn", seed=8)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("chunk_kib", [1, 16, 4096])
def test_pipelined_two_shot_chunking(world, chunk_kib):
    """The warp-specialised pipeline over K chunks: tiny chunks force K = 16 with ragged last cells, one huge chunk is the
    K = 1 degenerate case; sizes around the cell / slice boundaries; every mode; misaligned buffers."""
    w = World([0] * world, stage_mb=8)
    try:
        for c in w.comms:
            c.set_param("pipe_chunk_bytes", chunk_kib << 10)
        for i, n in enumerate((1, 255, 256 * world, 256 * world + 1, 8 * 32 * world * 3 - 7, 70001, (1 << 19) + 13)):
            for mode in MODES:
                _check_allreduce(w, n, mode, "twoshot_pipe", "special" if i % 2 else "randn", seed=100 + i)
        _check_allreduce(w, 40961, "f32_wire_bf16", "twoshot_pipe", "randn", seed=7, offset=1)
        _check_allreduce(w, 1 << 14, "bf16", "twoshot_pipe", "ints", seed=8, offset=3)
    finally:
        w.close()


# 1 = plain SUM (dist.all_reduce); 2^-130 turns every wire value into a bf16 / fp32 subnormal (a flush-to-zero would show);
# 2^100 overflows the large `special` inputs to +-inf, and inf - inf makes NaN in the sum
SCALES = [1.0, 1.0 / 3.0, 0.1, 2.0 ** -130, 2.0 ** 100]


@pytest.mark.parametrize("world", [2, 3, 7])
@pytest.mark.parametrize("algo", ["oneshot", "twoshot", "twoshot_pipe", "twoshot_ll"])
def test_allreduce_any_scale_matches_oracle(world, algo):
    w = World([0] * world)
    try:
        for mode in MODES:
            for i, scale in enumerate(SCALES):
                for n in (4099, 70001):
                    _check_allreduce(w, n, mode, algo, "special", seed=200 + i, scale=scale)
    finally:
        w.close()


def _sentinel_nans(rank, h):
    """NaNs whose bits are the sentinel of the LL / NVLS buffers (0xFFFFFFFF: in bf16 two adjacent 0xFFFF elements, which
    f32_to_bf16_bits would never produce) and the negative default NaN, at positions shared by all ranks and at positions
    of this rank alone."""
    rng = np.random.default_rng(77 + rank)
    words = np.sort(np.concatenate([np.arange(0, h.size // 2, 97), rng.integers(0, h.size // 2, size=h.size // 64)]))
    if h.dtype == np.uint16:
        h[2 * words] = 0xFFFF
        h[2 * words + 1] = 0xFFFF
        h[2 * words[::3] + 1] = 0xFFC0  # every third pair: a negative NaN in the upper half of the word
    else:
        bits = h.view(np.uint32)
        bits[2 * words] = 0xFFFFFFFF
        bits[2 * words + 1] = 0xFFC00000


@pytest.mark.parametrize("world", [2, 3, 7])
def test_sentinel_bit_patterns_in_the_input(world):
    """Input words equal to the LL sentinel must come out as NaN and must not be taken for "not written yet" (which
    would end in a peer-wait timeout that check() reports)."""
    w = World([0] * world)
    try:
        for mode in MODES:
            for n in (4099, 70001, (1 << 18) + 5):
                _check_allreduce(w, n, mode, "twoshot_ll", "randn", seed=n, poke=_sentinel_nans)
                _check_allreduce(w, n, mode, "twoshot_ll", "randn", seed=n, scale=1.0, poke=_sentinel_nans)
    finally:
        w.close()


def test_back_to_back_ops_reuse_staging_safely():
    """40 collectives of mixed size/algorithm without host syncs in between: exercises the double-buffered
    staging + monotonically increasing flag sequence (no resets)."""
    W = 4
    w = World([0] * W)
    try:
        for c in w.comms:
            c.set_param("pipe_chunk_bytes", 1 << 10)
        plan = [(1000 + 37 * i, ("oneshot", "twoshot", "twoshot_pipe", "twoshot_ll", "twoshot_ll")[i % 5]) for i in range(45)]
        tens = [[None] * len(plan) for _ in range(W)]
        wants = []
        for k, (n, _) in enumerate(plan):
            xs = make_inputs(W, n, 1000 + k, "randn")
            for r in range(W):
                tens[r][k] = torch.from_numpy(xs[r]).to("cuda:0")
            wants.append(oracle.allreduce(oracle.B2O_F32_WIRE_BF16, xs, 1.0 / W))

        def launch(r, c, s):
            for k, (_, algo) in enumerate(plan):
                c.allreduce_(tens[r][k], algo=algo, stream=s)

        w.run(launch)
        for k in range(len(plan)):
            for r in range(W):
                assert_bits_equal(tens[r][k].cpu().numpy(), wants[k], f"op {k} rank {r}")
        assert w.comms[0].launches == len(plan)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 8])
def test_broadcast_and_barrier(world):
    w = World([0] * world, stage_mb=1)
    try:
        for nbytes, root, off in ((1, 0, 0), (15, 1, 0), (4096, world - 1, 0), (100003, 0, 1), ((3 << 20) + 5, 1, 0)):
            src = np.random.default_rng(nbytes).integers(0, 256, size=nbytes + off, dtype=np.uint8)
            tens = []
            for r in range(world):
                data = src if r == root else np.full(nbytes + off, r, dtype=np.uint8)
                tens.append(torch.from_numpy(data.copy()).to("cuda:0")[off:])
            w.run(lambda r, c, s: c.broadcast_(tens[r], root=root, stream=s))
            for r in range(world):
                assert np.array_equal(tens[r].cpu().numpy(), src[off:]), (nbytes, root, r)
        w.run(lambda r, c, s: c.barrier(stream=s))
    finally:
        w.close()


def test_identical_inputs_property_full_bucket_sizes():
    """Size-independent property at the real DDP bucket sizes (ResNet-50's 30.04 MiB fp32 bucket): when every
    rank holds the same x and W is a power of two, every partial sum k * bf16(x)/W is exact, so the result
    must be float(bf16(x)) bit for bit - checked against torch's own cast, no oracle pass over 7.9M elements."""
    W = 4
    n = 7_875_584  # 30.04 MiB of fp32, SURVEY §8a
    w = World([0] * W, stage_mb=16)
    try:
        x = torch.randn(n, device="cuda:0", generator=torch.Generator("cuda:0").manual_seed(3))
        tens = [x.clone() for _ in range(W)]
        w.run(lambda r, c, s: c.allreduce_(tens[r], stream=s))
        want = x.to(torch.bfloat16).float()
        for r in range(W):
            assert torch.equal(tens[r], want), r
    finally:
        w.close()


def test_dead_peer_times_out_instead_of_hanging():
    w = World([0, 0], timeout_s=0.3)
    try:
        t = torch.ones(4096, device="cuda:0")
        w.comms[0].allreduce_(t, stream=w.streams[0])  # rank 1 never shows up
        w.streams[0].synchronize()
        from torchx_b200.ddp._native import B2Error, B2_ETIMEOUT

        with pytest.raises(B2Error) as ei:
            w.comms[0].check()
        assert ei.value.code == B2_ETIMEOUT
        with pytest.raises(B2Error):  # poisoned: refuses further work
            w.comms[0].allreduce_(t, stream=w.streams[0])
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("algo", ["oneshot", "twoshot", "twoshot_pipe", "twoshot_ll", "nvls", "auto"])
def test_allreduce_across_devices(world, algo, cuda_count):
    """Real NVLink/NVSwitch peers (skipped on a 1-GPU box).  In-process worlds over distinct devices use the VMM arena and,
    where the fabric offers it, the multicast object - the same mappings as the one-process-per-GPU path minus fd passing."""
    devs = devices(world, cuda_count, spread=True)
    w = World(devs, stage_mb=64)
    try:
        if algo == "nvls" and not w.comms[0].has_multicast:
            pytest.skip("no NVSwitch multicast on this box")
        for c in w.comms:
            c.set_param("pipe_chunk_bytes", 64 << 10)
            c.set_param("nvls_min_bytes", 64 << 10)   # AUTO crosses one-shot -> NVLS / pipelined inside the sizes below
            c.set_param("pipe_min_bytes", 256 << 10)
        for mode in MODES:
            if algo == "nvls" and mode == "f32":
                continue  # fp32-wire NVLS (multimem.ld_reduce.add.f32): the switch's fp32 summation order; tools/nvls_probe.py
            for n in (9, 4099, (1 << 20) + 5):
                _check_allreduce(w, n, mode, algo, "special", seed=n)
            _check_allreduce(w, (1 << 20) + 5, mode, algo, "randn", seed=3)
            _check_allreduce(w, 1 << 16, mode, algo, "onehot", seed=0)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("algo", ["twoshot_ll", "nvls"])
def test_sentinel_bit_patterns_across_devices(world, algo, cuda_count):
    """The NVLS output buffers use the same sentinel as LL: an input word equal to it must not stall the switch path."""
    w = World(devices(world, cuda_count, spread=True), stage_mb=64)
    try:
        if algo == "nvls" and not w.comms[0].has_multicast:
            pytest.skip("no NVSwitch multicast on this box")
        for mode in ("f32_wire_bf16", "bf16") if algo == "nvls" else MODES:
            for n in (4099, (1 << 20) + 5):
                _check_allreduce(w, n, mode, algo, "randn", seed=n, poke=_sentinel_nans)
    finally:
        w.close()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_messages_larger_than_a_stage_across_devices(world, cuda_count):
    """stage_mb=1: every algorithm has to cut the message into several launches that alternate between the two staging
    buffers while the peers run skewed on real NVLink."""
    devs = devices(world, cuda_count, spread=True)
    w = World(devs, stage_mb=1)
    try:
        for c in w.comms:
            c.set_param("pipe_chunk_bytes", 32 << 10)
        algos = ["twoshot", "twoshot_pipe", "twoshot_ll", "oneshot"] + (["nvls"] if w.comms[0].has_multicast else [])
        for algo in algos:
            before = w.comms[0].launches
            _check_allreduce(w, (3 << 20) + 17, "f32_wire_bf16", algo, "special", seed=5)
            assert w.comms[0].launches - before >= 3, algo
            _check_allreduce(w, (1 << 20) + 9, "f32" if algo != "nvls" else "bf16", algo, "randn", seed=6)
    finally:
        w.close()
