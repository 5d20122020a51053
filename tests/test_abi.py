"""The C-ABI library loads and exports every symbol include/b200ddp.h declares (no compute calls: no GPU here)."""
import ctypes
import os
import re

from torchx_b200.ddp import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "b200ddp.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_list_the_same_symbols():
    assert _declared() == sorted(N.SYMBOLS)


def test_library_exports_every_declared_symbol():
    N.build_library()
    L = ctypes.CDLL(N.LIB_PATH)
    for s in _declared():
        assert hasattr(L, s), s
    assert N.lib().b2_version() == N.B2_ABI_VERSION


def test_plain_c_consumer_builds_against_the_header_and_resolves_every_symbol(tmp_path):
    """The boundary is a C ABI: strict C99 (-pedantic, no C++), no torch anywhere - `gcc` + `dlopen` is all a host needs."""
    import subprocess

    N.build_library()
    exe = tmp_path / "consumer"
    syms = ", ".join(f'"{s}"' for s in _declared())
    cmd = ["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", f"-I{os.path.join(ROOT, 'include')}", f"-DB2_CONSUMER_SYMBOLS={syms}",
           os.path.join(ROOT, "tests", "abi", "consumer.c"), "-o", str(exe), "-ldl"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    res = subprocess.run([str(exe), N.LIB_PATH], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert res.stdout.strip() == f"ok {len(_declared())} symbols abi {N.B2_ABI_VERSION}"
    for binary in (str(exe), N.LIB_PATH):  # neither the consumer nor the library itself links torch or python (cudart is static)
        ldd = subprocess.run(["ldd", binary], capture_output=True, text=True).stdout
        assert "torch" not in ldd and "python" not in ldd, ldd


def test_header_constants_match_binding():
    src = open(os.path.join(ROOT, "include", "b200ddp.h")).read()
    for name in ("B2_OK", "B2_EINVAL", "B2_ECUDA", "B2_ESYS", "B2_ETIMEOUT", "B2_ENOPEER", "B2_ESTATE", "B2_F32_WIRE_BF16",
                 "B2_F32", "B2_BF16", "B2_ALGO_AUTO", "B2_ALGO_ONESHOT", "B2_ALGO_TWOSHOT", "B2_ALGO_TWOSHOT_PIPE", "B2_ALGO_NVLS", "B2_ALGO_TWOSHOT_LL", "B2_ENOTSUP", "B2_CAP_VMM", "B2_CAP_MULTICAST", "B2_ABI_VERSION", "B2_MAX_WORLD", "B2_MAX_SEGMENTS"):
        m = re.search(rf"#define\s+{name}\s+\(?(-?\d+)\)?", src)
        assert m, name
        assert int(m.group(1)) == getattr(N, name), name


def test_argument_validation_without_a_gpu():
    L = N.lib()
    out = ctypes.c_void_p()
    assert L.b2_comm_create(ctypes.byref(out), 3, 2, 0, b"/x", 0, 0, 10) == N.B2_EINVAL
    assert b"bad arguments" in L.b2_last_error()
    assert L.b2_allreduce(None, None, 8, 0, 1.0, 0, None) == N.B2_EINVAL
    assert L.b2_comm_status(None) == N.B2_EINVAL
    assert L.b2_comm_destroy(None) == N.B2_OK
    # the gather variant validates its segment table on the host before anything is launched
    segs = (N.B2Segment * 2)()
    segs[0].src, segs[0].begin, segs[0].end = 4096, 0, 10
    segs[1].src, segs[1].begin, segs[1].end = 8192, 12, 20  # gap: does not continue at element 10
    assert L.b2_allreduce_gather(None, ctypes.c_void_p(4096), 20, segs, 2, 0, 1.0, 0, None) == N.B2_EINVAL
    assert b"does not continue" in L.b2_last_error()
    assert L.b2_allreduce_gather(None, ctypes.c_void_p(4096), 20, segs, N.B2_MAX_SEGMENTS + 1, 0, 1.0, 0, None) == N.B2_EINVAL
    assert b"need 1..128 segments (got 129)" in L.b2_last_error()
    assert L.b2_comm_caps(None) == N.B2_EINVAL and L.b2_comm_last_algo(None) == N.B2_EINVAL
    assert L.b2_comm_set_param(None, b"max_ctas", 1) == N.B2_EINVAL


def _gather_table_error(table, n_elems, n_segments=None):
    """Return code and b2_last_error() of a gather call with this (src, begin, end) table; a null communicator, so the
    call can only get as far as the host-side validation of the table."""
    L = N.lib()
    segs = (N.B2Segment * max(1, len(table)))()
    for i, (src, begin, end) in enumerate(table):
        segs[i].src, segs[i].begin, segs[i].end = src, begin, end
    n = len(table) if n_segments is None else n_segments
    rc = L.b2_allreduce_gather(None, ctypes.c_void_p(4096), n_elems, segs, n, 0, 1.0, 0, None)
    return rc, L.b2_last_error().decode()


def test_gather_segment_table_validation_without_a_gpu():
    ok = [(4096, 0, 10), (8192, 10, 20)]
    assert _gather_table_error(ok, 20) == (N.B2_EINVAL, "null communicator")  # the table itself passes
    cases = [
        ([(4096, 0, 10), (8192, 10, 10), (8192, 10, 20)], 20, "segment 1 is empty"),
        ([(4096, 0, 0), (8192, 0, 20)], 20, "segment 0 is empty"),
        ([(4096, 0, 10), (None, 10, 20)], 20, "segment 1 has a null src"),
        ([(4096, 0, 10), (8192, 10, 20)], 21, "segments cover 20 elements, bucket has 21"),
        ([(4096, 0, 10), (8192, 10, 20)], 19, "segments cover 20 elements, bucket has 19"),
        ([(4096, 0, 10), (8192, 9, 20)], 20, "segment 1 does not continue the bucket at element 10"),
        ([(4096, 1, 10)], 9, "segment 0 does not continue the bucket at element 0"),
    ]
    for table, n_elems, msg in cases:
        assert _gather_table_error(table, n_elems) == (N.B2_EINVAL, f"b2_allreduce_gather: {msg}"), (table, n_elems)
    assert _gather_table_error(ok, 20, n_segments=0) == (N.B2_EINVAL, "b2_allreduce_gather: need 1..128 segments (got 0)")
    L = N.lib()
    assert L.b2_allreduce_gather(None, ctypes.c_void_p(4096), 20, None, 2, 0, 1.0, 0, None) == N.B2_EINVAL  # NULL table
    assert L.b2_last_error() == b"b2_allreduce_gather: null segment table"
