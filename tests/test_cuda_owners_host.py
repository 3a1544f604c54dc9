"""CPU tests of the CUDA owners (genedex_b200/csrc/cuda_owners.h), built on the host with g++ against stub runtime
functions (tests/host_emul/cuda_owners_emul.cpp) that count live device blocks, pinned blocks, events, streams and
stream-ordered blocks and can fail on request.  No GPU and no CUDA runtime library are used here."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
DEV, PINNED, EVENT, STREAM, ASYNC = range(5)
OOM = 2  # cudaErrorMemoryAllocation
NEVER = 2 ** 64 - 1
OWNERS = ("dev", "pinned", "async", "event", "stream")


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul_cuda_owners") / "libcudaowners.so"
    # -Bsymbolic: the owners call the stubs here even when a CUDA runtime is already loaded into the process
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-shared", "-fPIC", "-Wl,-Bsymbolic",
                           "-I" + CUDA_INCLUDE, "-o", str(out), os.path.join(ROOT, "tests", "host_emul", "cuda_owners_emul.cpp")])
    lib = C.CDLL(str(out))
    vp, u64 = C.c_void_p, C.c_uint64
    sig = {"emul_reset": (None, [u64, u64]), "emul_live": (u64, [C.c_int]), "emul_bad_frees": (u64, []),
           "emul_sizes": (u64, [C.POINTER(u64), u64]), "emul_async_frees": (u64, [C.POINTER(vp), u64]),
           "emul_cuda_free": (C.c_int, [vp]),
           "dev_alloc": (C.c_int, [vp, u64]), "dev_reserve": (C.c_int, [vp, u64]), "dev_reset": (None, [vp]),
           "dev_release": (vp, [vp]), "dev_ptr": (vp, [vp]), "dev_bytes": (u64, [vp]), "dev_adopt": (vp, [vp, u64]),
           "pinned_alloc": (C.c_int, [vp, u64]), "pinned_reserve": (C.c_int, [vp, u64]), "pinned_ptr": (vp, [vp]),
           "pinned_bytes": (u64, [vp]),
           "async_alloc": (C.c_int, [vp, u64, vp]), "async_free": (C.c_int, [vp]), "async_ptr": (vp, [vp]),
           "event_create": (C.c_int, [vp]), "event_handle": (vp, [vp]),
           "stream_create": (C.c_int, [vp]), "stream_handle": (vp, [vp])}
    for name in OWNERS:
        sig[name + "_new"] = (vp, [])
        sig[name + "_delete"] = (None, [vp])
        sig[name + "_move_new"] = (vp, [vp])
        sig[name + "_move_assign"] = (None, [vp, vp])
    for name, (res, args) in sig.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib


@pytest.fixture
def emul(lib):
    lib.emul_reset(0, NEVER)
    yield lib
    assert [lib.emul_live(k) for k in range(5)] == [0] * 5, "a resource outlived its owner"
    assert lib.emul_bad_frees() == 0, "a resource was freed twice, on the wrong stream or was never allocated"


def sizes(lib):
    buf = (C.c_uint64 * 64)()
    n = lib.emul_sizes(buf, 64)
    return list(buf[:n])


def round_up(v, a):
    return (v + a - 1) // a * a


def acquire(lib, kind, o, stream=None):
    """one resource into the owner o of this kind"""
    if kind == "dev":
        return lib.dev_alloc(o, 100)
    if kind == "pinned":
        return lib.pinned_alloc(o, 100)
    if kind == "async":
        return lib.async_alloc(o, 100, stream)
    return getattr(lib, kind + "_create")(o)


LIVE = {"dev": DEV, "pinned": PINNED, "async": ASYNC, "event": EVENT, "stream": STREAM}


@pytest.mark.parametrize("kind", OWNERS)
def test_destruction_move_and_reassignment_leave_nothing(emul, kind):
    lib, live = emul, LIVE[kind]
    new, delete = getattr(lib, kind + "_new"), getattr(lib, kind + "_delete")
    a = new()
    delete(a)  # an empty owner frees nothing
    a = new()
    assert acquire(lib, kind, a, 0x51) == 0 and lib.emul_live(live) == 1
    b = getattr(lib, kind + "_move_new")(a)  # moved: one owner, one resource
    delete(a)
    assert lib.emul_live(live) == 1
    c = new()
    assert acquire(lib, kind, c, 0x51) == 0 and lib.emul_live(live) == 2
    getattr(lib, kind + "_move_assign")(b, c)  # b takes c's resource; b's old one is freed by c at the latest
    delete(c)
    assert lib.emul_live(live) == 1
    getattr(lib, kind + "_move_assign")(b, b)  # self-assignment keeps the resource
    assert lib.emul_live(live) == 1
    assert acquire(lib, kind, b, 0x51) == 0  # a new resource in place of the old one
    assert lib.emul_live(live) == 1
    delete(b)
    assert lib.emul_live(live) == 0


@pytest.mark.parametrize("kind", OWNERS)
def test_failed_creation_leaves_an_empty_owner(emul, kind):
    lib, live = emul, LIVE[kind]
    o = getattr(lib, kind + "_new")()
    assert acquire(lib, kind, o, 0x51) == 0
    lib.emul_reset(1, NEVER)  # the next acquiring call fails (and writes garbage into the handle)
    assert acquire(lib, kind, o, 0x51) == OOM
    assert lib.emul_live(live) == 0  # the old resource went first
    getattr(lib, kind + "_delete")(o)  # frees nothing, in particular not the garbage


def test_dev_alloc_of_zero_bytes_is_one_byte(emul):
    o = emul.dev_new()
    assert emul.dev_alloc(o, 0) == 0 and emul.dev_ptr(o) and emul.dev_bytes(o) == 0
    assert sizes(emul) == [1]
    emul.dev_delete(o)


def test_dev_reserve_policy(emul):
    lib = emul
    o = lib.dev_new()
    assert lib.dev_reserve(o, 0) == 0 and not lib.dev_ptr(o) and sizes(lib) == []  # capacity 0 is enough
    # first growth: 1/8 more, rounded to 256
    assert lib.dev_reserve(o, 1000) == 0
    want = round_up(1000 + 1000 // 8, 256)
    assert sizes(lib) == [want] and lib.dev_bytes(o) == want and lib.emul_live(DEV) == 1
    # within the capacity nothing happens
    lib.emul_reset(0, NEVER)
    for n in (1, 1000, want):
        assert lib.dev_reserve(o, n) == 0
    assert sizes(lib) == [] and lib.dev_bytes(o) == want
    # growth frees the old block before the new one is asked for
    lib.emul_reset(1, NEVER)  # the first try fails ...
    n = 10_000
    assert lib.dev_reserve(o, n) == 0  # ... and the exact rounded size is taken
    assert sizes(lib) == [round_up(n + n // 8, 256), round_up(n, 256)]
    assert lib.dev_bytes(o) == round_up(n, 256) and lib.emul_live(DEV) == 1
    # a size limit between the exact and the grown size: the exact retry fits
    lib.emul_reset(0, round_up(20_000, 256))
    assert lib.dev_reserve(o, 20_000) == 0
    assert sizes(lib) == [round_up(20_000 + 2500, 256), round_up(20_000, 256)] and lib.emul_live(DEV) == 1
    # both tries fail: the owner is left empty, with its old block freed
    lib.emul_reset(0, 1 << 20)
    assert lib.dev_reserve(o, 2 << 20) == OOM
    assert sizes(lib) == [round_up((2 << 20) * 9 // 8, 256), 2 << 20]
    assert not lib.dev_ptr(o) and lib.dev_bytes(o) == 0 and lib.emul_live(DEV) == 0
    # and grows again from nothing
    lib.emul_reset(0, NEVER)
    assert lib.dev_reserve(o, 300) == 0 and lib.dev_bytes(o) == round_up(300 + 37, 256)
    lib.dev_delete(o)


def test_pinned_reserve_policy(emul):
    lib = emul
    o = lib.pinned_new()
    assert lib.pinned_reserve(o, 5000) == 0
    want = round_up(5000 + 625, 4096)
    assert sizes(lib) == [want] and lib.pinned_bytes(o) == want
    lib.emul_reset(0, NEVER)
    assert lib.pinned_reserve(o, want) == 0 and sizes(lib) == []
    lib.emul_reset(1, NEVER)  # no exact-size retry for pinned buffers: the owner is left empty
    assert lib.pinned_reserve(o, want + 1) == OOM
    assert sizes(lib) == [round_up((want + 1) * 9 // 8, 4096)]
    assert not lib.pinned_ptr(o) and lib.pinned_bytes(o) == 0 and lib.emul_live(PINNED) == 0
    lib.pinned_delete(o)


def test_dev_release_and_adopt(emul):
    lib = emul
    o = lib.dev_new()
    assert lib.dev_alloc(o, 64) == 0
    p = lib.dev_release(o)
    assert p and not lib.dev_ptr(o) and lib.dev_bytes(o) == 0
    lib.dev_delete(o)
    assert lib.emul_live(DEV) == 1  # the block now belongs to whoever took it
    a = lib.dev_adopt(p, 64)
    assert lib.dev_bytes(a) == 64
    lib.dev_delete(a)
    assert lib.emul_live(DEV) == 0


def async_frees(lib):
    buf = (C.c_void_p * 16)()
    n = lib.emul_async_frees(buf, 16)
    return [buf[i] for i in range(n)]


def test_async_block_is_freed_once_on_its_stream(emul):
    lib = emul
    # on the success path: the explicit free reports cudaFreeAsync's result, the owner frees nothing more
    o = lib.async_new()
    assert lib.async_alloc(o, 4096, 0x51) == 0 and lib.emul_live(ASYNC) == 1
    assert lib.async_free(o) == 0 and lib.emul_live(ASYNC) == 0
    assert lib.async_free(o) == 0  # nothing left to free
    lib.async_delete(o)
    assert async_frees(lib) == [0x51]
    # on an error path: the destructor frees it on the stream it came from
    lib.emul_reset(0, NEVER)
    o = lib.async_new()
    assert lib.async_alloc(o, 4096, 0x52) == 0
    lib.async_delete(o)
    assert async_frees(lib) == [0x52] and lib.emul_live(ASYNC) == 0
    # a second block in the same owner: the first goes back on its own stream
    lib.emul_reset(0, NEVER)
    o = lib.async_new()
    assert lib.async_alloc(o, 16, 0x53) == 0 and lib.async_alloc(o, 16, 0x54) == 0
    assert lib.emul_live(ASYNC) == 1
    lib.async_delete(o)
    assert async_frees(lib) == [0x53, 0x54]
    # a failed allocation leaves nothing to free: the second of two blocks fails, the first is still freed
    lib.emul_reset(2, NEVER)
    rows, big = lib.async_new(), lib.async_new()
    assert lib.async_alloc(rows, 8, 0x55) == 0
    assert lib.async_alloc(big, 2 ** 61, 0x55) == OOM and not lib.async_ptr(big)
    lib.async_delete(big)
    lib.async_delete(rows)
    assert async_frees(lib) == [0x55]
    # moved: freed once, by the new owner
    lib.emul_reset(0, NEVER)
    a = lib.async_new()
    assert lib.async_alloc(a, 16, 0x56) == 0
    b = lib.async_move_new(a)
    lib.async_delete(a)
    assert async_frees(lib) == []
    lib.async_delete(b)
    assert async_frees(lib) == [0x56]
