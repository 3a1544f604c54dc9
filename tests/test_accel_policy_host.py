"""CPU tests of the accelerator policy (genedex_b200/csrc/accel_policy.h), built on the host with g++.
The model is a plain transcription of the decisions api.cu made inline before the policy moved into the header
(auto_dense_sa, auto_seed_table, auto_row_context, row_context_possible and the GDX_VERIFY_MIN handling); the header
must decide the same for every input.  No GPU is used here."""
import ctypes as C
import os
import random
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNKNOWN = 2 ** 64 - 1  # free device memory could not be observed
NO_DENSE_SA, NO_SEED_TABLE, NO_ROW_CONTEXT = 1, 2, 4
ENVS = [None, "0", "1", "7", "abc"]


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul_accel_policy") / "libaccelpolicy.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(ROOT, "tests", "host_emul", "accel_policy_emul.cpp")])
    lib = C.CDLL(str(out))
    lib.emul_accel_policy.restype = None
    lib.emul_accel_policy.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_uint32,
                                      C.c_uint64, C.c_uint64, C.c_char_p, C.c_char_p, C.c_char_p,
                                      np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")]
    lib.emul_seed_entries.restype = C.c_uint64
    lib.emul_seed_entries.argtypes = [C.c_uint32, C.c_uint32]
    lib.emul_verify_min_remaining.restype = C.c_uint32
    lib.emul_verify_min_remaining.argtypes = [C.c_int, C.c_char_p]
    return lib


def atoi(s):
    m = re.match(r"\s*([+-]?\d+)", s)
    return int(m.group(1)) if m else 0


def seed_entries(ns, d):
    e = 1
    for _ in range(d):
        e *= ns
        if e > 1 << 36:
            return 0
    return e


class Case:
    def __init__(self, n, budget, ns, lookup_depth, wide, text, flags, used, free, env):
        self.n, self.budget, self.ns, self.lookup_depth = n, budget, ns, lookup_depth
        self.wide, self.text, self.flags, self.used, self.free, self.env = wide, text, flags, used, free, env

    def accel_room(self):
        if self.budget:
            return self.budget - self.used if self.budget > self.used else 0
        if self.free == UNKNOWN:
            return 0
        return self.free // 4

    def auto_dense_sa(self):
        e = self.env
        if self.n == 0:
            return False
        if e is not None and atoi(e) == 0:
            return False
        if not (e is not None and atoi(e) != 0):
            if self.flags & NO_DENSE_SA:
                return False
            if self.n * (8 if self.wide else 4) > self.accel_room():
                return False
        return True

    def auto_seed_table(self):
        e = self.env
        if self.n == 0 or self.ns < 2:
            return 0
        depth = 0
        if e is not None:
            if atoi(e) <= 0:
                return 0
            depth = atoi(e)
        else:
            if self.flags & NO_SEED_TABLE:
                return 0
            while seed_entries(self.ns, depth + 1) and seed_entries(self.ns, depth + 1) <= 4 * self.n:
                depth += 1
            esz, room = (16 if self.wide else 8), self.accel_room()
            if self.free == UNKNOWN:
                return 0
            while depth > 0 and (seed_entries(self.ns, depth) * esz > room or
                                 (seed_entries(self.ns, depth) + seed_entries(self.ns, depth - 1)) * esz > self.free):
                depth -= 1
        if depth <= self.lookup_depth:
            return 0
        return depth

    def row_context_possible(self):
        return self.n > 0 and not self.wide and self.n < 1 << 32 and 1 <= self.ns <= 4 and self.text

    def auto_row_context(self):
        e = self.env
        if not self.row_context_possible():
            return False
        if e is not None and atoi(e) == 0:
            return False
        if not (e is not None and atoi(e) != 0):
            if self.flags & NO_ROW_CONTEXT:
                return False
            room = self.accel_room() if self.budget else 2 * self.accel_room()
            if self.n * 16 > room:
                return False
        return True


def run_header(lib, c):
    out = np.zeros(4, dtype=np.uint64)
    env = None if c.env is None else c.env.encode()
    lib.emul_accel_policy(c.n, c.budget, c.ns, c.lookup_depth, int(c.wide), int(c.text), c.flags, c.used, c.free,
                          env, env, env, out)
    return bool(out[0]), int(out[1]), bool(out[2]), bool(out[3])


def near(rng, x):
    """a value at, just below or just above x, or anywhere below 4x"""
    return max(0, rng.choice([x, x - 1, x + 1, rng.randrange(4 * x + 1)]))


def random_case(rng):
    n = rng.choice([0, 1, rng.randrange(2, 100), rng.randrange(100, 100_000), rng.randrange(1 << 20, 1 << 33),
                    rng.randrange(1 << 31, 1 << 34)])
    ns = rng.choice([1, 2, 3, 4, 5, 20, rng.randrange(1, 256), 255])
    wide = rng.random() < 0.3 or n > 0xFFFFFFFF
    esz = 8 if wide else 4
    # sizes the decisions compare against, so that budgets and free memory land on both sides of them
    pivots = [n * esz, n * 16, 4 * n * 16, max(1, seed_entries(ns, rng.randrange(0, 20))) * 2 * esz]
    budget = 0 if rng.random() < 0.5 else near(rng, rng.choice(pivots)) + rng.choice([0, 0, 1 << rng.randrange(40)])
    used = rng.choice([0, 0, rng.randrange(0, 1 << 34), budget, near(rng, budget)])
    free = rng.choice([UNKNOWN, 0, near(rng, 4 * rng.choice(pivots)), near(rng, rng.choice(pivots)),
                       rng.randrange(1 << 38)])
    return Case(n, budget, ns, rng.choice([0, 0, 1, 2, 5, rng.randrange(0, 25)]), wide, rng.random() < 0.8,
                rng.randrange(8), used, free, rng.choice(ENVS))


def test_policy_matches_the_former_inline_decisions(lib):
    rng = random.Random(11)
    seen = set()
    for i in range(40_000):
        c = random_case(rng)
        want = (c.auto_dense_sa(), c.auto_seed_table(), c.auto_row_context(), c.row_context_possible())
        assert run_header(lib, c) == want, vars(c)
        seen.add((want[0], want[1] > 0, want[2], c.env, c.budget > 0, c.free == UNKNOWN))
    # every decision was taken both ways, under every override, with and without a budget and free-memory reading
    for env in ENVS:
        for budget in (False, True):
            assert any(s[3] == env and s[4] == budget and s[0] for s in seen) or env in ("0", "abc")
            assert any(s[3] == env and s[4] == budget and not s[0] for s in seen)
    assert any(s[1] and s[5] is False for s in seen) and any(s[2] and s[3] is None for s in seen)
    assert any(s[0] and s[3] is None and s[5] for s in seen)  # a budget decides without a free-memory reading


@pytest.mark.parametrize("ns,n", [(4, 40_000), (4, 3_100_000_000), (20, 500_000_000), (5, 1000), (2, 1), (255, 10)])
def test_automatic_seed_depth_is_the_deepest_with_four_entries_per_position(lib, ns, n):
    c = Case(n, 0, ns, 0, False, True, 0, 0, 1 << 50, None)
    d = run_header(lib, c)[1]
    assert d == c.auto_seed_table()
    if d:
        assert ns ** d <= 4 * n < ns ** (d + 1)
    if (ns, n) == (4, 3_100_000_000):
        assert d == 16  # the headline DNA index
    if (ns, n) == (20, 500_000_000):
        assert d == 7


def test_seed_entries(lib):
    for ns in range(1, 256):
        for d in range(0, 41):
            assert lib.emul_seed_entries(ns, d) == seed_entries(ns, d)


@pytest.mark.parametrize("env", ENVS + ["-3", " 12", "5x"])
def test_verify_min_remaining(lib, env):
    for dense in (False, True):
        want = 8
        if env is not None and atoi(env) > 0:
            want = atoi(env)
        if dense and env is None:
            want = 4
        assert lib.emul_verify_min_remaining(int(dense), None if env is None else env.encode()) == want
