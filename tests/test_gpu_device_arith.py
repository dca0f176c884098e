"""Device arithmetic on the B200, through tests/device/arith_harness.cu: the headers of csrc/ compiled for sm_100a with the library's
nvcc flags and called the way the kernels call them.
  * TestHostEmuCasesOnDevice runs the cases of tests/test_host_emu.py a second time, on the GPU: the same inputs and expectations,
    one item per launch, Fp products through the __noinline__ calls fp_mul_call / fp_sqr_call / fp_mul2_call;
  * the warp-cooperative Fp arithmetic of csrc/g1_coop.cuh (one element on four lanes): the raw semi-reduced lanes of every result
    against the limb-exact model of tests/test_coop_model.py, and the canonical value against Python integers -- on edge values,
    values in [p, 2p), lane patterns, the operand pairs whose final carry fold takes a second and a third pass, and neighbouring
    groups of a warp whose carries at the group edges disagree (the ballots of `resolve` are warp-wide);
  * the cooperative point formulas and the fixed-scalar ladder against oracle/pyref.py and the one-thread ladder;
  * every program of the Fp interpreter run over fpvm::Smem, the shared-memory slots of the hot kernels, against
    tools/fpvm_asm.emulate.
The tests without the gpu mark check, on any machine, that the harness compiles for sm_100a and that the inputs reach the cases
named above."""
import ctypes
import functools
import os
import random
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from oracle import pyref
from tests import test_coop_model as CM
from tests import test_host_emu as HE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rust-eth-kzg_b200", "csrc")
P, R = pyref.P, pyref.R
RM = 1 << 384
RINV = pow(RM, -1, P)
MONT_ONE = RM % P
M96 = (1 << 96) - 1


# ---- the harness ----------------------------------------------------------------------------------------------------------------
def _nvcc():
    cand = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else None


def build_device_harness():
    """tests/device/arith_harness.cu -> .so with the flags of the library's objects (rust-eth-kzg_b200/Makefile NVCCFLAGS), rebuilt
    when it or a header of csrc/ is newer; next to the source, or in a per-user temporary directory when the tree is read-only.
    None without nvcc."""
    nvcc = _nvcc()
    if nvcc is None:
        return None
    src = os.path.join(ROOT, "tests", "device", "arith_harness.cu")
    outdir = os.path.dirname(src)
    if not os.access(outdir, os.W_OK):
        outdir = os.path.join(tempfile.gettempdir(), "ekzg_arith_harness_%d" % os.getuid())
        os.makedirs(outdir, exist_ok=True)
    out = os.path.join(outdir, "arith_harness.so")
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".inc"))]
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I" + CSRC, "-diag-suppress", "550",
                               "-Xcompiler", "-fPIC", "-shared", "-o", out, src])
    return out


class DeviceHarness:
    """the harness with the CUDA status checked after every call: a failed call fails the test once, with the error's name, and
    the harness launches nothing after it"""

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        self.lib.harness_error_name.restype = ctypes.c_char_p

    def __getattr__(self, name):
        fn = getattr(self.lib, name)

        def call(*args):
            r = fn(*args)
            err = self.lib.harness_error()
            if err:
                pytest.fail("%s: CUDA error %s" % (name, self.lib.harness_error_name(err).decode()), pytrace=False)
            return r
        self.__dict__[name] = call
        return call


_device = []


def device_harness():
    """the built harness on the GPU (skips without one); one instance per process"""
    if not _device:
        path = build_device_harness()
        if path is None:
            pytest.skip("no nvcc")
        lib = DeviceHarness(path)
        if lib.lib.harness_device_count() < 1:
            pytest.skip("no CUDA device")
        _device.append(lib)
    return _device[0]


class TestHostEmuCasesOnDevice:
    """every case of tests/test_host_emu.py whose code runs on the device, run a second time on the GPU with the same inputs and
    expectations (emu_set_window is host-side table arithmetic; the interpreter and the G1-NTT units have their own device tests)"""
    pytestmark = pytest.mark.gpu

    @pytest.fixture
    def emu_field(self):
        return device_harness()

    @pytest.fixture
    def emu_g1(self):
        return device_harness()

    test_field_ops = staticmethod(HE.test_field_ops)
    test_field_mul_adversarial_limbs = staticmethod(HE.test_field_mul_adversarial_limbs)
    test_fp_inversion_by_division_steps = staticmethod(HE.test_fp_inversion_by_division_steps)
    test_g1_compress_roundtrip = staticmethod(HE.test_g1_compress_roundtrip)
    test_g1_binops = staticmethod(HE.test_g1_binops)
    test_g1_chains = staticmethod(HE.test_g1_chains)
    test_g1_scalar_mul = staticmethod(HE.test_g1_scalar_mul)
    test_subgroup_check_matches_naive = staticmethod(HE.test_subgroup_check_matches_naive)
    test_booth_digits = staticmethod(HE.test_booth_digits)


def limbs(x, n=12):
    return [(x >> (32 * i)) & 0xFFFFFFFF for i in range(n)]


def value(ws):
    return sum(int(w) << (32 * i) for i, w in enumerate(ws))


def flat(lanes):
    return [w for lane in lanes for w in lane]


def u32(rows, width):
    return np.ascontiguousarray(np.array(rows, dtype=np.uint32).reshape(-1, width))


def ptr(a, ctype=ctypes.c_uint32):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


@pytest.fixture(scope="module")
def dev():
    return device_harness()


# ---- inputs --------------------------------------------------------------------------------------------------------------------
def fold_passes(a, b):
    """(result lanes, passes of the final carry fold) of the model's cmul (tests/test_coop_model.py), its rows restated from the
    model's own pieces so that the fold can be counted; the result is checked against CM.cmul wherever this is used"""
    a, b = CM.lanes(a), CM.lanes(b)
    T = [[0] * 5 for _ in range(4)]
    ypend = [0] * 4
    for i in range(12):
        bi = b[i // 3][i % 3]
        for l in range(4):
            CM.mad3(T[l], a[l], bi)
        m = (T[0][0] * CM.M0) & CM.W
        for l in range(4):
            acc = T[l][2] + (T[l][3] << 32) + (T[l][4] << 64) + ypend[l]
            T[l][2], T[l][3], T[l][4] = acc & CM.W, (acc >> 32) & CM.W, (acc >> 64) & CM.W
        for l in range(4):
            CM.mad3(T[l], CM.P_L[l], m)
        ypend = [T[l + 1][0] if l < 3 else 0 for l in range(4)]
        for l in range(4):
            T[l] = [T[l][1], T[l][2], T[l][3], T[l][4], 0]
    for l in range(4):
        acc = T[l][2] + (T[l][3] << 32) + ypend[l]
        T[l][2], T[l][3] = acc & CM.W, acc >> 32
    passes = 0
    while True:
        cin = [0] + [T[l][3] for l in range(3)]
        for l in range(4):
            acc = T[l][0] + (T[l][1] << 32) + (T[l][2] << 64) + cin[l]
            T[l][0], T[l][1], T[l][2], T[l][3] = acc & CM.W, (acc >> 32) & CM.W, (acc >> 64) & CM.W, acc >> 96
        passes += 1
        if not any(T[l][3] for l in range(4)):
            return [T[l][:3] for l in range(4)], passes


@functools.lru_cache(maxsize=None)
def fold_cases():
    """operand pairs whose cmul takes more than one pass of the final carry fold, found with the model: every a whose lanes are
    all-ones, zero, one or the top bit, against Montgomery 1 and 2 and 1 + p, in both orders.  Random operands fold in one pass.
    Returns {passes: [(a, b), ...]}; three is the most there can be: a carry crosses at most three lane boundaries."""
    found = {}
    pats = [0, M96, 1, 1 << 95]
    for k in range(4 ** 4):
        a = sum(pats[(k >> (2 * l)) & 3] << (96 * l) for l in range(4))
        if a >= 2 * P:
            continue
        for b in (MONT_ONE, 2 * MONT_ONE % P, MONT_ONE + P):
            for x, y in ((a, b), (b, a)):
                n = fold_passes(x, y)[1]
                if n > 1:
                    found.setdefault(n, []).append((x, y))
    return found


@functools.lru_cache(maxsize=None)
def values():
    """semi-reduced operands: the model's edge values, values in [p, 2p), random values and lane patterns"""
    rng = random.Random(21)
    vals = [e for e in CM.EDGE if e < 2 * P]
    vals += [P + rng.randrange(P) for _ in range(8)] + [rng.randrange(2 * P) for _ in range(16)]
    while len(vals) < 48:
        v = sum(rng.choice([0, M96, 1 << 95, rng.randrange(1 << 96)]) << (96 * l) for l in range(4))
        if v < 2 * P:
            vals.append(v)
    return vals


def _lane(x, l):
    return (x >> (96 * l)) & M96


def _votes(op, a, b):
    """(generate, propagate) lane votes of each ballot round of cadd / csub (cneg = csub(0, a)) on (a, b), from the model"""
    def add(x, y):
        s = [_lane(x, l) + _lane(y, l) for l in range(4)]
        return [v >> 96 for v in s], [int(v == M96) for v in s]

    def sub(x, y):
        d = [_lane(x, l) - _lane(y, l) for l in range(4)]
        return [int(v < 0) for v in d], [int(v == 0) for v in d]
    if op == "cadd":
        s = CM.value(CM.add_raw(CM.lanes(a), CM.lanes(b))[0])
        return [add(a, b), sub(s, 2 * P)]
    d, below = CM.sub_raw(CM.lanes(a), CM.lanes(b))
    return [sub(a, b), add(CM.value(d), 2 * P if below else 0)]


def edge_disagreements(op, pairs):
    """{(vote, top)}: the ways in which, somewhere in the batch, group g's top lane votes `top` while group g + 1 of the same warp
    votes the opposite in its lane 0, in one ballot round (vote 0 = generate, 1 = propagate)"""
    seen = set()
    vs = [_votes(op, a, b) for a, b in pairs]
    for g in range(len(pairs) - 1):
        if g % 8 == 7:
            continue    # g + 1 starts the next warp
        for r in range(2):
            for k in range(2):
                top, low = vs[g][r][k][3], vs[g + 1][r][k][0]
                if top != low:
                    seen.add((k, top))
    return seen


@functools.lru_cache(maxsize=None)
def add_sub_batch(op):
    """operand pairs for cadd / csub / cneg (b ignored): first adjacent pairs whose carries at the group edges disagree in every
    way (generate and propagate, top lane set and lane 0 clear and the reverse), then all pairs of values(); length not a multiple
    of eight, so the last warp is padded"""
    vals = values()
    two_p = 2 * P
    pool = [(a, b) for a in vals for b in vals]
    for a in vals:     # equal lanes (propagate in the subtraction), sums at 2p and at all-ones lanes
        pool += [(a, a ^ 1), (a, a ^ (1 << 300)), (a, (a & ~M96) | (M96 - _lane(a, 0)))]
        pool += [(a, two_p - a - 1)] + ([(a, two_p - a + (1 << 96))] if a > 1 << 96 else [])
    pool = [(a, b) for a, b in pool if a < two_p and b < two_p]
    if op == "cneg":
        pool = [(0, a) for a in vals]
    vs = [_votes("csub" if op == "cneg" else op, a, b) for a, b in pool]
    lead = []
    for k in range(2):
        for top in range(2):
            for r in range(2):
                i = next((i for i in range(len(pool)) if vs[i][r][k][3] == top), None)
                j = next((j for j in range(len(pool)) if vs[j][r][k][0] == 1 - top), None)
                if i is not None and j is not None:
                    lead += [pool[i], pool[j]]
                    break
    rest = [(a, b) for a in vals for b in vals[::5]] if op != "cneg" else pool
    return lead + rest + [(vals[3], vals[5])] * 3


# ---- without a GPU ------------------------------------------------------------------------------------------------------------
def test_harness_compiles_for_sm100a():
    path = build_device_harness()
    if path is None:
        pytest.skip("no nvcc")
    lib = ctypes.CDLL(path)
    for name in ("coop_fp", "coop_pt", "fpvm_smem_run", "harness_error", "emu_fp_mul", "emu_g1_mul_twiddle_ops", "emu_booth_digit"):
        assert hasattr(lib, name), name


def test_fold_cases_reach_second_and_third_pass():
    cases = fold_cases()
    assert len(cases.get(2, [])) >= 4 and len(cases.get(3, [])) >= 2
    assert ((M96 << 192, MONT_ONE) in cases[2]) and ((1 << 288, MONT_ONE) in cases[3])
    assert all(a < 2 * P and b < 2 * P for n in cases for a, b in cases[n])
    assert all(fold_passes(a, b)[0] == CM.cmul(CM.lanes(a), CM.lanes(b)) for n in cases for a, b in cases[n])
    # cmul2: each half of the hard x easy batch is the hard pair somewhere, in both orders
    quads = cmul2_batch()
    for n in (2, 3):
        hard = set(cases[n])
        assert any((a, b) in hard and (c, d) not in hard for a, b, c, d in quads)
        assert any((c, d) in hard and (a, b) not in hard for a, b, c, d in quads)


@pytest.mark.parametrize("op", ["cadd", "csub", "cneg"])
def test_neighbouring_groups_disagree_at_their_edges(op):
    pairs = add_sub_batch(op)
    assert len(pairs) % 8 != 0
    assert edge_disagreements("csub" if op == "cneg" else op, pairs) == {(0, 0), (0, 1), (1, 0), (1, 1)}


# ---- cooperative Fp -----------------------------------------------------------------------------------------------------------
def run_coop_fp(dev, op, a, b=None, c=None, d=None):
    """raw (the lanes' limbs, both results) and canonical values of op on the elements a[i] (b[i], c[i], d[i])"""
    n = len(a)
    ins = [u32([limbs(x) for x in (v if v is not None else [0] * n)], 12) for v in (a, b, c, d)]
    raw, canon = np.zeros((n, 24), np.uint32), np.zeros((n, 24), np.uint32)
    ops = {"cmul": 0, "cmul2": 1, "cadd": 2, "csub": 3, "cneg": 4, "from_fp": 5}
    assert dev.coop_fp(ops[op], n, *[ptr(x) for x in ins], ptr(raw), ptr(canon)) == 0
    return ([(raw[i, :12].tolist(), raw[i, 12:].tolist()) for i in range(n)],
            [(value(canon[i, :12]), value(canon[i, 12:])) for i in range(n)])


def check_semi(raw, canon, want_lanes, want, what):
    assert raw == flat(want_lanes), "%s: raw lanes differ from the model" % what
    assert value(raw) < 2 * P, what
    assert canon == want, "%s: canonical value" % what


@functools.lru_cache(maxsize=None)
def cmul_batch():
    """all pairs of values(), with the multi-pass pairs spread among them: warps that mix hard and easy products"""
    vals = values()
    pairs = [(a, b) for a in vals for b in vals]
    hard = [p for n in sorted(fold_cases()) for p in fold_cases()[n]]
    for i, p in enumerate(hard):
        pairs.insert(37 * i % len(pairs), p)
    return pairs + [hard[0]] * 5


@functools.lru_cache(maxsize=None)
def cmul2_batch():
    """(a1, b1, a2, b2): hard pair with easy pair, easy with hard, hard with hard, and easy pairs"""
    rng = random.Random(22)
    vals = values()
    easy = [(a, b) for a in vals for b in vals[::7]]
    hard = [p for n in sorted(fold_cases()) for p in fold_cases()[n]]
    quads = []
    for h in hard:
        e = rng.choice(easy)
        quads += [h + e, e + h, h + rng.choice(hard)]
    quads += [rng.choice(easy) + rng.choice(easy) for _ in range(200)]
    rng.shuffle(quads)
    return quads + [quads[0]] * 3


@pytest.mark.gpu
def test_coop_mul_matches_model(dev):
    pairs = cmul_batch()
    raws, canons = run_coop_fp(dev, "cmul", [a for a, _ in pairs], [b for _, b in pairs])
    for (a, b), (raw, _), (canon, _) in zip(pairs, raws, canons):
        check_semi(raw, canon, CM.cmul(CM.lanes(a), CM.lanes(b)), a * b * RINV % P, "cmul(%#x, %#x)" % (a, b))


@pytest.mark.gpu
def test_coop_mul2_matches_model(dev):
    quads = cmul2_batch()
    raws, canons = run_coop_fp(dev, "cmul2", *[[q[k] for q in quads] for k in range(4)])
    for (a, b, c, d), (r1, r2), (c1, c2) in zip(quads, raws, canons):
        check_semi(r1, c1, CM.cmul(CM.lanes(a), CM.lanes(b)), a * b * RINV % P, "cmul2 first half (%#x, %#x | %#x, %#x)" % (a, b, c, d))
        check_semi(r2, c2, CM.cmul(CM.lanes(c), CM.lanes(d)), c * d * RINV % P, "cmul2 second half (%#x, %#x | %#x, %#x)" % (a, b, c, d))


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["cadd", "csub", "cneg"])
def test_coop_add_sub_neg_match_model(dev, op):
    pairs = add_sub_batch(op)
    if op == "cneg":
        raws, canons = run_coop_fp(dev, op, [b for _, b in pairs])
    else:
        raws, canons = run_coop_fp(dev, op, [a for a, _ in pairs], [b for _, b in pairs])
    for (a, b), (raw, _), (canon, _) in zip(pairs, raws, canons):
        if op == "cadd":
            want_lanes, want = CM.cadd(CM.lanes(a), CM.lanes(b)), (a + b) % P
        elif op == "csub":
            want_lanes, want = CM.csub(CM.lanes(a), CM.lanes(b)), (a - b) % P
        else:
            want_lanes, want = CM.csub(CM.lanes(0), CM.lanes(b)), -b % P
        check_semi(raw, canon, want_lanes, want, "%s(%#x, %#x)" % (op, a, b))


@pytest.mark.gpu
def test_coop_from_to_fp_round_trip(dev):
    vals = values() + [P - 1, P, 2 * P - 1]
    raws, canons = run_coop_fp(dev, "from_fp", vals)
    for a, (raw, _), (canon, _) in zip(vals, raws, canons):
        check_semi(raw, canon, CM.lanes(a), a % P, "from_fp / to_fp %#x" % a)


# ---- cooperative point formulas and the fixed-scalar ladder ---------------------------------------------------------------------
def _points(rng, n):
    return [pyref.g1_mul(pyref.G1_GEN, rng.randrange(1, R)) for _ in range(n)]


def _jac_mont(pt, z, semi):
    """Jacobian (X, Y, Z) = (x z^2, y z^3, z) in Montgomery form, p added to every coordinate if `semi` ([p, 2p): semi-reduced)"""
    x, y = pt
    return [(c * RM % P) + (P if semi else 0) for c in (x * z * z % P, y * z ** 3 % P, z)]


def _affine(out36):
    """canonical Montgomery Jacobian -> affine point (None for the identity)"""
    X, Y, Z = (value(out36[12 * k:12 * k + 12]) for k in range(3))
    assert max(X, Y, Z) < P
    X, Y, Z = X * RINV % P, Y * RINV % P, Z * RINV % P
    if Z == 0:
        return None
    zi = pow(Z, -1, P)
    return X * zi * zi % P, Y * zi ** 3 % P


def run_coop_pt(dev, op, jac, aff=None, rows=None):
    n = len(jac)
    p = u32([flat([limbs(c) for c in j]) for j in jac], 36)
    q = u32([flat([limbs(c) for c in a]) for a in (aff or [(0, 0)] * n)], 24)
    w = np.ascontiguousarray(np.array(rows or [1] * ((n + 7) // 8), dtype=np.int32))
    out, zr = np.zeros((n, 36), np.uint32), np.zeros((n, 12), np.uint32)
    ops = {"cjac_dbl": 0, "cjac_madd": 1, "cjac_madd_zr": 2, "cjac_mul_ops": 3, "jac_mul_ops": 4}
    assert dev.coop_pt(ops[op], n, ptr(p), ptr(q), ptr(w, ctypes.c_int), ptr(out), ptr(zr)) == 0
    return [out[i].tolist() for i in range(n)], [value(zr[i]) for i in range(n)]


@pytest.mark.gpu
def test_coop_point_formulas(dev):
    rng = random.Random(23)
    n = 43
    qs, gs = _points(rng, n), _points(rng, n)
    zs = [rng.randrange(1, P) for _ in range(n)]
    jac = [_jac_mont(q, z, i % 2) for i, (q, z) in enumerate(zip(qs, zs))]
    aff = [tuple((c * RM % P) + (P if i % 3 == 0 else 0) for c in g) for i, g in enumerate(gs)]
    out, _ = run_coop_pt(dev, "cjac_dbl", jac)
    for i in range(n):
        assert _affine(out[i]) == pyref.g1_add(qs[i], qs[i]), ("cjac_dbl", i)
    out, _ = run_coop_pt(dev, "cjac_madd", jac, aff)
    for i in range(n):
        assert _affine(out[i]) == pyref.g1_add(qs[i], gs[i]), ("cjac_madd", i)
    out, zr = run_coop_pt(dev, "cjac_madd_zr", jac, aff)
    for i in range(n):
        assert _affine(out[i]) == pyref.g1_add(qs[i], gs[i]), ("cjac_madd_zr", i)
        assert zr[i] < P and value(out[i][24:]) * RINV % P == zs[i] * (zr[i] * RINV) % P, ("cjac_madd_zr: Z3 = Z1 zr", i)


@pytest.mark.gpu
def test_coop_mul_ops_every_twiddle_row(dev):
    """cjac_mul_ops for each op list it runs (twiddle rows 1-63 and 65-127; 0 and 64 never reach it), one row per warp on eight
    different points, against k P with Python integers and against the one-thread jac_mul_ops on the device"""
    rng = random.Random(24)
    pts = _points(rng, 8)
    rows = [e for e in range(1, 128) if e != 64]
    jac = [_jac_mont(pts[i], rng.randrange(1, P), i % 2) for _ in rows for i in range(8)]
    coop, _ = run_coop_pt(dev, "cjac_mul_ops", jac, rows=rows)
    one, _ = run_coop_pt(dev, "jac_mul_ops", [[c % P for c in j] for j in jac], rows=rows)
    w128 = pyref.root_of_unity(128)
    for r, e in enumerate(rows):
        k = pow(w128, e, R)
        for i in range(8):
            want = pyref.g1_mul(pts[i], k)
            assert _affine(coop[8 * r + i]) == want, ("cjac_mul_ops", e, i)
            assert _affine(one[8 * r + i]) == want, ("jac_mul_ops", e, i)


# ---- the Fp interpreter over shared memory ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fpvm_programs_over_shared_memory(dev):
    """every program of tools/fpvm_asm.PROGRAMS through fpvm::step on fpvm::Smem: two CTAs of 128 threads, each thread with its own
    eight slots; every eighth thread with the planted equal, zero and p - 1 operands"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import fpvm_asm as A
    assert dev.fpvm_words() == sum(len(p) for p in A.PROGRAMS.values())
    rng = random.Random(25)
    nt = 256
    pc = 0
    for name, prog in A.PROGRAMS.items():
        vals, exps, masks = [], [], []
        for t in range(nt):
            v = [rng.randrange(P) for _ in range(8)]
            if t % 8 == 0:
                v[3] = v[0]; v[4] = v[1]; v[5] = 0; v[6] = P - 1
            e = list(v)
            masks.append(A.emulate(prog, e))
            vals.append(v)
            exps.append(e)
        slots = u32([limbs(x * RM % P) for v in vals for x in v], 12)
        got_mask = np.zeros(nt, np.uint32)
        assert dev.fpvm_smem_run(pc, len(prog), nt, ptr(slots), ptr(got_mask)) == 0
        for t in range(nt):
            got = [value(slots[8 * t + s]) for s in range(8)]
            assert all(g < P for g in got), (name, t)
            assert [g * RINV % P for g in got] == exps[t], (name, t)
            assert int(got_mask[t]) == masks[t], (name, t)
        pc += len(prog)
