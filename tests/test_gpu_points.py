"""Curve points outside the prime-order subgroup, on the device.

Every other test hands the library multiples of a generator.  Two parts of it only ever see other points:

* the curve and subgroup check (`bb_points_validate`), which decides whether a parameters file from outside is
  accepted (`params_io.read_parameters`);
* the group arithmetic of the MSM and the prover when a key was read with `checked=False`
  (`from_uncompressed_unchecked` upstream): the reference proves with such keys, so the proof bytes must match for
  them too.  With points of small order, the cases P = Q, P = -Q and a sum reaching the identity are the common
  case in the buckets, the batched-affine rounds, the window-multiple tables and the host ladder.

The expected values come from plain Python integers: the curve equation, and [k]P by double-and-add on the exact
integer k (`oracle0.fields.Curve.mul` reduces k mod r, which would hide every point outside the subgroup).
test_emulated_points.py runs the same bodies at small sizes against the host-thread build of the sources.
"""
import ctypes as C
import functools
import random
import re

import numpy as np
import pytest

import bellman_b200 as bb
from bellman_b200 import params_io
from oracle import o1
from oracle.oracle0 import fields as F

pytestmark = pytest.mark.gpu

R = o1.FR_MODULUS
P = o1.FP_MODULUS
Z = F.BLS_X
H1 = (Z - 1) ** 2 // 3                                                        # #E(Fp) = H1 r
H2 = (Z ** 8 - 4 * Z ** 7 + 5 * Z ** 6 - 4 * Z ** 4 + 6 * Z ** 3 - 4 * Z ** 2 - 4 * Z + 13) // 9   # #E'(Fp2) = H2 r
assert H1 == 3 * 11 ** 2 * 10177 ** 2 * 859267 ** 2 * 52437899 ** 2
assert H2 % (13 ** 2 * 23 ** 2 * 2713 * 11953 * 262069) == 0
ORDERS = {bb.G1: (3, 11, 10177), bb.G2: (13, 23, 2713)}
NONE = C.c_size_t(-1).value                                                   # first_bad when every point passes


def _curve(group):
    return F.G1 if group == bb.G1 else F.G2


def _cofactor(group):
    return H1 if group == bb.G1 else H2


def mul_exact(group, pt, k):
    """[k]pt for a non-negative integer k, by double-and-add: no reduction of k"""
    cv = _curve(group)
    acc = None
    while k:
        if k & 1:
            acc = cv.add(acc, pt)
        pt = cv.add(pt, pt)
        k >>= 1
    return acc


def py_check(group, pt):
    """what from_uncompressed decides: 0 accepted (the identity included), 1 off the curve, 2 outside the subgroup"""
    if pt is None:
        return 0
    if not _curve(group).is_on_curve(pt):
        return 1
    return 0 if mul_exact(group, pt, R) is None else 2


def _sqrt_fp(a):
    y = pow(a, (P + 1) // 4, P)                                               # p = 3 mod 4
    return y if y * y % P == a % P else None


def _sqrt_fp2(a):
    """a square root in Fp2 = Fp[u]/(u^2 + 1) through the norm, or None; checked by squaring"""
    a0, a1 = a
    cands = []
    if a1 == 0:
        s = _sqrt_fp(a0)
        cands.append((s, 0) if s is not None else None)
        s = _sqrt_fp(-a0 % P)                                                 # (s u)^2 = -s^2
        cands.append((0, s) if s is not None else None)
    else:
        n = _sqrt_fp((a0 * a0 + a1 * a1) % P)
        if n is not None:
            for t in (n, P - n):
                x0 = _sqrt_fp((a0 + t) * pow(2, -1, P) % P)
                if x0:
                    cands.append((x0, a1 * pow(2 * x0, -1, P) % P))
    for c in cands:
        if c is not None and F.Fp2Ops.mul(c, c) == (a0 % P, a1 % P):
            return c
    return None


def random_curve_point(group, rng):
    """a random point of E(Fp) or E'(Fp2) from a random x; outside the subgroup with overwhelming probability"""
    cv = _curve(group)
    while True:
        x = rng.randrange(P) if group == bb.G1 else (rng.randrange(P), rng.randrange(P))
        rhs = cv.F.add(cv.F.mul(cv.F.mul(x, x), x), cv.b)
        y = _sqrt_fp(rhs) if group == bb.G1 else _sqrt_fp2(rhs)
        if y is not None:
            pt = (x, y)
            assert cv.is_on_curve(pt)
            return pt


@functools.lru_cache(maxsize=None)
def torsion_point(group, ell, seed):
    """a point of order exactly ell (a prime dividing the cofactor).  [(h r) / ell]Q is not enough: the ell-part of the
    group can be Z/ell x Z/ell (it is for ell = 11 in G1), and then that multiple is always the identity.  So Q is
    multiplied by h r with every factor ell removed, and the result by ell until one more step would reach the identity."""
    h = _cofactor(group)
    assert h % ell == 0
    m = h * R
    while m % ell == 0:
        m //= ell
    rng = random.Random(seed * 1000 + ell)
    for _ in range(40):
        t = mul_exact(group, random_curve_point(group, rng), m)
        if t is None:
            continue
        while (u := mul_exact(group, t, ell)) is not None:
            t = u
        assert _curve(group).is_on_curve(t)
        return t
    raise AssertionError(f"no point of order {ell} found")


@functools.lru_cache(maxsize=None)
def subgroup_point(group, seed):
    return mul_exact(group, _curve(group).gen, random.Random(seed).randrange(1, R))


def to_abi(group, pts):
    """affine integer points (None = identity) -> the library's Montgomery rows"""
    return o1.g1_from_affine_ints(list(pts)) if group == bb.G1 else o1.g2_from_affine_ints(list(pts))


def from_abi(group, arr):
    return o1.g1_to_affine_ints(arr) if group == bb.G1 else o1.g2_to_affine_ints(arr)


def _add_one_to_y(group, pt):
    x, y = pt
    return (x, (y + 1) % P) if group == bb.G1 else (x, ((y[0] + 1) % P, y[1]))


@functools.lru_cache(maxsize=None)
def bad_points(group):
    """(name, point, why) of points from_uncompressed refuses: why 1 off the curve, 2 outside the subgroup"""
    cv = _curve(group)
    pg = subgroup_point(group, 7)
    pts = [(f"order {ell}", torsion_point(group, ell, 1)) for ell in ORDERS[group]]
    pts += [(f"P + order-{ell}", cv.add(pg, torsion_point(group, ell, 2))) for ell in ORDERS[group][::2]]
    pts.append(("E minus G", random_curve_point(group, random.Random(11 + group))))
    pts.append(("y + 1", _add_one_to_y(group, pg)))
    pts.append(("torsion y + 1", _add_one_to_y(group, torsion_point(group, ORDERS[group][0], 1))))
    if group == bb.G1:
        pts += [("(0, 2)", (0, 2)), ("(0, -2)", (0, P - 2))]
    else:
        g1 = subgroup_point(bb.G1, 8)                                         # on y^2 = x^3 + 4, not on the twist
        pts.append(("G1 point in Fp2", ((g1[0], 0), (g1[1], 0))))
    out = [(name, pt, py_check(group, pt)) for name, pt in pts]
    assert py_check(group, pg) == 0 and py_check(group, None) == 0
    assert {w for _, _, w in out} == {1, 2}
    if group == bb.G1:                                                        # (0, +-2) has order 3, and [r](0, 2) = (0, 2)
        assert dict((n, w) for n, _, w in out)["(0, 2)"] == 2 and mul_exact(group, (0, 2), R) == (0, 2)
    return tuple(out)


def validate(worker, group, arr, check_subgroup=1):
    first, why = C.c_size_t(), C.c_int()
    a = np.ascontiguousarray(arr, dtype=np.uint64)
    bb._check(bb.load_library().bb_points_validate(worker._h, C.c_int(group), a.ctypes.data_as(C.c_void_p), C.c_size_t(a.shape[0]),
                                                   C.c_int(check_subgroup), C.byref(first), C.byref(why)))
    return first.value, why.value


def subgroup_vector(worker, group, n, seed):
    """n points [k]G, every 61st one the identity (accepted by the check); long vectors are made on the device"""
    ks = o1.fr_random(seed, n)
    fixed = o1.g1_fixed_mul if group == bb.G1 else o1.g2_fixed_mul
    if n <= 4096:
        v = fixed(ks)
    else:
        v = bb.fixed_base_mul(worker, group, ks)
        assert np.array_equal(v[:3], fixed(ks[:3]))
    v[5::61] = 0
    return v


@pytest.fixture(scope="module")
def worker():
    w = bb.Worker(0)
    yield w
    w.close()


# --------------------------------------------------------------------------------------------
# 1. the curve and subgroup check against Python
# --------------------------------------------------------------------------------------------
def validation_case(worker, group, n, sites=(0, 127, 128, -1)):
    """bad points planted at indices 0, 127, 128 and n - 1 (both sides of the 128-thread blocks), alone and in pairs of
    different kinds: the lower index wins, with its own reason.  check_subgroup = 0 passes subgroup failures only."""
    bad = bad_points(group)
    for name, pt, why in bad:                                                 # each one alone first
        assert validate(worker, group, to_abi(group, [pt])) == (0, why), (group, name)
    v = subgroup_vector(worker, group, n, 900 + n + group)
    for cs in (1, 0):
        assert validate(worker, group, v, cs) == (NONE, 0), (n, cs)
    sites = sorted({i % n for i in sites if -n <= i < n})

    def expect(planted, cs):                                                  # planted: {index: why}
        hits = sorted(i for i, w in planted.items() if w == 1 or cs)
        return (hits[0], planted[hits[0]]) if hits else (NONE, 0)

    def run(planted_pts, cs):
        saved = {i: v[i].copy() for i in planted_pts}
        try:
            for i, pt in planted_pts.items():
                v[i] = to_abi(group, [pt])[0]
            return validate(worker, group, v, cs)
        finally:
            for i, row in saved.items():
                v[i] = row

    for name, pt, why in bad:
        for i in sites:
            for cs in (1, 0):
                assert run({i: pt}, cs) == expect({i: why}, cs), (group, n, name, i, cs)
    off = [b for b in bad if b[2] == 1]
    sub = [b for b in bad if b[2] == 2]
    combos = [(off[0], sub[0]), (sub[0], off[0]), (sub[1], sub[-1]), (off[-1], off[0]), (sub[-1], off[-1])]
    for i in sites:
        for j in sites:
            if i >= j:
                continue
            for (na, pa, wa), (nb, pb, wb) in combos:
                for cs in (1, 0):
                    assert run({i: pa, j: pb}, cs) == expect({i: wa, j: wb}, cs), (group, n, na, i, nb, j, cs)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 1000])
@pytest.mark.parametrize("group", [bb.G1, bb.G2])
def test_points_validate_matches_python(worker, group, n):
    validation_case(worker, group, n)


@pytest.mark.parametrize("group,log_n", [(bb.G1, 20), (bb.G2, 16)])
def test_points_validate_long_vectors(worker, group, log_n):
    validation_case(worker, group, 1 << log_n)


def test_points_validate_identity_and_subgroup(worker):
    for group in (bb.G1, bb.G2):
        assert validate(worker, group, np.zeros((0, 12 * group), np.uint64)) == (NONE, 0)
        assert validate(worker, group, np.zeros((200, 12 * group), np.uint64)) == (NONE, 0)
        pts = [subgroup_point(group, s) for s in range(4)] + [None]
        assert all(py_check(group, p) == 0 for p in pts)
        assert validate(worker, group, to_abi(group, pts)) == (NONE, 0)


# --------------------------------------------------------------------------------------------
# 2. read_parameters on the device, element by element
# --------------------------------------------------------------------------------------------
def _layout(p):
    """(name, index or None, is_g2, byte offset) of every point of write_parameters(p)"""
    out, off = [], 0
    for name, g2 in (("alpha_g1", False), ("beta_g1", False), ("beta_g2", True), ("gamma_g2", True), ("delta_g1", False), ("delta_g2", True)):
        out.append((name, None, g2, off))
        off += 192 if g2 else 96
    for name, g2 in (("ic", False), ("h", False), ("l", False), ("a", False), ("b_g1", False), ("b_g2", True)):
        off += 4
        for i in range(np.asarray(p[name]).reshape(-1, 24 if g2 else 12).shape[0]):
            out.append((name, i, g2, off))
            off += 192 if g2 else 96
    return out, off


def _encode(group, pt):
    return F.g1_uncompressed(pt) if group == bb.G1 else F.g2_uncompressed(pt)


def read_parameters_case(worker, rounds=4):
    """each VerifyingKey element, every ic entry, and one element of each vector, replaced by an off-curve point and by
    a point outside the subgroup: checked=True refuses naming the element and index, checked=False loads the vectors
    unchanged and still refuses the VerifyingKey"""
    rng = random.Random(rounds)
    mc = o1.Mimc(rounds, seed=rounds + 1)
    mc.set_toxic([rng.randrange(1, R) for _ in range(5)])
    mc.generate()
    p = mc.export_params()
    data = params_io.write_parameters(p)
    layout, end = _layout(p)
    assert end == len(data)
    good = params_io.read_parameters(data, worker=worker)
    for k in ("vk_g1", "vk_g2", "ic", "h", "l", "a", "b_g1", "b_g2"):
        assert np.array_equal(good[k].reshape(-1), np.asarray(p[k]).reshape(-1)), k
    vk_rows = {"alpha_g1": ("vk_g1", 0), "beta_g1": ("vk_g1", 1), "delta_g1": ("vk_g1", 2),
               "beta_g2": ("vk_g2", 0), "gamma_g2": ("vk_g2", 1), "delta_g2": ("vk_g2", 2)}
    chosen = [e for e in layout if e[1] is None or e[0] == "ic"]
    for name in ("h", "l", "a", "b_g1", "b_g2"):
        rows = [e for e in layout if e[0] == name]
        chosen.append(rows[rng.randrange(len(rows))])
    for name, idx, g2, off in chosen:
        group = bb.G2 if g2 else bb.G1
        key, row = vk_rows[name] if idx is None else (name, idx)
        orig = from_abi(group, np.asarray(p[key]).reshape(-1, 24 if g2 else 12)[row:row + 1])[0]
        ell = ORDERS[group][rng.randrange(3)]
        for pt, why, reason in ((_add_one_to_y(group, orig), 1, "not on the curve"),
                                (_curve(group).add(orig, torsion_point(group, ell, 3)), 2, "not in the prime-order subgroup")):
            assert py_check(group, pt) == why
            blob = bytearray(data)
            size = 192 if g2 else 96
            blob[off:off + size] = _encode(group, pt)
            what = re.escape(f"invalid {'G2' if g2 else 'G1'}: {name}[{0 if idx is None else idx}] is {reason}")
            with pytest.raises(params_io.InvalidData, match=what):
                params_io.read_parameters(bytes(blob), checked=True, worker=worker)
            if idx is None or name == "ic":                                   # VerifyingKey::read has no unchecked mode
                with pytest.raises(params_io.InvalidData, match=what):
                    params_io.read_parameters(bytes(blob), checked=False, worker=worker)
                continue
            q = params_io.read_parameters(bytes(blob), checked=False, worker=worker)
            want = np.asarray(p[key]).reshape(-1, 24 if g2 else 12).copy()
            want[row] = to_abi(group, [pt])[0]
            assert np.array_equal(q[key], want), (name, idx, why)
            for k in ("vk_g1", "vk_g2", "ic", "h", "l", "a", "b_g1", "b_g2"):
                if k != key:
                    assert np.array_equal(q[k].reshape(-1), np.asarray(p[k]).reshape(-1)), (name, k)


def test_read_parameters_refuses_each_element(worker):
    read_parameters_case(worker)


# --------------------------------------------------------------------------------------------
# 3. MSM over points outside the subgroup, against the oracle
# --------------------------------------------------------------------------------------------
def mixed_bases(group, n, seed):
    """subgroup points, torsion points of each order, and P + T, in random order; the P + T rows come from the oracle's
    affine addition, checked against Python on a sample"""
    rng = random.Random(seed)
    fixed, add = (o1.g1_fixed_mul, o1.g1_add) if group == bb.G1 else (o1.g2_fixed_mul, o1.g2_add)
    bases = fixed(o1.fr_random(seed, n))
    tors = to_abi(group, [torsion_point(group, ell, s) for ell in ORDERS[group] for s in (1, 2)])
    kind = np.array([rng.randrange(5) for _ in range(n)])                    # 0, 1: P   2: T   3, 4: P + T
    t_rows = tors[[rng.randrange(tors.shape[0]) for _ in range(n)]]
    pt_rows = add(bases, t_rows)
    out = bases.copy()
    out[kind == 2] = t_rows[kind == 2]
    out[kind >= 3] = pt_rows[kind >= 3]
    cv = _curve(group)
    for i in [i for i in range(n) if kind[i] >= 3][:4]:
        want = cv.add(from_abi(group, bases[i:i + 1])[0], from_abi(group, t_rows[i:i + 1])[0])
        assert from_abi(group, out[i:i + 1])[0] == want
    return out


def edge_scalars(n, seed):
    ex = o1.fr_random(seed, n)
    edge = o1.fr_from_ints([0, 1, R - 1, 2, 3, R - 2])
    for i in range(0, n, 7):
        ex[i] = edge[(i // 7) % edge.shape[0]]
    return ex


def _msm(worker, group, bases, ex):
    return bb.multiexp(worker, (bb.Bases(worker, group, bases), 0), bb.FullDensity, ex).wait()


def msm_outside_subgroup_case(worker, group, n, forms=(0, 1, 2), windows=(2, 3, 8, 13, 15, 16), rounds=(1, 2, 3, 4, 5)):
    """mixed bases under every MSM form, forced window sizes, forced batched-affine rounds and task splitting; and one
    small-order point T repeated n times, whose MSM is [(sum k_i) mod ell]T whatever the oracle says"""
    bases = mixed_bases(group, n, 7000 + n + group)
    ex = edge_scalars(n, 8000 + n + group)
    rc, want = o1.multiexp(group, bases, 0, None, ex)
    assert rc == 0
    ell = ORDERS[group][0]
    t = torsion_point(group, ell, 1)
    same = to_abi(group, [t] * n)
    ks = o1.fr_random(9000 + n, n)
    closed = to_abi(group, [mul_exact(group, t, sum(o1.fr_to_ints(ks)) % ell)])
    rc, want_same = o1.multiexp(group, same, 0, None, ks)
    assert rc == 0 and np.array_equal(want_same, closed)
    try:
        for form in forms:
            worker.set_option("msm_precompute", form)
            settings = [(None, None)] + [("msm_window_bits", c) for c in windows] + [("msm_affine_rounds", r) for r in rounds] + [("msm_big_cap", 3)]
            for key, value in settings:
                if key:
                    worker.set_option(key, value)
                try:
                    assert np.array_equal(_msm(worker, group, bases, ex), want), (group, n, form, key, value)
                    assert np.array_equal(_msm(worker, group, same, ks), closed), (group, n, form, key, value, "same T")
                finally:
                    if key:
                        worker.set_option(key, -1 if key == "msm_affine_rounds" else 0)
    finally:
        worker.set_option("msm_precompute", 0)
        worker.set_option("msm_window_bits", 0)
        worker.set_option("msm_affine_rounds", -1)
        worker.set_option("msm_big_cap", 0)


@pytest.mark.parametrize("group,n", [(bb.G1, 1), (bb.G1, 33), (bb.G1, 1000), (bb.G1, 1 << 14), (bb.G2, 3), (bb.G2, 300), (bb.G2, 1 << 12)])
def test_msm_outside_subgroup(worker, group, n):
    msm_outside_subgroup_case(worker, group, n)


# --------------------------------------------------------------------------------------------
# 5. proving with a key read unchecked
# --------------------------------------------------------------------------------------------
def unchecked_key_prove_case(worker, rounds=322, shard_counts=(2, 8), pairs=3):
    """a few entries of h, l, a, b_g1 and b_g2 become P + T, one of h a pure torsion point; read_parameters(checked=False)
    loads the key and the device proves to the oracle's bytes, whole, sharded and under the table form"""
    rng = random.Random(rounds + 500)
    mc = o1.Mimc(rounds, seed=rounds + 501)
    mc.set_toxic([rng.randrange(1, R) for _ in range(5)])
    mc.generate()
    p = mc.export_params()
    for name in ("h", "l", "a", "b_g1", "b_g2"):
        group = bb.G2 if name == "b_g2" else bb.G1
        arr = np.array(p[name], copy=True)
        rows = rng.sample(range(arr.shape[0]), min(3, arr.shape[0]))
        for row, ell in zip(rows, ORDERS[group]):
            arr[row] = to_abi(group, [_curve(group).add(from_abi(group, arr[row:row + 1])[0], torsion_point(group, ell, 4))])[0]
        if name == "h":
            arr[(rows[0] + 1) % arr.shape[0]] = to_abi(group, [torsion_point(group, ORDERS[group][1], 5)])[0]
        p[name] = arr
    blob = params_io.write_parameters(p)
    with pytest.raises(params_io.InvalidData, match="subgroup"):
        params_io.read_parameters(blob, checked=True, worker=worker)
    q = params_io.read_parameters(blob, checked=False, worker=worker)
    for k in ("vk_g1", "vk_g2", "h", "l", "a", "b_g1", "b_g2"):
        assert np.array_equal(q[k].reshape(-1), np.asarray(p[k]).reshape(-1)), k
    params = bb.Parameters(worker, q)
    mc.import_params(q)
    w = mc.witness()
    asg = bb.ProvingAssignment(w["a"], w["b"], w["c"], w["inputs"], w["aux"], w["a_aux_density"], w["b_input_density"], w["b_aux_density"])
    try:
        for _ in range(pairs):
            r, s = rng.randrange(R), rng.randrange(R)
            proof = bb.create_proof(asg, params, r, s)
            assert proof == mc.prove(r, s)
            assert proof != mc.expected_proof(r, s)                         # the torsion parts did reach the proof
        for count in shard_counts:
            parts = []
            for k in range(count):
                pk = bb.Parameters(worker, q, shard_index=k, shard_count=count)
                parts.append(bb.prove_partials(asg, pk))
                pk.free()
            assert bb.finalize(params, parts, r, s) == proof, count
        params.apply_tuning(1)
        assert bb.create_proof(asg, params, r, s) == proof
    finally:
        params.apply_tuning(0)
        params.free()


def test_prove_with_unchecked_key(worker):
    unchecked_key_prove_case(worker)
