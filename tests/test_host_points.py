"""Host-side pieces of the product that run without a GPU (they sit on the multi-GPU reduction
path and in bb_groth16_finalize): affine point addition, scalar multiplication and the ZCash
compressed encoding (GroupEncoding::to_bytes, groth16/src/lib.rs:39-45), against the oracle."""
import ctypes as C
import random

import numpy as np

import bellman_b200 as bb
from oracle import o1

import test_gpu_points as GP

R = o1.FR_MODULUS


def test_point_add_mul_compress_host():
    lib = bb.load_library()
    rng = random.Random(5)
    ks = [rng.randrange(1, R) for _ in range(12)]
    for group, fixed, add, mul, comp, w in ((bb.G1, o1.g1_fixed_mul, o1.g1_add, o1.g1_mul, o1.g1_compress, 12),
                                            (bb.G2, o1.g2_fixed_mul, o1.g2_add, o1.g2_mul, o1.g2_compress, 24)):
        pts = fixed(o1.fr_from_ints(ks))
        zero = np.zeros((1, w), np.uint64)
        for i in range(0, 10, 2):
            a, b = pts[i:i + 1], pts[i + 1:i + 2]
            assert np.array_equal(bb.point_add(group, a, b), add(a, b))
        assert np.array_equal(bb.point_add(group, pts[0:1], pts[0:1]), add(pts[0:1], pts[0:1]))      # doubling
        assert np.array_equal(bb.point_add(group, pts[0:1], zero), pts[0:1])                          # + identity
        neg = mul(pts[0:1], o1.fr_from_ints([R - 1]))
        assert not bb.point_add(group, pts[0:1], neg).any()                                           # P + (-P)
        # the multiplication is a regular signed-digit ladder (odd digits, even scalars as (k + 1) P - P): digit boundaries,
        # even / odd, all-ones and sparse scalars
        for k in [0, 1, 2, 15, 16, 17, 31, 32, 33, R - 1, R - 2, (R - 1) // 2, 1 << 252, (1 << 252) - 1, (1 << 254) + 1,
                  int("f" * 63, 16), int("8" * 63, 16), int("10" * 31, 16)] + [rng.randrange(R) for _ in range(12)]:
            km = o1.fr_from_ints([k])
            out = np.zeros((1, w), np.uint64)
            assert lib.bb_point_mul(C.c_int(group), pts[2:3].ctypes.data_as(C.c_void_p), km.ctypes.data_as(C.c_void_p),
                                    C.c_int(bb.FORM_MONTGOMERY), out.ctypes.data_as(C.c_void_p)) == 0
            assert np.array_equal(out, mul(pts[2:3], km)), k
            kc = o1.fr_to_canonical(km)
            assert lib.bb_point_mul(C.c_int(group), pts[2:3].ctypes.data_as(C.c_void_p), kc.ctypes.data_as(C.c_void_p),
                                    C.c_int(bb.FORM_CANONICAL), out.ctypes.data_as(C.c_void_p)) == 0
            assert np.array_equal(out, mul(pts[2:3], km)), k
        out = np.ones((1, w), np.uint64)                                                              # k * identity = identity
        km = o1.fr_from_ints([rng.randrange(R)])
        assert lib.bb_point_mul(C.c_int(group), zero.ctypes.data_as(C.c_void_p), km.ctypes.data_as(C.c_void_p),
                                C.c_int(bb.FORM_MONTGOMERY), out.ctypes.data_as(C.c_void_p)) == 0 and not out.any()
        want = comp(pts)
        for i in range(len(ks)):
            assert bb.point_compress(group, pts[i:i + 1]) == bytes(want[i])
        assert bb.point_compress(group, zero) == bytes([0xC0] + [0] * (47 if group == bb.G1 else 95))
        # points outside the prime-order subgroup (a key read unchecked may hold them): small-order points T and P + T,
        # against exact integer arithmetic.  For T of order 3 the ladder's table entries 3T, 9T, 15T are the identity.
        cv = GP._curve(group)
        p_int = GP.subgroup_point(group, 3)
        odd = [GP.torsion_point(group, ell, 6) for ell in GP.ORDERS[group]]
        odd += [cv.add(p_int, t) for t in odd] + [GP.random_curve_point(group, random.Random(6))]
        for a in odd:
            a_arr = GP.to_abi(group, [a])
            for b in odd[:4] + [a, cv.neg(a), p_int, None]:
                assert GP.from_abi(group, bb.point_add(group, a_arr, GP.to_abi(group, [b])))[0] == cv.add(a, b)
            for k in [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, R - 1, R - 2] + [rng.randrange(R) for _ in range(3)]:
                out = np.zeros((1, w), np.uint64)
                kc = o1.fr_to_canonical(o1.fr_from_ints([k]))
                assert lib.bb_point_mul(C.c_int(group), a_arr.ctypes.data_as(C.c_void_p), kc.ctypes.data_as(C.c_void_p),
                                        C.c_int(bb.FORM_CANONICAL), out.ctypes.data_as(C.c_void_p)) == 0
                assert GP.from_abi(group, out)[0] == GP.mul_exact(group, a, k), k
