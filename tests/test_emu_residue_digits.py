"""The residue conversion of the emulated dense Schur product (emu_residue_kernel, k3_schur_syrk.cu)
reduces a' = rint(x 2^e) modulo each p through the unsigned bytes u_0..u_6 of a' + 2^55: two dp4a
products against the weights 256^k mod p give f = 2^23 + c_p + sum_k u_k (256^k mod p), congruent to a'
and below 2^24, and q = rint(f / p) is taken from one single-precision fma with the float nearest 1 / p.
That q must be the exact nearest integer for every f the digits can produce, so that r = f - p q lies in
[-127, 127]; this checks all of them, and the whole digit path against Python integers.  For p = 255
the f of that range do not all round right, so the kernel takes q from f - 2^23 there.  No GPU."""
import numpy as np
import pytest

MODULI = [256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193]
F_MAX = 2**23 + 7 * 255 * 255 + 2 * 256  # f below this for every digit vector and bias


def _rint_by_reciprocal(f, p):
    """rint(f * fl32(1 / p)) as one fma with the 1.5 * 2^23 constant rounds it (the product is exact in
    float64: 24 x 24 bits)."""
    return np.rint(f.astype(np.float64) * np.float64(np.float32(1.0 / p))).astype(np.int64)


@pytest.mark.parametrize("p", [p for p in MODULI if p not in (256, 255)])
def test_quotient_by_reciprocal_is_exact(p):
    f = np.arange(2**23, F_MAX, dtype=np.int64)
    q = _rint_by_reciprocal(f, p)
    assert np.array_equal(q, (2 * f + p) // (2 * p))
    assert np.abs(f - p * q).max() <= 127


def test_quotient_of_255_from_small_f():
    f = np.arange(0, 2 * 255 + 7 * 255, dtype=np.int64)  # f - 2^23 = c + digit sum, weights all 1
    q = _rint_by_reciprocal(f, 255)
    assert np.array_equal(q, (2 * f + 255) // 510)


def _residue_byte(a, p):
    """The kernel's arithmetic for one modulus, on Python integers: the int8 it stores."""
    v = (a + 2**55) & (2**64 - 1)
    u = [(v >> (8 * k)) & 0xFF for k in range(8)]
    assert u[7] == 0
    if p == 256:
        byte = u[0]
    else:
        c = (-(2**23) - 2**55) % p
        if p == 255:
            c += 2**23 % p
        f = 2**23 + c + sum(u[k] * (256**k % p) for k in range(7))
        g = f - 2**23 if p == 255 else f
        q = int(np.rint(np.float64(g) * np.float64(np.float32(1.0 / p))))
        byte = (f - p * q) & 0xFF
    return byte - 256 if byte > 127 else byte


def test_digit_path_gives_residues():
    rng = np.random.default_rng(3)
    vals = [0, 1, -1, 2**53, -(2**53), 2**53 - 1, -(2**53) + 1, 255, -256, 2**32, -(2**32) - 1]
    vals += [int(x) for x in rng.integers(-(2**53), 2**53, 2000)]
    for a in vals:
        for p in MODULI:
            r = _residue_byte(a, p)
            assert -128 <= r <= 127 and (r - a) % p == 0, (a, p, r)
