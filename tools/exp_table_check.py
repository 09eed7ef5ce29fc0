#!/usr/bin/env python
"""Exact-arithmetic check of the table-driven exp of csrc/models.cuh (exp_fast): every FMA is
evaluated in rationals and rounded once, as the hardware does; the result is compared with a 50-digit exp.
Prints the maximum relative error (measured: 1.93e-16 over 20,000 arguments in [-700, 700])."""
import math
import random
from decimal import Decimal, getcontext
from fractions import Fraction as F

getcontext().prec = 50
LN2 = Decimal(2).ln()
TAB = [float((LN2 * Decimal(j) / Decimal(32)).exp()) for j in range(32)]
A = float.fromhex('0x1.71547652b82fep+5')
H = -float.fromhex('0x1.62e42fefa39efp-6')
L = -float.fromhex('0x1.abc9e3b39803fp-61')
C = [float.fromhex(s) for s in ('0x1.6c16c16c16c17p-10', '0x1.1111111111111p-7', '0x1.5555555555555p-5',
                                '0x1.5555555555555p-3', '0x1.0000000000000p-1')]
MAGIC = 6755399441055744.0


def fma(a, b, c):
    return float(F(a) * F(b) + F(c))


def exp_table(x):
    t0 = fma(x, A, MAGIC)
    t = t0 - MAGIC
    ti = int(t)
    r = fma(t, L, fma(t, H, x))
    p = fma(C[0], r, C[1])
    for c in C[2:]:
        p = fma(p, r, c)
    q = fma(p, r * r, r)
    return math.ldexp(fma(TAB[ti & 31], q, TAB[ti & 31]), ti >> 5)


if __name__ == '__main__':
    random.seed(1)
    worst = 0.0
    for i in range(20000):
        x = random.uniform(-60, 60) if i % 2 else random.uniform(-700, 700)
        ex = Decimal(x).exp()
        worst = max(worst, float(abs((Decimal(exp_table(x)) - ex) / ex)))
    print(f'max relative error {worst:.3e} ({worst / 2 ** -53:.2f} x 2^-53)')
