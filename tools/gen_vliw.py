#!/usr/bin/env python3
"""Generate kzg_rs_b200/csrc/vliw_programs.cuh: straight-line Fp programs for the cooperative pairing engine.

The serial tails of the batch (one pairing check, the Horner recombination of the MSM) are long chains of
Fp12 / point operations.  One thread runs them at ~1 us per Fp multiplication; a CTA can run the independent
Fp multiplications inside each Fp12 / point operation side by side.  This script traces the tower / curve
formulas symbolically, keeps additions lazy (values are small-integer linear combinations of materialised
registers), and emits each operation as a short list of LEVELS of independent instructions over a register file
of Fp values in shared memory:
    MUL : dst = s0*s1 [+/- s2*s3]      (fused dual Montgomery product)
    LIN : dst = sum_k (+/-)(1|2) * src_k
Instruction k of a level is executed by thread k; levels are separated by a barrier (vliw.cuh).

Self-check: every program is interpreted here with Python integers and compared with oracle/pyref.py.
    python tools/gen_vliw.py
"""
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyref as R

P = R.P
MAX_LIN_TERMS = 24
MAX_OPERAND_TERMS = 4


class Val:
    """small-integer linear combination of registers"""
    __slots__ = ("t",)

    def __init__(self, t=None):
        self.t = {k: v for k, v in (t or {}).items() if v != 0}

    def __add__(self, o):
        t = dict(self.t)
        for k, v in o.t.items():
            t[k] = t.get(k, 0) + v
        return Val(t)

    def __sub__(self, o):
        t = dict(self.t)
        for k, v in o.t.items():
            t[k] = t.get(k, 0) - v
        return Val(t)

    def __neg__(self):
        return Val({k: -v for k, v in self.t.items()})

    def scale(self, c):
        return Val({k: v * c for k, v in self.t.items()})


class Builder:
    headroom = False            # Builder29: values carry slack (multiples of p) instead of being reduced after every sum

    def __init__(self, name, n_inputs):
        self.name = name
        self.n_inputs = n_inputs
        self.next_reg = n_inputs
        self.level_of = {r: 0 for r in range(n_inputs)}   # reg -> level at which it becomes available
        self.instrs = []                                    # (level, kind, dst, payload)
        self.cache = {}

    def input(self, i):
        return Val({i: 1})

    def _new(self, level):
        r = self.next_reg
        self.next_reg += 1
        self.level_of[r] = level
        return r

    def materialize(self, v):
        """register holding v (emits a LIN unless v is a plain register)"""
        if len(v.t) == 1 and list(v.t.values())[0] == 1:
            return list(v.t.keys())[0]
        key = tuple(sorted(v.t.items()))
        if key in self.cache:
            return self.cache[key]
        terms = []
        for r, c in sorted(v.t.items()):
            neg, c = c < 0, abs(c)
            while c >= 2:
                terms.append((r, neg, True))
                c -= 2
            if c:
                terms.append((r, neg, False))
        if len(terms) > MAX_LIN_TERMS:   # split long sums
            half = len(v.t) // 2
            items = sorted(v.t.items())
            a = self.materialize(Val(dict(items[:half])))
            b = self.materialize(Val(dict(items[half:])))
            return self.materialize(Val({a: 1}) + Val({b: 1}))
        level = 1 + max((self.level_of[r] for r, _, _ in terms), default=0)
        dst = self._new(level)
        self.instrs.append((level, "LIN", dst, terms))
        self.cache[key] = dst
        return dst

    def operand(self, v):
        """A multiplication operand = up to MAX_OPERAND_TERMS registers with signs (small coefficients expand into repeated terms):
        the multiplying thread forms the sum itself, lazily: sum(pos) + #neg * p - sum(neg) < 4p, one conditional subtraction of
        2p brings it below 2p, which the Montgomery products tolerate (4 operands < 2p: ab + cd < 8 p^2 < R p).  Longer sums are
        materialised by a LIN instruction.  Returns [(reg, minus), ...]."""
        terms = []
        for r, c in sorted(v.t.items()):
            terms += [(r, c < 0)] * abs(c)
        if 1 <= len(terms) <= MAX_OPERAND_TERMS and any(not minus for _, minus in terms):
            terms.sort(key=lambda t: t[1])          # a positive term first
            return terms
        return [(self.materialize(v), False)]

    def mul(self, a, b, c=None, d=None, neg=False):
        """a*b (+|-) c*d"""
        ops = [self.operand(a), self.operand(b)]
        if c is not None:
            ops += [self.operand(c), self.operand(d)]
        level = 1 + max(self.level_of[r] for o in ops for r, _ in o)
        dst = self._new(level)
        self.instrs.append((level, "MUL", dst, (ops, neg)))
        return Val({dst: 1})

    def output(self, v, reg):
        """force v into register `reg` (an input slot being overwritten or a dedicated output slot)"""
        terms = []
        for r, c in sorted(v.t.items()):
            ng, c = c < 0, abs(c)
            while c >= 2:
                terms.append((r, ng, True)); c -= 2
            if c:
                terms.append((r, ng, False))
        if len(terms) > MAX_LIN_TERMS:
            m = self.materialize(v)
            terms = [(m, False, False)]
        level = 1 + max((self.level_of[r] for r, _, _ in terms), default=0)
        self.instrs.append((level, "OUT", reg, terms))

    def finish(self):
        """Level schedule.  ASAP levels first; then MUL instructions sink to the latest level their consumers
        allow (so an operation's independent products share ONE multiplication level instead of splitting into
        "products of raw inputs" and "products of sums"); all OUT instructions form one extra final level, which
        makes overwriting input registers safe."""
        body = [list(i) for i in self.instrs if i[1] != "OUT"]
        outs = [i for i in self.instrs if i[1] == "OUT"]
        last = max([i[0] for i in body] + [0])
        by_dst = {i[2]: i for i in body}
        def srcs_of(i):
            return mul_srcs(i[3][0]) if i[1] == "MUL" else [r for r, _, _ in i[3]]
        changed = True
        while changed:
            changed = False
            limit = {}
            for i in body:
                for r in srcs_of(i):
                    if r in by_dst:
                        limit[r] = min(limit.get(r, last + 1), i[0])
            for i in body:
                if i[1] != "MUL":
                    continue
                alap = limit.get(i[2], last + 1) - 1
                if alap > i[0]:
                    i[0] = alap
                    changed = True
        levels = {}
        for lv, k, dst, pay in body:
            levels.setdefault((lv, k), []).append((k, dst, pay))
        prog = []
        # LIN instructions of a level sorted by length: the threads of a warp then run sums of similar length (a warp runs as
        # many term iterations as its longest sum)
        by_len = lambda ins: sorted(ins, key=lambda i: -len(i[2]))
        for lv in range(1, last + 1):
            for kind in ("LIN", "MUL"):
                if (lv, kind) in levels:
                    prog.append((kind, by_len(levels[(lv, kind)]) if kind == "LIN" else levels[(lv, kind)]))
        if outs:
            prog.append(("LIN", by_len([("LIN", dst, pay) for _, _, dst, pay in outs])))
        return prog


BUILDER = Builder

# ------------------------------------------------------------------------------------------ headroom programs (vliw29.cuh)
# Second engine representation: Fp values as 14 SIGNED limbs of 29 bits (Montgomery radix 2^406 = 2^25.3 p), products as
# carry-free 64-bit column sums.  The 25 spare bits replace the modular reduction after every sum: a register holds ANY
# representative v with |v| < bound * p; the bounds are tracked HERE, statically:
#   MUL  d = (a b +- c d) / 2^406 (mod p): needs A B + C D <= 2^23 (bounds in units of p); |d| < 1.25 p;
#   LIN  d = sum +-(1|2) src: no reduction unless the bound leaves LIN_LIMIT (program outputs: IO_BOUND), in which case the
#        instruction carries a `reduce` flag: the executing lanes subtract round-estimate(v / p) * p (float estimate from the two
#        top columns), leaving |d| < RED_BOUND * p.
import math
from fractions import Fraction

W29, N29 = 29, 14
R29 = 1 << (W29 * N29)
IO_BOUND = 8
RED_BOUND = 4
LIN_LIMIT = 1024
MUL_BOUND = Fraction(5, 4)
MULSUM_LIMIT = 1 << 23


class Terms(list):
    """LIN payload of the headroom programs: the term list + the reduce flag"""
    reduce = False


class Builder29(Builder):
    headroom = True

    def __init__(self, name, n_inputs):
        super().__init__(name, n_inputs)
        self.bound = {r: Fraction(IO_BOUND) for r in range(n_inputs)}

    @staticmethod
    def _terms(v):
        terms = []
        for r, c in sorted(v.t.items()):
            neg, c = c < 0, abs(c)
            while c >= 2:
                terms.append((r, neg, True))
                c -= 2
            if c:
                terms.append((r, neg, False))
        return terms

    def _meta(self, terms, limit):
        b = sum(((2 if t[2] else 1) * self.bound[t[0]] for t in terms), Fraction(0))
        assert b < (1 << 20), "sum too large for the float quotient estimate"
        t = Terms(terms)
        t.reduce = b > limit
        return t, (Fraction(RED_BOUND) if t.reduce else b)

    def materialize(self, v):
        if len(v.t) == 1 and list(v.t.values())[0] == 1:
            return list(v.t.keys())[0]
        key = tuple(sorted(v.t.items()))
        if key in self.cache:
            return self.cache[key]
        terms = self._terms(v)
        if len(terms) > MAX_LIN_TERMS:
            items = sorted(v.t.items())
            half = len(items) // 2
            a = self.materialize(Val(dict(items[:half])))
            b = self.materialize(Val(dict(items[half:])))
            return self.materialize(Val({a: 1}) + Val({b: 1}))
        level = 1 + max((self.level_of[r] for r, _, _ in terms), default=0)
        dst = self._new(level)
        pay, self.bound[dst] = self._meta(terms, LIN_LIMIT)
        self.instrs.append((level, "LIN", dst, pay))
        self.cache[key] = dst
        return dst

    def operand(self, v):
        return [(self.materialize(v), False)]

    def mul(self, a, b, c=None, d=None, neg=False):
        ops = [self.operand(a), self.operand(b)]
        if c is not None:
            ops += [self.operand(c), self.operand(d)]
        bs = [self.bound[o[0][0]] for o in ops]
        total = bs[0] * bs[1] + (bs[2] * bs[3] if c is not None else 0)
        assert total + 1 <= MULSUM_LIMIT, "operand bounds too large"
        level = 1 + max(self.level_of[r] for o in ops for r, _ in o)
        dst = self._new(level)
        self.bound[dst] = MUL_BOUND
        self.instrs.append((level, "MUL", dst, (ops, bool(neg))))
        return Val({dst: 1})

    def output(self, v, reg):
        terms = self._terms(v)
        if len(terms) > MAX_LIN_TERMS:
            terms = [(self.materialize(v), False, False)]
        level = 1 + max((self.level_of[r] for r, _, _ in terms), default=0)
        pay, b = self._meta(terms, IO_BOUND)
        assert b <= IO_BOUND
        self.instrs.append((level, "OUT", reg, pay))


def limbs29(v):
    """signed limbs: 13 limbs in [0, 2^29), the top limb carries the sign"""
    assert -R29 < v < R29
    l = [(v >> (W29 * i)) & ((1 << W29) - 1) for i in range(N29 - 1)]
    return l + [v >> (W29 * (N29 - 1))]


def lin29_exact(values, pay):
    """the LIN instruction as vliw29.cuh executes it: 64-bit column sums, then the float32 quotient estimate"""
    import numpy as np
    f32 = np.float32
    pl = limbs29(P)
    t = [0] * N29
    for r, ng, db in pay:
        c = (2 if db else 1) * (-1 if ng else 1)
        for i, x in enumerate(limbs29(values[r])):
            t[i] += c * x
    if pay.reduce:
        vf = f32(f32(t[13]) * f32(536870912.0)) + f32(t[12])
        pinv = f32(1.0) / f32(f32(f32(pl[13]) * f32(536870912.0)) + f32(pl[12]))
        q = int(np.rint(f32(vf * pinv)))
        for i in range(N29):
            t[i] -= q * pl[i]
    return sum(x << (W29 * i) for i, x in enumerate(t))


def run29_exact(prog, regs):
    """registers hold the actual (signed) integers: Montgomery residues to the radix 2^406 with slack; bounds are asserted"""
    pinv = (-pow(P, -1, R29)) % R29
    for kind, ins in prog:
        new = {}
        for _, dst, pay in ins:
            if kind == "MUL":
                ops, neg = pay
                assert all(len(o) == 1 and not o[0][1] for o in ops)
                x = [regs[o[0][0]] for o in ops]
                t = x[0] * x[1]
                if len(x) == 4:
                    t = t - x[2] * x[3] if neg else t + x[2] * x[3]
                m = (t * pinv) % R29
                v = (t + m * P) >> (W29 * N29)
                assert (t + m * P) % R29 == 0 and abs(v) < MUL_BOUND * P
            else:
                v = lin29_exact(regs, pay)
                assert abs(v) < (RED_BOUND if pay.reduce else 1 << 20) * P, (v // P, pay.reduce)
            assert dst >= N_IN or abs(v) < IO_BOUND * P
            new[dst] = v
        regs.update(new)


def run29(prog, regs):
    """selftest adapter: canonical values in, canonical values out; inside, random representatives with |v| < IO_BOUND p"""
    rnd = random.Random(len(prog) * 7919 + 1)
    def rep(v):
        k = rnd.randrange(-IO_BOUND, IO_BOUND) if rnd.random() < 0.7 else rnd.choice((-IO_BOUND, IO_BOUND - 1))
        return v * R29 % P + k * P
    enc = {k: rep(v) for k, v in regs.items()}
    run29_exact(prog, enc)
    rinv = pow(R29, -1, P)
    for k, v in enc.items():
        regs[k] = v * rinv % P


def mul_srcs(ops):
    return [r for o in ops for r, _ in o]


def reallocate(prog, n_inputs):
    """Register reuse.  The builders number their temporaries in SSA fashion (a fresh register per instruction); here they are
    packed by a linear scan over the levels: a temporary's register is free again from the level AFTER its last read (a level may
    not write a register that another instruction of the same level still reads).  The register file of a check shrinks, so more
    checks fit one CTA's shared memory (many-tuple kernel) -- registers below n_inputs (inputs / outputs) keep their numbers."""
    srcs_of = lambda kind, pay: mul_srcs(pay[0]) if kind == "MUL" else [r for r, _, _ in pay]
    last_use = {}
    for lv, (kind, ins) in enumerate(prog):
        for _, dst, pay in ins:
            for r in srcs_of(kind, pay):
                last_use[r] = lv
    phys, free, next_phys, busy_until = {}, [], n_inputs, {}
    out = []
    for lv, (kind, ins) in enumerate(prog):
        for r, until in list(busy_until.items()):
            if until < lv:
                free.append(phys[r]); del busy_until[r]
        free.sort()
        new_ins = []
        for k, dst, pay in ins:
            if dst >= n_inputs:
                if free:
                    p = free.pop(0)
                else:
                    p = next_phys; next_phys += 1
                phys[dst] = p
                busy_until[dst] = last_use.get(dst, lv)
            new_ins.append((k, dst, pay))
        out.append((kind, new_ins))
    m = lambda r: phys.get(r, r)
    res = []
    for kind, ins in out:
        mapped = []
        for k, dst, pay in ins:
            if kind == "MUL":
                ops, neg = pay
                npay = ([[(m(r), minus) for r, minus in o] for o in ops], neg)
            else:
                npay = type(pay)((m(r), ng, db) for r, ng, db in pay)
                if isinstance(pay, Terms):
                    npay.reduce = pay.reduce
            mapped.append((k, m(dst), npay))
        res.append((kind, mapped))
    return res


def check_hazards(prog, n_inputs):
    """within a level no instruction may read a register written in the same level"""
    for kind, ins in prog:
        written = set(d for _, d, _ in ins)
        assert len(written) == len(ins), "two instructions of a level write the same register"
        for _, d, pay in ins:
            srcs = mul_srcs(pay[0]) if kind == "MUL" else [r for r, _, _ in pay]
            assert not ((set(srcs) - {d}) & written), "read/write hazard inside a level"


# ------------------------------------------------------------------------------------------ symbolic tower
class F2:
    def __init__(self, c0, c1): self.c0, self.c1 = c0, c1
    def __add__(s, o): return F2(s.c0 + o.c0, s.c1 + o.c1)
    def __sub__(s, o): return F2(s.c0 - o.c0, s.c1 - o.c1)
    def neg(s): return F2(-s.c0, -s.c1)
    def dbl(s): return F2(s.c0.scale(2), s.c1.scale(2))
    def conj(s): return F2(s.c0, -s.c1)
    def mul_xi(s): return F2(s.c0 - s.c1, s.c0 + s.c1)
    def mul(s, o, B): return F2(B.mul(s.c0, o.c0, s.c1, o.c1, neg=True), B.mul(s.c0, o.c1, s.c1, o.c0))
    def sqr(s, B): return F2(B.mul(s.c0 + s.c1, s.c0 - s.c1), B.mul(s.c0, s.c1).scale(2))
    def mul_fp(s, k, B): return F2(B.mul(s.c0, k), B.mul(s.c1, k))


class F6:
    def __init__(self, c0, c1, c2): self.c0, self.c1, self.c2 = c0, c1, c2
    def __add__(s, o): return F6(s.c0 + o.c0, s.c1 + o.c1, s.c2 + o.c2)
    def __sub__(s, o): return F6(s.c0 - o.c0, s.c1 - o.c1, s.c2 - o.c2)
    def neg(s): return F6(s.c0.neg(), s.c1.neg(), s.c2.neg())
    def mul_v(s): return F6(s.c2.mul_xi(), s.c0, s.c1)
    def mul(a, b, B):
        t0, t1, t2 = a.c0.mul(b.c0, B), a.c1.mul(b.c1, B), a.c2.mul(b.c2, B)
        r0 = t0 + ((a.c1 + a.c2).mul(b.c1 + b.c2, B) - t1 - t2).mul_xi()
        r1 = (a.c0 + a.c1).mul(b.c0 + b.c1, B) - t0 - t1 + t2.mul_xi()
        r2 = (a.c0 + a.c2).mul(b.c0 + b.c2, B) - t0 - t2 + t1
        return F6(r0, r1, r2)


class F12:
    def __init__(self, c0, c1): self.c0, self.c1 = c0, c1
    def mul(a, b, B):
        t0, t1 = a.c0.mul(b.c0, B), a.c1.mul(b.c1, B)
        m = (a.c0 + a.c1).mul(b.c0 + b.c1, B) - t0 - t1
        return F12(t0 + t1.mul_v(), m)
    def sqr(a, B):
        ab = a.c0.mul(a.c1, B)
        s = (a.c0 + a.c1).mul(a.c0 + a.c1.mul_v(), B) - ab - ab.mul_v()
        return F12(s, ab + ab)
    def conj(a): return F12(a.c0, a.c1.neg())
    def flat(a): return [a.c0.c0.c0, a.c0.c0.c1, a.c0.c1.c0, a.c0.c1.c1, a.c0.c2.c0, a.c0.c2.c1,
                         a.c1.c0.c0, a.c1.c0.c1, a.c1.c1.c0, a.c1.c1.c1, a.c1.c2.c0, a.c1.c2.c1]


def f12_in(B, base):
    v = [B.input(base + i) for i in range(12)]
    return F12(F6(F2(v[0], v[1]), F2(v[2], v[3]), F2(v[4], v[5])), F6(F2(v[6], v[7]), F2(v[8], v[9]), F2(v[10], v[11])))


def f2_in(B, base):
    return F2(B.input(base), B.input(base + 1))


def out12(B, x, base):
    for i, v in enumerate(x.flat()):
        B.output(v, base + i)


# Register-file layout shared with vliw.cuh -------------------------------------------------------------------
# pairing programs: F = regs 0..11 (the Miller / exponentiation accumulator), G = 12..23, H = 24..35 (second /
# third Fp12 operand or result), line inputs 36..47: two lines (A, Bx, Cy as Fp2: 6 Fp each), constants 48..57
# (Frobenius coefficients xi^(k(p-1)/6), k = 1..5, as Fp2), scratch from 64.
RF = 12
RG = 12
RH = 24
RL = 36
RC = 48
RP = 58          # xP1, yP1, xP2, yP2 (G1 arguments of the two pairs)
N_IN = 64


def prog_f12_mul():        # F <- F * G
    B = BUILDER("f12_mul", N_IN)
    out12(B, f12_in(B, 0).mul(f12_in(B, RG), B), 0)
    return B


def prog_f12_sqr():        # F <- F^2
    B = BUILDER("f12_sqr", N_IN)
    out12(B, f12_in(B, 0).sqr(B), 0)
    return B


def prog_f12_sqr_k(k):     # F <- F^(2^k): k squarings in one program; the lazy additions fuse each output level with the next
    def mk():              # squaring's operand level, so a squaring costs 2 levels instead of 3
        B = BUILDER("f12_sqr%d" % k, N_IN)
        x = f12_in(B, 0)
        for _ in range(k):
            x = x.sqr(B)
        out12(B, x, 0)
        return B
    return mk


def prog_miller_step():    # F <- F^2 * line1(P1) * line2(P2)   (one doubling step of the Miller loop, both pairs live)
    B = BUILDER("miller_step", N_IN)
    f2 = f12_in(B, 0).sqr(B)
    L = sparse_mul(line_in(B, 0), line_in(B, 1), B)
    out12(B, f2.mul(L, B), 0)
    return B


def prog_miller_add():     # F <- F * line1(P1) * line2(P2)     (an addition step)
    B = BUILDER("miller_add", N_IN)
    L = sparse_mul(line_in(B, 0), line_in(B, 1), B)
    out12(B, f12_in(B, 0).mul(L, B), 0)
    return B


def fp4_square(a, b, B):
    """(a + b s)^2 in Fp4 = Fp2[s]/(s^2 - xi): (a^2 + xi b^2, 2ab)"""
    t0, t1 = a.sqr(B), b.sqr(B)
    return t0 + t1.mul_xi(), (a + b).sqr(B) - t0 - t1


def cyclotomic_sqr(f, fr, B):
    """Granger-Scott squaring for f in the cyclotomic subgroup (f^(p^4-p^2+1) = 1).  With Fp12 = Fp4[w]/(w^3 - s), s = w^3,
    f = A + B w + C w^2, A = z0 + z1 s, B = z2 + z3 s, C = z4 + z5 s:
        f^2 = (3A^2 - 2 conj A) + (3 s C^2 + 2 conj B) w + (3B^2 - 2 conj C) w^2.
    f = the input as lazy linear combinations (feeds the multiplication operands), fr = the same values as plain
    registers (used for the +-2z terms, so that coefficients do not compound over a chain of squarings)."""
    z0, z4, z3 = f.c0.c0, f.c0.c1, f.c0.c2
    z2, z1, z5 = f.c1.c0, f.c1.c1, f.c1.c2
    r0, r4, r3 = fr.c0.c0, fr.c0.c1, fr.c0.c2
    r2, r1, r5 = fr.c1.c0, fr.c1.c1, fr.c1.c2
    a0, a1 = fp4_square(z0, z1, B)
    b0, b1 = fp4_square(z2, z3, B)
    c0, c1 = fp4_square(z4, z5, B)
    three = lambda x: x + x + x
    n0 = three(a0) - r0.dbl(); n1 = three(a1) + r1.dbl()
    n4 = three(b0) - r4.dbl(); n5 = three(b1) + r5.dbl()
    n2 = three(c1.mul_xi()) + r2.dbl(); n3 = three(c0) - r3.dbl()
    return F12(F6(n0, n4, n3), F6(n2, n1, n5))


def materialize12(B, x):
    m = lambda v: Val({B.materialize(v): 1})
    m2 = lambda a: F2(m(a.c0), m(a.c1))
    return F12(F6(m2(x.c0.c0), m2(x.c0.c1), m2(x.c0.c2)), F6(m2(x.c1.c0), m2(x.c1.c1), m2(x.c1.c2)))


def prog_cyc_sqr_k(k):     # F <- F^(2^k) for F in the cyclotomic subgroup (hard part of the final exponentiation)
    def mk():
        B = BUILDER("cyc_sqr%d" % k, N_IN)
        x = xr = f12_in(B, 0)
        for i in range(k):
            x = cyclotomic_sqr(x, xr, B)
            if i + 1 < k:
                xr = materialize12(B, x)     # same level as the next squaring's operand sums
        out12(B, x, 0)
        return B
    return mk


def sparse014(A, Bx, Cy):
    z = Val()
    return F12(F6(A, Bx, F2(z, z)), F6(F2(z, z), Cy, F2(z, z)))


def line_in(B, j):
    """line j (raw A, B, C at RL + 6j) evaluated at P_j = (regs RP+2j, RP+2j+1): A + (B xP) v + (C yP) vw"""
    A, Bc, Cc = f2_in(B, RL + 6 * j), f2_in(B, RL + 6 * j + 2), f2_in(B, RL + 6 * j + 4)
    xP, yP = B.input(RP + 2 * j), B.input(RP + 2 * j + 1)
    return sparse014(A, Bc.mul_fp(xP, B), Cc.mul_fp(yP, B))


def prog_sqr_lines():      # F <- F^2 ; G <- line1(P1) * line2(P2)
    B = BUILDER("sqr_lines", N_IN)
    f2 = f12_in(B, 0).sqr(B)
    out12(B, f2, 0)
    out12(B, sparse_mul(line_in(B, 0), line_in(B, 1), B), RG)
    return B


def prog_lines():          # G <- line1(P1) * line2(P2)
    B = BUILDER("lines", N_IN)
    out12(B, sparse_mul(line_in(B, 0), line_in(B, 1), B), RG)
    return B


def prog_line1():          # G <- line1(P1) as a full Fp12 element (the other pair is skipped)
    B = BUILDER("line1", N_IN)
    out12(B, line_in(B, 0), RG)
    return B


def prog_conj_g():         # G <- conj(G)
    B = BUILDER("conj_g", N_IN)
    out12(B, f12_in(B, RG).conj(), RG)
    return B


def sparse_mul(a, b, B):
    """(a0 + a1 v + a4 vw)(b0 + b1 v + b4 vw) written out (zero coefficients skipped)"""
    a0, a1, a4 = a.c0.c0, a.c0.c1, a.c1.c1
    b0, b1, b4 = b.c0.c0, b.c0.c1, b.c1.c1
    c0 = a0.mul(b0, B) + a4.mul(b4, B).mul_xi()
    c1 = a0.mul(b1, B) + a1.mul(b0, B)
    c2 = a1.mul(b1, B)
    d0 = F2(Val(), Val())
    d1 = a0.mul(b4, B) + a4.mul(b0, B)
    d2 = a1.mul(b4, B) + a4.mul(b1, B)
    return F12(F6(c0, c1, c2), F6(d0, d1, d2))


def prog_conj():           # F <- conj(F)
    B = BUILDER("conj", N_IN)
    out12(B, f12_in(B, 0).conj(), 0)
    return B


def frob(B, a):
    g = [None] + [f2_in(B, RC + 2 * (k - 1)) for k in range(1, 6)]
    c = a
    return F12(F6(c.c0.c0.conj(), c.c0.c1.conj().mul(g[2], B), c.c0.c2.conj().mul(g[4], B)),
               F6(c.c1.c0.conj().mul(g[1], B), c.c1.c1.conj().mul(g[3], B), c.c1.c2.conj().mul(g[5], B)))


def prog_frob():           # G <- frob(F)
    B = BUILDER("frob", N_IN)
    out12(B, frob(B, f12_in(B, 0)), RG)
    return B


def prog_frob2():          # G <- frob(frob(F))
    B = BUILDER("frob2", N_IN)
    out12(B, frob(B, frob(B, f12_in(B, 0))), RG)
    return B


def prog_inv_prep():
    """Fp12 inversion, part 1: F = a0 + a1 w.  t = a0^2 - v a1^2 (Fp6); its Fp6 inverse needs the Fp2 norm
    n2 = t0*c0 + xi(t2*c1 + t1*c2) and then the Fp norm n = n2.c0^2 + n2.c1^2.  Outputs: H[0..5] = (c0,c1,c2)
    cofactors, H[6..7] = n2, H[8] = n (to be inverted by the caller), G = copy of F."""
    B = BUILDER("inv_prep", N_IN)
    a = f12_in(B, 0)
    t = a.c0.mul(a.c0, B) - a.c1.mul(a.c1, B).mul_v()
    c0 = t.c0.sqr(B) - t.c1.mul(t.c2, B).mul_xi()
    c1 = t.c2.sqr(B).mul_xi() - t.c0.mul(t.c1, B)
    c2 = t.c1.sqr(B) - t.c0.mul(t.c2, B)
    n2 = t.c0.mul(c0, B) + (t.c2.mul(c1, B) + t.c1.mul(c2, B)).mul_xi()
    n = B.mul(n2.c0, n2.c0, n2.c1, n2.c1)
    for i, v in enumerate([c0.c0, c0.c1, c1.c0, c1.c1, c2.c0, c2.c1, n2.c0, n2.c1, n]):
        B.output(v, RH + i)
    out12(B, a, RG)
    return B


def prog_inv_finish():
    """part 2: H[8] now holds 1/n.  n2^-1 = conj(n2)/n ; t^-1 = (c0,c1,c2) * n2^-1 ; F <- (a0 t^-1, -a1 t^-1)
    with a = G."""
    B = BUILDER("inv_finish", N_IN)
    a = f12_in(B, RG)
    c = [f2_in(B, RH), f2_in(B, RH + 2), f2_in(B, RH + 4)]
    n2, ninv = f2_in(B, RH + 6), B.input(RH + 8)
    n2i = F2(B.mul(n2.c0, ninv), -B.mul(n2.c1, ninv))
    ti = F6(c[0].mul(n2i, B), c[1].mul(n2i, B), c[2].mul(n2i, B))
    out12(B, F12(a.c0.mul(ti, B), a.c1.mul(ti, B).neg()), 0)
    return B


def prog_copy(src, dst, name):
    B = BUILDER(name, N_IN)
    for i in range(12):
        B.output(B.input(src + i), dst + i)
    return B


# G1 Jacobian programs for the MSM recombination: point X,Y,Z = regs 0,1,2 ; second point 3,4,5
def prog_g1_dbl():
    B = BUILDER("g1_dbl", N_IN)
    X, Y, Z = B.input(0), B.input(1), B.input(2)
    A, Bq = B.mul(X, X), B.mul(Y, Y)
    C = B.mul(Bq, Bq)
    t = X + Bq
    D = (B.mul(t, t) - A - C).scale(2)
    E = A.scale(3)
    F = B.mul(E, E)
    X3 = F - D.scale(2)
    Y3 = B.mul(E, D - X3) - C.scale(8)
    Z3 = B.mul(Y, Z).scale(2)
    B.output(X3, 0); B.output(Y3, 1); B.output(Z3, 2)
    return B


def prog_g1_add():
    """generic Jacobian addition (0,1,2) += (3,4,5); the caller handles identities / equal points.
    Also leaves H = U2-U1 in reg 6 and R = S2-S1 in reg 7 for the caller's special-case test."""
    B = BUILDER("g1_add", N_IN)
    X1, Y1, Z1, X2, Y2, Z2 = (B.input(i) for i in range(6))
    Z1Z1, Z2Z2 = B.mul(Z1, Z1), B.mul(Z2, Z2)
    U1, U2 = B.mul(X1, Z2Z2), B.mul(X2, Z1Z1)
    S1, S2 = B.mul(B.mul(Y1, Z2Z2), Z2), B.mul(B.mul(Y2, Z1Z1), Z1)
    H, Rr = U2 - U1, S2 - S1
    H2 = B.mul(H, H)
    H3, UH2 = B.mul(H2, H), B.mul(U1, H2)
    X3 = B.mul(Rr, Rr) - H3 - UH2.scale(2)
    Y3 = B.mul(Rr, UH2 - X3) - B.mul(S1, H3)
    Z3 = B.mul(B.mul(Z1, Z2), H)
    B.output(X3, 0); B.output(Y3, 1); B.output(Z3, 2); B.output(H, 6); B.output(Rr, 7)
    return B


PROGRAMS = [prog_cyc_sqr_k(1), prog_f12_mul, prog_f12_sqr, prog_sqr_lines, prog_lines, prog_line1, prog_conj, prog_conj_g, prog_frob, prog_frob2,
            prog_inv_prep, prog_inv_finish, prog_g1_dbl, prog_g1_add]


# ------------------------------------------------------------------------------------------ python interpreter
def run(prog, regs):
    for kind, ins in prog:
        new = {}
        for _, dst, pay in ins:
            if kind == "MUL":
                (ops, neg) = pay
                val = lambda o: sum(-regs[r] if minus else regs[r] for r, minus in o)
                v = val(ops[0]) * val(ops[1])
                if len(ops) == 4:
                    w = val(ops[2]) * val(ops[3])
                    v = v - w if neg else v + w
            else:
                v = 0
                for r, ng, db in pay:
                    t = regs[r] * (2 if db else 1)
                    v = v - t if ng else v + t
            new[dst] = v % P
        regs.update(new)


def selftest(progs, run=None):
    run = run or globals()['run']
    rnd = random.Random(11)
    def rnd12():
        return tuple(tuple((rnd.randrange(P), rnd.randrange(P)) for _ in range(3)) for _ in range(2))
    def flat(a):
        return [x for c6 in a for c2 in c6 for x in c2]
    def unflat(v):
        return ((tuple(v[0:2]), tuple(v[2:4]), tuple(v[4:6])), (tuple(v[6:8]), tuple(v[8:10]), tuple(v[10:12])))
    G6 = [R.f2_pow(R.XI, k * (P - 1) // 6) for k in range(6)]
    def fresh():
        regs = {i: rnd.randrange(P) for i in range(4096)}
        for k in range(1, 6):
            regs[RC + 2 * (k - 1)], regs[RC + 2 * (k - 1) + 1] = G6[k]
        return regs
    for _ in range(3):
        f, g = rnd12(), rnd12()
        regs = fresh()
        for i, v in enumerate(flat(f)): regs[i] = v
        for i, v in enumerate(flat(g)): regs[RG + i] = v
        r2 = dict(regs); run(progs["f12_mul"], r2)
        assert unflat([r2[i] for i in range(12)]) == R.f12_mul(f, g)
        r2 = dict(regs); run(progs["f12_sqr"], r2)
        assert unflat([r2[i] for i in range(12)]) == R.f12_sqr(f)
        r2 = dict(regs); run(progs["conj"], r2)
        assert unflat([r2[i] for i in range(12)]) == R.f12_conj(f)
        # cyclotomic squarings: on an element of the cyclotomic subgroup g = f^((p^6-1)(p^2+1))
        g1_ = R.f12_mul(R.f12_conj(f), R.f12_inv(f))
        gc = R.f12_mul(R.f12_frob(R.f12_frob(g1_)), g1_)
        rc = dict(regs)
        for i, v in enumerate(flat(gc)): rc[i] = v
        for k in (1,):
            r2 = dict(rc); run(progs["cyc_sqr%d" % k], r2)
            want = gc
            for _ in range(k): want = R.f12_sqr(want)
            assert unflat([r2[i] for i in range(12)]) == want
        r2 = dict(regs); run(progs["frob"], r2)
        assert unflat([r2[RG + i] for i in range(12)]) == R.f12_frob(f)
        r2 = dict(regs); run(progs["frob2"], r2)
        assert unflat([r2[RG + i] for i in range(12)]) == R.f12_frob(R.f12_frob(f))
        # lines
        lines = [(rnd.randrange(P), rnd.randrange(P)) for _ in range(6)]
        for i, (a, b) in enumerate(lines):
            regs[RL + 2 * i], regs[RL + 2 * i + 1] = a, b
        Z = R.F2_ZERO
        pc = [rnd.randrange(P) for _ in range(4)]
        for i in range(4): regs[RP + i] = pc[i]
        sc = lambda v, k: (v[0] * k % P, v[1] * k % P)
        l1 = ((lines[0], sc(lines[1], pc[0]), Z), (Z, sc(lines[2], pc[1]), Z))
        l2 = ((lines[3], sc(lines[4], pc[2]), Z), (Z, sc(lines[5], pc[3]), Z))
        r2 = dict(regs); run(progs["sqr_lines"], r2)
        assert unflat([r2[i] for i in range(12)]) == R.f12_sqr(f)
        assert unflat([r2[RG + i] for i in range(12)]) == R.f12_mul(l1, l2)
        r2 = dict(regs); run(progs["lines"], r2)
        assert unflat([r2[RG + i] for i in range(12)]) == R.f12_mul(l1, l2)

        r2 = dict(regs); run(progs["line1"], r2)
        assert unflat([r2[RG + i] for i in range(12)]) == l1
        r2 = dict(regs); run(progs["conj_g"], r2)
        assert unflat([r2[RG + i] for i in range(12)]) == R.f12_conj(g)
        # inversion
        r2 = dict(regs); run(progs["inv_prep"], r2)
        r2[RH + 8] = pow(r2[RH + 8], P - 2, P)
        run(progs["inv_finish"], r2)
        assert unflat([r2[i] for i in range(12)]) == R.f12_inv(f)
        # G1
        p1 = R.g1_mul(R.G1_GEN, rnd.randrange(R.Q)); p2 = R.g1_mul(R.G1_GEN, rnd.randrange(R.Q))
        z1, z2 = rnd.randrange(1, P), rnd.randrange(1, P)
        regs[0], regs[1], regs[2] = p1[0] * z1 * z1 % P, p1[1] * z1 ** 3 % P, z1
        regs[3], regs[4], regs[5] = p2[0] * z2 * z2 % P, p2[1] * z2 ** 3 % P, z2
        def aff(r):
            zi = pow(r[2], P - 2, P); return (r[0] * zi * zi % P, r[1] * zi ** 3 % P)
        r2 = dict(regs); run(progs["g1_dbl"], r2)
        assert aff(r2) == R.g1_add(p1, p1)
        r2 = dict(regs); run(progs["g1_add"], r2)
        assert aff(r2) == R.g1_add(p1, p2)
    print("python self-test of all programs: ok")


def tables_of(progs):
    mul_tab, lin_tab, term_tab, level_tab, prog_tab, names, stats = [], [], [], [], [], [], []
    for name, prog in progs.items():
        first_level = len(level_tab)
        n_regs = N_IN
        nmul = nlin = 0
        for kind, ins in prog:
            if kind == "MUL":
                level_tab.append((1, len(ins), len(mul_tab)))
                for _, dst, (ops, neg) in ins:
                    ops = list(ops) + [[]] * (4 - len(ops))
                    signs = 0
                    row = [dst]
                    for i, terms in enumerate(ops):
                        slots = [r for r, _ in terms] + [0xffff] * (4 - len(terms))
                        row += slots
                        for j, (_, minus) in enumerate(terms):
                            signs |= (1 << (4 * i + j)) if minus else 0
                    mul_tab.append(tuple(row + [signs, 1 if neg else 0]))
                    n_regs = max(n_regs, dst + 1)
                nmul += len(ins)
            else:
                level_tab.append((0, len(ins), len(lin_tab)))
                for _, dst, terms in ins:
                    lin_tab.append((dst, len(term_tab), len(terms)))
                    for r, ng, db in terms:
                        term_tab.append(r | (1 << 14 if ng else 0) | (1 << 15 if db else 0))
                    n_regs = max(n_regs, dst + 1)
                nlin += len(ins)
        prog_tab.append((first_level, len(level_tab) - first_level, n_regs))
        names.append(name)
        stats.append((name, len(level_tab) - first_level, nmul, nlin, n_regs))
    return mul_tab, lin_tab, term_tab, level_tab, prog_tab, names, stats


def emit(sets, path):
    """sets: {"lat": programs for ONE check on one CTA (latency: sums are formed once, by LIN levels, in parallel),
              "thr": programs for many checks in lockstep (throughput: multiplication operands of up to 4 terms are summed by
                     the multiplying thread, which removes the operand LIN levels and their barriers)}"""
    out = ["// GENERATED by tools/gen_vliw.py -- do not edit.  Level-scheduled Fp programs for vliw.cuh.",
           "#pragma once", "#include <stdint.h>", "namespace kzgb200 { namespace vliw {",
           "constexpr int kRegF = 0, kRegG = %d, kRegH = %d, kRegLines = %d, kRegConst = %d, kRegP = %d, kNumInputRegs = %d;" % (RG, RH, RL, RC, RP, N_IN),
           "// MUL instruction (19 x u16): dst, then four operands of four register slots each (0xffff = unused; the first slot of an",
           "// operand is always a positive term; the third operand unused: single product), then the sign bits: bit 4i+j = slot j of",
           "// operand i is subtracted; last word: 1 = the second product as a whole is subtracted",
           "// LIN instruction: dst, first term index, term count; a term = reg | neg << 14 | dbl << 15",
           "struct Level { uint16_t kind /*0 LIN, 1 MUL*/, count; uint32_t first; };",
           "struct Program { uint16_t first_level, n_levels, n_regs; };"]
    first = True
    maxes = [0, 0, 0, 0]
    for tag, progs in sets.items():
        mul_tab, lin_tab, term_tab, level_tab, prog_tab, names, stats = tables_of(progs)
        if first:
            out.append("enum ProgramId { " + ", ".join("kProg_%s = %d" % (n, i) for i, n in enumerate(names)) + ", kNumPrograms = %d };" % len(names))
            first = False
        maxes = [max(a, b) for a, b in zip(maxes, [len(mul_tab), len(lin_tab), len(term_tab), len(level_tab)])]
        out.append("namespace %s {" % tag)
        out.append("constexpr int kMaxRegs = %d;" % max(p[2] for p in prog_tab))
        out.append("constexpr int kMaxRegsNoSqrLines = %d;   // the multi-group form runs f12_sqr and lines separately: smaller register files" %
                   max(p[2] for p, nm in zip(prog_tab, names) if nm != "sqr_lines"))
        out.append("constexpr int kNumMul = %d, kNumLin = %d, kNumTerm = %d, kNumLevel = %d;" % (len(mul_tab), len(lin_tab), len(term_tab), len(level_tab)))
        row = lambda m: "{" + ",".join(str(x) for x in m) + "}"
        for qual, pre in (("static __device__ const", "d"), ("static const", "h")):
            if pre == "h":
                out.append("#ifndef __CUDA_ARCH__")
            out.append("%s uint16_t %s_mul[%d][19] = {%s};" % (qual, pre, len(mul_tab), ",".join(row(m) for m in mul_tab)))
            out.append("%s uint32_t %s_lin[%d][3] = {%s};" % (qual, pre, len(lin_tab), ",".join(row(m) for m in lin_tab)))
            out.append("%s uint16_t %s_term[%d] = {%s};" % (qual, pre, len(term_tab), ",".join(str(t) for t in term_tab)))
            out.append("%s Level %s_level[%d] = {%s};" % (qual, pre, len(level_tab), ",".join(row(l) for l in level_tab)))
            out.append("%s Program %s_prog[%d] = {%s};" % (qual, pre, len(prog_tab), ",".join(row(p) for p in prog_tab)))
            if pre == "h":
                out.append("#endif")
        out.append("}  // namespace %s" % tag)
        print("-- %s" % tag)
        for st in stats:
            print("%-14s levels %2d  MUL %3d  LIN %3d  regs %3d" % st)
    out.append("constexpr int kNumMulMax = %d, kNumLinMax = %d, kNumTermMax = %d, kNumLevelMax = %d;" % tuple(maxes))
    out.append("}}  // namespace kzgb200::vliw")
    open(path, "w").write("\n".join(out) + "\n")


OP_RUN, OP_COPY, OP_LINES, OP_INV, OP_TICK = range(5)
BLS_X_ABS = 0xd201000000010000


def pairing_script(names, max_regs, two_pairs, part="all"):
    """The pairing check e(P1, Q1) e(P2, Q2) == 1 (one pair when the other G1 argument is the identity) as a straight list of
    engine steps -- run a program, copy an Fp12 slot, load the line coefficients of Miller step k, invert one register, stamp a
    profiling tick -- so that the kernel contains ONE interpreter loop with the two instruction executors inlined once.
    Same sequence as vliw.cuh coop_pairing_product_is_one: Miller loop with precomputed lines, then f^(3(p^12-1)/r) with the
    hard part (x-1)^2 (x+p)(x^2+p^2-1) + 3 on cyclotomic squarings.
    part = "miller": the Miller loop alone, up to and including tick 2 (f left in the F slot, conjugated); part = "fe": the final
    exponentiation alone, from the F slot (the batch verifier's split tail multiplies per-window Miller values in between)."""
    P = {n: i for i, n in enumerate(names)}
    S = [max_regs + 12 * i for i in range(5)]
    F, G = 0, RG
    s = []
    run = lambda n: s.append((OP_RUN, P[n], 0))
    copy = lambda d, src: s.append((OP_COPY, d, src))
    tick = lambda i: s.append((OP_TICK, i, 0))
    def exp_by_x(base):
        copy(F, base)
        pending = 0
        for bit in range(62, -1, -1):
            pending += 1
            if (BLS_X_ABS >> bit) & 1:
                for _ in range(pending): run("cyc_sqr1")
                pending = 0
                copy(G, base); run("f12_mul")
        for _ in range(pending): run("cyc_sqr1")
        run("conj")
    tick(1)
    k = 0
    for bit in range(62, -1, -1):
        s.append((OP_LINES, k, 0)); k += 1
        if two_pairs:
            run("sqr_lines")
        else:
            run("f12_sqr"); run("line1")
        run("f12_mul")
        if (BLS_X_ABS >> bit) & 1:
            s.append((OP_LINES, k, 0)); k += 1
            run("lines" if two_pairs else "line1"); run("f12_mul")
    run("conj"); tick(2)
    copy(S[0], F); run("inv_prep"); s.append((OP_INV, 0, 0)); run("inv_finish")
    copy(G, F); copy(F, S[0]); run("conj"); run("f12_mul")          # f0^(p^6-1)
    run("frob2"); run("f12_mul"); copy(S[0], F); tick(3)            # S0 = f = f0^((p^6-1)(p^2+1))
    exp_by_x(S[0]); copy(G, S[0]); run("conj_g"); run("f12_mul"); copy(S[1], F)          # f^(x-1)
    exp_by_x(S[1]); copy(G, S[1]); run("conj_g"); run("f12_mul"); copy(S[1], F)          # a = f^((x-1)^2)
    exp_by_x(S[1]); copy(S[2], F); copy(F, S[1]); run("frob"); copy(F, S[2]); run("f12_mul"); copy(S[2], F)   # b = a^(x+p)
    exp_by_x(S[2]); copy(S[3], F); exp_by_x(S[3]); copy(S[4], F)                          # b^(x^2)
    copy(F, S[2]); run("frob2"); copy(F, S[4]); run("f12_mul")
    copy(G, S[2]); run("conj_g"); run("f12_mul"); copy(S[4], F)                           # c = b^(x^2+p^2-1)
    copy(F, S[0]); run("f12_sqr"); copy(G, S[0]); run("f12_mul")                          # f^3
    copy(G, S[4]); run("f12_mul"); tick(4)                                                # c f^3
    cut = s.index((OP_TICK, 2, 0)) + 1
    s = s[:cut] if part == "miller" else (s[cut:] if part == "fe" else s)
    return [op | a << 8 | b << 20 for op, a, b in s]


def emit29(progs, path):
    """tables of the headroom programs (vliw29.cuh): MUL row = {dst | a << 16, b | c << 16, d | flags << 16, 0} with flags bit 0 =
    dual product, bit 1 = the second product is subtracted; LIN row = {dst, first term, term count, reduce}; a term = byte offset of the source register | coefficient (+-1, +-2) << 16"""
    mul_tab, lin_tab, term_tab, level_tab, prog_tab, names = [], [], [], [], [], []
    print("-- lat29")
    for name, prog in progs.items():
        first_level, n_regs, nmul, nlin = len(level_tab), N_IN, 0, 0
        for kind, ins in prog:
            if kind == "MUL":
                level_tab.append((1, len(ins), len(mul_tab)))
                for _, dst, (ops, neg) in ins:
                    r = [o[0][0] for o in ops] + [0xffff] * (4 - len(ops))
                    flags = (1 if len(ops) == 4 else 0) | (2 if neg else 0)
                    mul_tab.append((dst | r[0] << 16, r[1] | r[2] << 16, r[3] | flags << 16, 0))
                    n_regs = max(n_regs, dst + 1)
                nmul += len(ins)
            else:
                level_tab.append((0, len(ins), len(lin_tab)))
                for _, dst, terms in ins:
                    lin_tab.append((dst, len(term_tab), len(terms), 1 if terms.reduce else 0))
                    for r, ng, db in terms:
                        coef = (2 if db else 1) * (-1 if ng else 1)
                        term_tab.append((r * 64) | ((coef & 0xffff) << 16))
                    n_regs = max(n_regs, dst + 1)
                nlin += len(ins)
        prog_tab.append((first_level, len(level_tab) - first_level, n_regs))
        names.append(name)
        print("%-14s levels %2d  MUL %3d  LIN %3d  regs %3d" % (name, len(level_tab) - first_level, nmul, nlin, n_regs))
    row = lambda m: "{" + ",".join("%du" % x if x > 0x7fffffff else str(x) for x in m) + "}"
    out = ["// GENERATED by tools/gen_vliw.py -- do not edit.  Level-scheduled Fp programs for vliw29.cuh (29-bit limbs, headroom instead of",
           "// reductions; the bounds that make this sound are tracked and asserted by the generator).",
           "#pragma once", "#include <stdint.h>", "namespace kzgb200 { namespace vliw29 {",
           "constexpr int kRegF = 0, kRegG = %d, kRegH = %d, kRegLines = %d, kRegConst = %d, kRegP = %d, kNumInputRegs = %d;" % (RG, RH, RL, RC, RP, N_IN),
           "constexpr int kIoBound = %d;   // every register at a program boundary holds a value below kIoBound * p" % IO_BOUND,
           "struct Level { uint16_t kind /*0 LIN, 1 MUL*/, count; uint32_t first; };",
           "struct Program { uint16_t first_level, n_levels, n_regs; };",
           "enum ProgramId { " + ", ".join("kProg_%s = %d" % (n, i) for i, n in enumerate(names)) + ", kNumPrograms = %d };" % len(names),
           "constexpr int kMaxRegs = %d;" % max(p[2] for p in prog_tab),
           "constexpr int kNumMul = %d, kNumLin = %d, kNumTerm = %d, kNumLevel = %d;" % (len(mul_tab), len(lin_tab), len(term_tab), len(level_tab))]
    for qual, pre in (("static __device__ const", "d"), ("static const", "h")):
        if pre == "h":
            out.append("#ifndef __CUDA_ARCH__")
        out.append("%s uint32_t %s_mul[%d][4] = {%s};" % (qual, pre, len(mul_tab), ",".join(row(m) for m in mul_tab)))
        out.append("%s uint32_t %s_lin[%d][4] = {%s};" % (qual, pre, len(lin_tab), ",".join(row(m) for m in lin_tab)))
        out.append("%s uint32_t %s_term[%d] = {%s};" % (qual, pre, len(term_tab), ",".join("%du" % t for t in term_tab)))
        out.append("%s Level %s_level[%d] = {%s};" % (qual, pre, len(level_tab), ",".join(row(l) for l in level_tab)))
        out.append("%s Program %s_prog[%d] = {%s};" % (qual, pre, len(prog_tab), ",".join(row(p) for p in prog_tab)))
        for tag, two, part in (("script2", True, "all"), ("script1", False, "all"),
                               ("miller2", True, "miller"), ("miller1", False, "miller"), ("final_exp", True, "fe")):
            sc = pairing_script(names, max(p[2] for p in prog_tab), two, part)
            if pre == "d":
                out.append("constexpr int kLen_%s = %d;" % (tag, len(sc)))
            out.append("%s uint32_t %s_%s[%d] = {%s};" % (qual, pre, tag, len(sc), ",".join(str(x) for x in sc)))
        if pre == "h":
            out.append("#endif")
    out.append("enum ScriptOp { kOpRun = %d, kOpCopy = %d, kOpLines = %d, kOpInv = %d, kOpTick = %d };   // step = op | a << 8 | b << 20" % (OP_RUN, OP_COPY, OP_LINES, OP_INV, OP_TICK))
    out.append("}}  // namespace kzgb200::vliw29")
    open(path, "w").write("\n".join(out) + "\n")


def build_all(max_operand_terms, builder=Builder):
    global MAX_OPERAND_TERMS, BUILDER
    MAX_OPERAND_TERMS = max_operand_terms
    BUILDER = builder
    progs = {}
    for mk in PROGRAMS:
        B = mk()
        prog = reallocate(B.finish(), N_IN)
        check_hazards(prog, N_IN)
        progs[B.name] = prog
    selftest(progs, run29 if builder is Builder29 else None)
    BUILDER = Builder
    return progs


if __name__ == "__main__":
    sets = {"lat": build_all(1), "thr": build_all(4)}
    lat29 = build_all(1, Builder29)
    if "--check" not in sys.argv:
        emit(sets, os.path.join(ROOT, "kzg_rs_b200", "csrc", "vliw_programs.cuh"))
        emit29(lat29, os.path.join(ROOT, "kzg_rs_b200", "csrc", "vliw29_programs.cuh"))
