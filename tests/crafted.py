"""Deterministic CRAFTED signatures that drive the verification kernels into the rare branches of the group law.

Honest or random signatures reach P + P, P - P or the point at infinity inside a double-scalar multiplication with probability
about 2^-128; a Byzantine validator reaches them on purpose.  Every case here is built so that one of those branches is taken,
with oracle/secp256k1.py as the reference of record.  All R used below are multiples t*G with a known t, so the key a recovery of
(z, r, s, v) yields is ((+-t) s - z) / r * G -- one scalar multiplication per case; tests/test_emul_crafted.py checks every one
of them against the oracle's own recover_pubkey.

Families (labels start with the family letter):
  A  forced (u1, u2, R): R = P for the base points of test_gpu_primitives.py::test_ecmult, u1 = a, u2 = b for its special pairs
     (r = P.x, s = b r, z = -a r): the recovery computes exactly a*G + b*P;
  B  final-combination collisions: R = kG, s = -z/k makes u1*G = u2*R (the split kernels' final addition doubles; the key is
     -2z/r * G), s = +z/k makes the sum the point at infinity (verdict 0); each with its high-s twin, for digests, payloads and
     committed seals;
  C  Booth-digit edges: u1, u2 from GLV halves on the window edges (0, +-1, +-8, 127, +-128, 129, all-0x80 bytes, 2^127, ...);
  D  known-key collisions: signatures of Q in {G, -G, lambda G, -lambda G, 2G, 0xC0FFEE G} with u1 = +-u2 (the generator and
     the key streams meet inside the comb walk) and u1*G = u2*Q (the known-key finish doubles).
Next to valid cases: the recovery id flipped (another key), the same signature claimed by another validator, r that is not an
abscissa, and r, s, v out of range.
"""
from __future__ import annotations

import functools
import random
from dataclasses import dataclass

import numpy as np

import workloads as wl
from oracle import coracle as co
from oracle import secp256k1 as ec

N, P = ec.N, ec.P
LAM = 0x5363AD4CC05C30E0A5261C028812645A122E22EA20816678DF02967C1B23BD72
ALL80 = int.from_bytes(b"\x80" * 16, "big")
# GLV halves on the window edges: the 4-bit windows of R (0, +-8), the 8-bit comb (+-128), Booth carries (127, 129, 255, 256)
HALVES = [0, 1, -1, 8, -8, 127, 128, -128, 129, 255, 256, 0x8000, ALL80, -ALL80, 2**127, 2**128 - 1, -(2**127) - 5, 0x7F80 << 64]
# base points P = d*G of test_gpu_primitives.py::test_ecmult and its special scalar pairs (a, b)
BASES = [("12345G", 12345), ("G", 1), ("-G", N - 1), ("2G", 2), ("lamG", LAM), ("-lamG", N - LAM), ("8G", 8), ("-8G", N - 8)]
SPECIAL = [(0, 0), (1, 0), (0, 1), (2, 0), (0, 2), (N - 1, 0), (0, N - 1), (1, N - 1), (5, 7), (N - 1, N - 1), (LAM, 0), (0, LAM),
           (N - LAM, LAM), (1, 1), (2, N - 1), (N - 2, 1), (8, 1), (8, N - 1), (3, 5), (LAM, 1), (1, LAM), (7, 1), (16, N - 2)]
KNOWN_KEYS = [("G", 1), ("-G", N - 1), ("lamG", LAM), ("-lamG", N - LAM), ("2G", 2), ("C0FFEE", 0xC0FFEE)]
FILLER_SEED = 0xC4AF7


@functools.lru_cache(maxsize=None)
def gmul(k: int):
    """k*G (None = infinity), memoised: the families share many multiples"""
    return ec.point_mul(k % N, ec.G)


@functools.lru_cache(maxsize=None)
def address(pt) -> bytes:
    return ec.pubkey_to_address(pt)


def filler() -> wl.ValidatorSet:
    """honest validators: the ordinary signatures around the crafted ones, and the 'other validator' a signature is claimed by"""
    return wl.ValidatorSet(FILLER_SEED, 8)


@dataclass(frozen=True)
class Case:
    label: str
    kind: int            # 0: data is the digest z; 1: data is the signed payload (z = Keccak-256); 2: data is a proposal hash (seal)
    data: bytes
    r: int
    s: int
    v: int
    key: tuple | None    # the key the recovery of (z, r, s, v) yields; None: invalid or the point at infinity
    signer: bytes        # the claimed signer

    @property
    def sig(self) -> bytes:
        return self.r.to_bytes(32, "big") + self.s.to_bytes(32, "big") + bytes([self.v])

    @property
    def digest(self) -> bytes:
        return digest_of(self.kind, self.data)

    @property
    def valid(self) -> bool:
        """the verdict when the signer is a member"""
        return self.key is not None and address(self.key) == self.signer

    @property
    def in_range(self) -> bool:
        return 1 <= self.r < N and 1 <= self.s < N and self.v in (0, 1)

    @property
    def recovered(self) -> bytes:
        return address(self.key) if self.key is not None else bytes(20)


def digest_of(kind: int, data: bytes) -> bytes:
    if kind == 0:
        return data
    if kind == 1:
        return co.keccak256(data)
    return wl.seal_digest(data)


def _key(z: int, r: int, s: int, v: int, t: int | None):
    """the key the recovery of (z, r, s, v) yields when the curve point of abscissa r is +-t*G (t None: r is no abscissa)"""
    if t is None or not (1 <= r < N and 1 <= s < N) or v not in (0, 1):
        return None
    R = gmul(t)
    assert R[0] == r
    tt = t if (R[1] & 1) == v else -t
    return gmul((tt * s - z) * pow(r, -1, N))


def _case(label, kind, data, r, s, v, t, decoy):
    z = int.from_bytes(digest_of(kind, data), "big")
    key = _key(z, r, s, v, t)
    return Case(label, kind, data, r, s, v, key, address(key) if key is not None else decoy)


def _not_abscissa(x: int) -> int:
    while ec.lift_x(x, 0) is not None:
        x += 1
    return x


def _with_negatives(c: Case, t: int, decoy: bytes, out: list, vflip: bool, claim: bool):
    out.append(c)
    if vflip and c.v in (0, 1):   # the other curve point of abscissa r: recovery yields another key
        z = int.from_bytes(c.digest, "big")
        k2 = _key(z, c.r, c.s, c.v ^ 1, t)
        out.append(Case(c.label + "/vflip", c.kind, c.data, c.r, c.s, c.v ^ 1, k2, c.signer))
    if claim:                     # the very signature, claimed by another validator
        out.append(Case(c.label + "/claimed", c.kind, c.data, c.r, c.s, c.v, c.key, decoy))


def _range_negatives(c: Case, out: list):
    """next to a valid case: r no abscissa; r, s, v out of range -- all claimed by the valid case's signer"""
    x = _not_abscissa(c.r)
    for tag, r, s, v in (("r_no_abscissa", x, c.s, c.v), ("r0", 0, c.s, c.v), ("rN", N, c.s, c.v), ("s0", c.r, 0, c.v),
                         ("sN", c.r, N, c.v), ("v2", c.r, c.s, 2), ("v27", c.r, c.s, 27)):
        out.append(Case(f"{c.label}/{tag}", c.kind, c.data, r, s, v, None, c.signer))


def family_a(decoys):
    out = []
    for bi, (name, d) in enumerate(BASES):
        Pt = gmul(d)
        assert Pt[0] < N
        for j, (a, b) in enumerate(SPECIAL):
            r, v = Pt[0], Pt[1] & 1
            c = _case(f"A:{name}:{j}", 0, ((-a * r) % N).to_bytes(32, "big"), r, b * r % N, v, d, decoys[j % len(decoys)])
            _with_negatives(c, d, decoys[(j + 1) % len(decoys)], out, vflip=c.valid and j % 3 == bi % 3, claim=c.valid and j % 3 == (bi + 1) % 3)
    return out


def family_b(decoys, rnd):
    out = []
    sources = [(0, z.to_bytes(32, "big")) for z in (0, 1, N - 1, N, 2**256 - 1)]
    sources += [(0, rnd.getrandbits(256).to_bytes(32, "big")) for _ in range(3)]
    sources += [(1, bytes(rnd.getrandbits(8) for _ in range(ln))) for ln in (0, 77, 136)]
    sources += [(2, rnd.getrandbits(256).to_bytes(32, "big")) for _ in range(3)]
    for i, (kind, data) in enumerate(sources):
        z = int.from_bytes(digest_of(kind, data), "big") % N
        while True:
            k = rnd.getrandbits(256) % N
            R = gmul(k)
            if k and R[0] < N:
                break
        r, v = R[0], R[1] & 1
        kinv = pow(k, -1, N)
        decoy = decoys[i % len(decoys)]
        for tag, s in (("dbl", -z * kinv % N), ("inf", z * kinv % N)):
            c = _case(f"B:{kind}:{i}:{tag}", kind, data, r, s, v, k, decoy)
            _with_negatives(c, k, decoys[(i + 1) % len(decoys)], out, vflip=c.valid, claim=c.valid)
            out.append(_case(f"B:{kind}:{i}:{tag}/highs", kind, data, r, (N - s) % N if s else N, v ^ 1, k, decoy))
    return out


def family_c(decoys):
    out = []
    L = len(HALVES)
    for j in range(L + 6):
        name, d = BASES[j % len(BASES)]
        Pt = gmul(d)
        u2 = (HALVES[j % L] + HALVES[(5 * j + 1) % L] * LAM) % N
        u1 = (HALVES[(3 * j + 2) % L] + HALVES[(7 * j + 3) % L] * LAM) % N
        if j >= L:
            u1 = 0 if j % 2 else u2     # zero digest; the two generator streams equal the two R streams
        if u2 == 0:
            u2 = (8 - 8 * LAM) % N
        r, v = Pt[0], Pt[1] & 1
        c = _case(f"C:{name}:{j}", 0, ((-u1 * r) % N).to_bytes(32, "big"), r, u2 * r % N, v, d, decoys[j % len(decoys)])
        _with_negatives(c, d, decoys[(j + 3) % len(decoys)], out, vflip=c.valid and j % 2 == 0, claim=c.valid and j % 2 == 1)
    return out


def family_d(decoys):
    out = []
    u2s = [(HALVES[6] + HALVES[7] * LAM) % N, (ALL80 - ALL80 * LAM) % N, (2**127 + (2**128 - 1) * LAM) % N]
    for qi, (name, dq) in enumerate(KNOWN_KEYS):
        for ui, u2 in enumerate(u2s):
            for tag, u1 in (("u1=u2", u2), ("u1=-u2", N - u2), ("u1G=u2Q", u2 * dq % N)):
                t = (u1 + u2 * dq) % N
                if t == 0:
                    continue                      # R would be the point at infinity
                R = gmul(t)
                if R[0] >= N:
                    continue
                r, v = R[0], R[1] & 1
                s = r * pow(u2, -1, N) % N
                z = u1 * s % N
                c = _case(f"D:{name}:{ui}:{tag}", 0, z.to_bytes(32, "big"), r, s, v, t, decoys[ui % len(decoys)])
                assert c.key == gmul(dq)
                _with_negatives(c, t, decoys[(qi + ui) % len(decoys)], out, vflip=(qi + ui) % 2 == 0, claim=(qi + ui) % 2 == 1)
    return out


@functools.lru_cache(maxsize=1)
def all_cases() -> tuple[Case, ...]:
    rnd = random.Random(20261017)
    decoys = filler().addrs
    fams = [family_a(decoys), family_b(decoys, rnd), family_c(decoys), family_d(decoys)]
    out = []
    for fam in fams:
        out += fam
        valid = [c for c in fam if c.valid]
        for c in valid[:2]:
            _range_negatives(c, out)
    return tuple(out)


def family_counts(cases) -> dict:
    cnt = {}
    for c in cases:
        f = c.label[0]
        tot, val = cnt.get(f, (0, 0))
        cnt[f] = (tot + 1, val + int(c.valid))
    return cnt


def to_items(cases, group: int = 0, arena: bytearray | None = None):
    """(items, arena) for a list of cases; payload cases append their bytes to `arena`"""
    arena = bytearray() if arena is None else arena
    rows = []
    for c in cases:
        if c.kind == 1:
            rows.append(wl.make_item(c.sig, c.signer, 1, b"", group, len(arena), len(c.data)))
            arena += c.data
        else:
            rows.append(wl.make_item(c.sig, c.signer, c.kind, c.data, group))
    return np.concatenate(rows), arena


def honest_cases(n: int) -> list[Case]:
    """n ordinary valid signatures of the filler validators (fixed digests)"""
    vs = filler()
    out = []
    for i in range(n):
        k = i % vs.n
        dig = co.keccak256(b"honest" + i.to_bytes(4, "big"))
        sig = wl.sign(vs.keys[k], dig)
        out.append(Case(f"honest:{i}", 0, dig, int.from_bytes(sig[:32], "big"), int.from_bytes(sig[32:64], "big"), sig[64],
                        gmul(vs.keys[k]), vs.addrs[k]))
    return out
