"""Crafted signatures (crafted.py: colliding points, points at infinity, Booth-digit edges) through every verification kernel,
and the device-built comb tables read back entry by entry.

Honest and random signatures reach the exceptional branches of the group law with probability about 2^-128, so the parity
fixtures never exercise them on the GPU; a Byzantine validator reaches them on purpose.  Here the four recover kernels, the
known-key kernels with their worklist recovery, and the tables those kernels read are checked against the oracle where a
GPU-only mistake (a quad whose doubling branch desynchronises, a PTX result fe_is_zero misreads, a wrong table entry) would
otherwise pass unnoticed.  test_emul_crafted.py has already pinned every case on the CPU pipelines of the same headers."""
import functools

import numpy as np
import pytest

import crafted
import ibft_b200 as ib
import workloads as wl
from oracle import coracle as co
from oracle import secp256k1 as ec
from test_gpu_verify import expected_groups

pytestmark = pytest.mark.gpu
P, N = ec.P, ec.N
BETA = 0x7AE96A2B657C07106E64479EAC3434E99CF0497512F58995C1396C28719501EE  # lambda * (x, y) = (beta x, y)
SLOT, HEIGHT = 7, 4242
# Crafted positions inside a batch of honest signatures, chosen for the layouts of all four recover kernels:
#   5            alone in its warp (thread: items 0-31; quad / four-lane chain: 0-7)
#   40, 47       first and last quad of a quad-kernel warp (40-47)
#   5, 40, 70    the three chain warps of the first split CTA (0-95); 99, 158, 191 those of the second (96-191)
#   5 / 158 / 40 the three four-lane chain warps of a qsplit CTA (24 signatures: 0-7, 152-159 of 144-167, 40-47 of 24-47)
#   200, 211     the partial last CTA of every kernel (212 items); in the split kernel their helper lanes' other two
#                signatures (i + 32, i + 64) are out of range -- the batched inversion multiplies in neutral elements
PLACES = [5, 40, 47, 70, 99, 158, 191, 200, 211]
BATCH = 212


@functools.lru_cache(maxsize=1)
def world():
    """crafted cases, honest filler signatures, and the validator table: every crafted key that signs validly + the filler"""
    cases = crafted.all_cases()
    honest = crafted.honest_cases(BATCH)
    keys = sorted({c.key for c in cases if c.valid})
    addrs = [crafted.address(k) for k in keys] + list(crafted.filler().addrs)
    powers = [1 + (i * 7919) % 13 for i in range(len(addrs))]
    A = np.frombuffer(b"".join(addrs), np.uint8).reshape(-1, 20).copy()
    W = np.frombuffer(b"".join(p.to_bytes(32, "big") for p in powers), np.uint8).reshape(-1, 32).copy()
    assert all(c.signer in set(addrs) for c in cases)   # every item is a member's: only the signature decides
    return cases, honest, A, W


def bits_of(bm, n):
    return np.unpackbits(bm.view(np.uint8), bitorder="little")[:n].astype(bool)


def check(eng, cs, slot=SLOT, want_recovered=True, pad=0):
    """verify `cs` as one batch; bitmap, recovered addresses and the group result must be the oracle's"""
    _, _, A, W = world()
    items, arena = crafted.to_items(cs)
    arena = bytes(arena) + bytes(pad)
    bm, res, rec = eng.verify_batch(items, arena, eng.groups(1, slot), want_recovered=want_recovered)
    want = np.array([c.valid for c in cs])
    wrong = [cs[i].label for i in np.nonzero(bits_of(bm, len(cs)) != want)[0]]
    assert not wrong, wrong[:12]
    if want_recovered:
        wrong = [c.label for i, c in enumerate(cs) if bytes(rec[i]) != c.recovered]
        assert not wrong, wrong[:12]
    exp, _ = expected_groups(items, bm, A, W)
    nv, nd, power, hq = exp.get(0, (0, 0, 0, False))
    r = res[0]
    assert (int(r["n_valid"]), int(r["n_distinct"]), bool(r["has_quorum"])) == (nv, nd, hq)
    assert sum(int(r["power"][k]) << (64 * k) for k in range(5)) == power
    return bm, res


def place(chunk):
    _, honest, _, _ = world()
    batch = list(honest)
    for pos, c in zip(PLACES, chunk):
        batch[pos] = c
    return batch


def set_table(eng):
    _, _, A, W = world()
    eng.set_validators(SLOT, HEIGHT, A, W)


def test_crafted_cases_placed_among_honest_signatures(engine):
    cases, _, _, _ = world()
    set_table(engine)
    for k in range(0, len(cases), len(PLACES)):
        check(engine, place(cases[k:k + len(PLACES)]))


def test_crafted_cases_only_and_each_alone(engine):
    cases, _, A, _ = world()
    set_table(engine)
    bm, _ = check(engine, list(cases))
    items, arena = crafted.to_items(cases)
    assert np.array_equal(bm, co.verify_batch(items, bytes(arena), tables=[A], group_table=[0], n_threads=8))
    for c in cases:
        check(engine, [c])


# --------------------------------------------------------------------------------------------- known-key kernels
def deferred_known(cs):
    """k_verify_known leaves every member item it does not accept to the recover pass (out-of-range scalars included)"""
    return sum(not c.valid for c in cs)


def deferred_split(cs):
    """k_verify_split settles out-of-range scalars itself and leaves the other member items it does not accept"""
    return sum(c.in_range and not c.valid for c in cs)


def test_known_key_kernels_on_crafted_cases():
    """Pass 1 learns every crafted key through recovery; pass 2 sends the same signatures through k_verify_known<32> (+ the
    four-lane worklist recovery), the round cut in four pieces, k_verify_known<128> (+ k_recover<128> on the worklist),
    k_verify_split and the long-payload form.  Verdicts and group results equal pass 1 and the oracle on every path, and the
    known-key pass defers exactly the items it must: a kernel that rejected valid signatures would still give the right verdicts
    through the worklist, but not the right count."""
    cases, honest, A, W = world()
    base = list(cases) + honest[:64]
    items, arena = crafted.to_items(base)
    arena = bytes(arena)
    want = np.array([c.valid for c in base])
    eng = ib.Engine(device=0, max_items=1 << 16, max_payload_bytes=1 << 24, max_groups=4, max_table_slots=2, max_validators=4096, key_cache=True)
    try:
        sms = eng.device_info()["sm_count"]
        eng.set_validators(0, 9, A, W)
        g = eng.groups(1, 0)
        bm1, res1 = check(eng, base, slot=0, want_recovered=False)
        assert eng.last_deferred() == len(base)                          # nothing known yet: every member item is recovered
        assert eng.refresh_key_tables() == len(A)
        # small batch: k_verify_known<32>, then k_recover_qsplit on the worklist
        bm, res = check(eng, base, slot=0, want_recovered=False)
        assert np.array_equal(bm, bm1) and res.tobytes() == res1.tobytes()
        assert eng.last_deferred() == deferred_known(base)
        # long payloads (arena / count > 256): k_recover<128> on the worklist
        bm, res = check(eng, base, slot=0, want_recovered=False, pad=300 * len(base))
        assert np.array_equal(bm, bm1) and res.tobytes() == res1.tobytes()
        assert eng.last_deferred() == deferred_known(base)
        # forced chain + helper form: k_verify_split
        eng.set_recover_path(ib.Engine.PATH_SPLIT)
        bm, res = check(eng, base, slot=0, want_recovered=False)
        assert np.array_equal(bm, bm1) and res.tobytes() == res1.tobytes()
        assert eng.last_deferred() == deferred_split(base)
        eng.set_recover_path(ib.Engine.PATH_AUTO)
        # tiled: a mid-size round in four pieces (four worklists), and a batch above SMs x 256 (k_verify_known<128>)
        for reps in ((sms * 48) // len(base) + 1, (sms * 256) // len(base) + 1):
            big = np.tile(items, reps)
            assert len(big) <= 1 << 16
            bm, res, _ = eng.verify_batch(big, arena, g)
            assert np.array_equal(bits_of(bm, len(big)), np.tile(want, reps)), reps
            assert eng.last_deferred() == reps * deferred_known(base), reps
            r, r1 = res[0], res1[0]
            assert int(r["n_valid"]) == reps * int(r1["n_valid"])
            assert (int(r["n_distinct"]), int(r["has_quorum"]), r["power"].tobytes()) == (int(r1["n_distinct"]), int(r1["has_quorum"]), r1["power"].tobytes())
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------ device-built tables
def points(words):
    """(n, 16) little-endian uint32 words -> [(x, y)]"""
    b = np.ascontiguousarray(words, dtype="<u4").tobytes()
    return [(int.from_bytes(b[64 * i:64 * i + 32], "little"), int.from_bytes(b[64 * i + 32:64 * i + 64], "little")) for i in range(len(words))]


def is_sum(a, b, c):
    """c == a + b for verified a, b with distinct abscissas, without an inversion: c is canonical, on the curve, and -c is the
    third point of the chord through a and b (a line meets the curve in exactly three points)"""
    x1, y1 = a
    x2, y2 = b
    x3, y3 = c
    return (x3 < P and y3 < P and x3 != x1 and x3 != x2 and (y3 * y3 - x3 * x3 * x3 - 7) % P == 0
            and ((y2 - y1) * (x3 - x1) + (y3 + y1) * (x2 - x1)) % P == 0)


def dbl(a):
    return ec.point_add(a, a)


def test_generator_comb_every_entry():
    """All 17 positions of the generator comb k_build_ctable writes (positions 1.. feed ecmult_gen_comb and the known-key walk):
    entry (d1, d2) of position j = 2^(8j) (d1 + d2 lambda) G.  Anchored with the oracle's scalar multiplication, every other entry
    checked against its neighbour with the chord relation."""
    eng = ib.Engine(device=0, max_items=64, max_payload_bytes=1024, max_groups=1, max_table_slots=1, max_validators=8)
    try:
        wc, per = eng.combined_table_info()
        assert wc == 8 and per == 129 * 257
        positions = 17
        with pytest.raises(ib.EngineError):
            eng.combined_table_entries(positions * per - 1, 2)            # one past the last position
        assert ec.point_mul(crafted.LAM, ec.G) == (BETA * ec.G[0] % P, ec.G[1])
        half, d2n = 128, 257
        Gj = ec.G
        for j in range(positions):
            E = points(eng.combined_table_entries(j * per, per))
            at = lambda d1, d2: E[d1 * d2n + d2 + half]  # noqa: E731
            Lj = (BETA * Gj[0] % P, Gj[1])
            nL = ec.point_neg(Lj)
            scale = pow(2, 8 * j, N)
            assert at(0, 0) == (0, 0), j                                      # infinity: never looked up
            assert (at(1, 0), at(0, 1), at(0, -1)) == (Gj, Lj, nL), j
            assert (at(2, 0), at(0, 2), at(0, -2)) == (dbl(Gj), dbl(Lj), ec.point_neg(dbl(Lj))), j
            for d1, d2 in ((128, -128), (128, 128), (97, -31)):
                assert at(d1, d2) == crafted.gmul((d1 + d2 * crafted.LAM) * scale), (j, d1, d2)
            bad = []
            for d1 in range(half + 1):
                if d1 >= 3 and not is_sum(at(d1 - 1, 0), Gj, at(d1, 0)):
                    bad.append((d1, 0))
                for d2 in range(1, half + 1):
                    if (d1, d2) not in ((0, 1), (0, 2)):
                        if not is_sum(at(d1, d2 - 1), Lj, at(d1, d2)):
                            bad.append((d1, d2))
                        if not is_sum(at(d1, -d2 + 1), nL, at(d1, -d2)):
                            bad.append((d1, -d2))
            assert not bad, (j, bad[:8])
            for _ in range(8):
                Gj = dbl(Gj)
    finally:
        eng.close()


def check_keytab(tab, d):
    """the 17 x 128 entries of a validator's key comb: entry j * 128 + m - 1 = m 2^(8j) Q for Q = d G"""
    E = points(tab)
    B = crafted.gmul(d)
    for j in range(17):
        row = E[128 * j:128 * (j + 1)]
        assert row[0] == B and row[1] == dbl(B), j
        assert row[127] == crafted.gmul(128 * pow(2, 8 * j, N) * d), j
        bad = [m + 1 for m in range(2, 128) if not is_sum(row[m - 1], B, row[m])]
        assert not bad, (j, bad[:8])
        for _ in range(8):
            B = dbl(B)


def test_key_tables_built_and_carried():
    """k_build_keytabs for the known-key family's special keys and two ordinary keys; k_carry_keys to another slot and height
    (byte-identical to the donor); a validator that never signed is never READY."""
    special = [d for _, d in crafted.KNOWN_KEYS] + [wl.privkey(91, 0), wl.privkey(91, 1)]
    never = wl.privkey(91, 2)
    addrs = [crafted.address(crafted.gmul(d)) for d in special + [never]]
    A = np.frombuffer(b"".join(addrs), np.uint8).reshape(-1, 20).copy()
    eng = ib.Engine(device=0, max_items=64, max_payload_bytes=1024, max_groups=1, max_table_slots=2, max_validators=16, key_cache=True)
    try:
        eng.set_validators(0, 5, A, None)
        dig = co.keccak256(b"key tables")
        items = np.concatenate([wl.make_item(wl.sign(d, dig), a, 0, dig) for d, a in zip(special, addrs)])
        bm, _, _ = eng.verify_batch(items, b"", eng.groups(1, 0))
        assert bits_of(bm, len(special)).all()
        assert eng.refresh_key_tables() == len(special)
        tabs = {}
        for v, d in enumerate(special):
            st, tab = eng.key_table_entries(0, v, 0, 17 * 128)
            assert st == 2, v                                                # READY
            check_keytab(tab, d)
            tabs[addrs[v]] = tab
        assert eng.key_table_entries(0, len(special))[0] == 0                 # never signed: unknown
        with pytest.raises(ib.EngineError):
            eng.key_table_entries(0, 0, 17 * 128 - 1, 2)
        # next height in the other slot, validators in reverse order: the finished tables are carried over by address
        A2 = A[::-1].copy()
        eng.set_validators(1, 6, A2, None)
        assert eng.refresh_key_tables() == 2 * len(special)
        for v in range(len(A2)):
            st, tab = eng.key_table_entries(1, v, 0, 17 * 128)
            a = bytes(A2[v])
            if a in tabs:
                assert st == 2 and tab.tobytes() == tabs[a].tobytes(), v
            else:
                assert st == 0, v
        check_keytab(eng.key_table_entries(1, len(A2) - 1, 0, 17 * 128)[1], special[0])
    finally:
        eng.close()
