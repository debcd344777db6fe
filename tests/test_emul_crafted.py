"""The crafted signatures of crafted.py (colliding points, points at infinity, Booth-digit edges) through every CPU pipeline:
the Python oracle's recovery, the C oracle, and the host emulation of the device arithmetic -- the one-thread recovery, the
level-structured law of the four-lane kernel, the split and four-lane split pipelines, and the known-key verification with its
chain / helper cut.  All of them must agree case by case.  This pins the construction before any GPU time is spent: a GPU
mismatch on the same cases then points at GPU-only code (PTX field arithmetic, exec_quad, named barriers, device-built tables)."""
import ctypes

import numpy as np

import crafted
from oracle import coracle as co
from oracle import secp256k1 as ec


def _run(fn, item, arena):
    out = (ctypes.c_uint8 * 20)()
    rc = fn(item.ctypes.data_as(ctypes.c_void_p), arena.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(len(arena)), out)
    return rc, bytes(out)


def _known(emul, item, arena, key):
    rk = ctypes.c_int(0)
    key64 = (ctypes.c_uint8 * 64).from_buffer_copy(key[0].to_bytes(32, "big") + key[1].to_bytes(32, "big"))
    ok = emul.emul_verify_item_known(item.ctypes.data_as(ctypes.c_void_p), arena.ctypes.data_as(ctypes.c_void_p),
                                     ctypes.c_size_t(len(arena)), key64, ctypes.byref(rk))
    return ok, rk.value


def test_crafted_cases_agree_on_every_cpu_pipeline(emul):
    cases = crafted.all_cases()
    counts = crafted.family_counts(cases)
    # every family produces its cases, valid ones and rejected ones
    assert set(counts) == {"A", "B", "C", "D"}
    for fam, (total, valid) in counts.items():
        assert 0 < valid < total, fam
    assert len(cases) >= 500
    # the branches the families are built for: a final doubling (B) and infinity, known keys with colliding streams (D)
    assert any(c.label.startswith("B:") and c.label.endswith(":dbl") and c.valid for c in cases)
    assert any(c.label.startswith("B:") and ":inf" in c.label and c.in_range and c.key is None for c in cases)
    assert sum(c.label.startswith("D:") and c.valid for c in cases) >= 36
    signer_key = {crafted.address(c.key): c.key for c in cases if c.valid}
    recovered = {}
    for c in cases:
        z = int.from_bytes(c.digest, "big")
        t = (z, c.r, c.s, c.v)
        if t not in recovered:
            recovered[t] = ec.recover_pubkey(z, c.r, c.s, c.v)
        assert recovered[t] == c.key, c.label                             # the construction IS the oracle's recovery
        want_addr = crafted.address(c.key) if c.key is not None else None
        assert co.ecrecover_address(c.digest, c.sig) == want_addr, c.label
        item, arena = crafted.to_items([c])
        a = np.frombuffer(bytes(arena), np.uint8) if arena else np.zeros(1, np.uint8)
        want = (int(c.valid), c.recovered)
        for fn in (emul.emul_verify_item, emul.emul_verify_item_levels, emul.emul_verify_item_split, emul.emul_verify_item_qsplit):
            assert _run(fn, item, a) == want, (c.label, fn.__name__)
        # known-key verification against the claimed signer's learned key, and against the key the recovery yields
        q = signer_key.get(c.signer)
        if q is not None:
            hit = int(c.key == q)
            assert _known(emul, item, a, q) == (hit, hit), c.label
        if c.key is not None and c.key != q:
            assert _known(emul, item, a, c.key) == (1, 1), c.label
