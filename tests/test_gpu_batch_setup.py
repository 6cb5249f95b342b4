"""Batched set-up of many statements: bpg_witness_eval_batch must leave every entry byte-identical to bpg_witness_eval (and to
the big-integer evaluation) for the reference fixtures, the configs[4] shapes, edge statements and batches above one pass, in
at most one launch per pass, and fail whole (no caller buffer written) on bad arguments.  Handles of bpg_circuit_create_batch
must prove and verify exactly like bpg_circuit_create handles, outlive the other handles of their call, and fail whole.  The
Python API builds its circuits and witnesses with the two calls (api.prove_batch) and verifies in one call (api.verify_batch)."""
import ctypes as C
import hashlib
import os
import random

import pytest

import bench
from circuits import host_witness
from oracle import pyref as pr

pytestmark = pytest.mark.gpu

L = pr.L
FX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures")
FIXTURES = ["bounds_check", "equality", "example", "inequality", "less_than", "merkle_tree", "mimc_hash", "or", "or2", "or3", "or4", "or5",
            "set_membership"]
CAP = 1 + 32 * (14 + 64 + 2)
E_SIZE, E_ARG = -2, -4
FLAG_LEGACY = 1
enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)


@pytest.fixture(scope="module")
def ctx():
    import bulletproofs_gadgets_b200 as bpg
    c = bpg.Context(0)
    c.gens_ensure(16384)
    yield c
    c.close()


def rd(name):
    with open(os.path.join(FX, name)) as f:
        return f.read()


def fixture_prover(ctx, name):
    from bulletproofs_gadgets_b200 import frontend as fe
    return fe.ProverRun(name.encode(), rd(name + ".gadgets"), rd(name + ".inst"), rd(name + ".wtns"), test_seed=1, ctx=ctx).prover


def cfg5_item(k, valid=True):
    """witness item (Context.witness_eval_batch) and CSR entry (Context.circuit_create_batch) of configs[4] statement k"""
    k, label, n, m, rp, tv, tc, (inL, inR, wp, wv, wc), v, vb, valid = bench._cfg5_assemble(("sm" if k % 2 == 0 else "lt", k, valid))
    return (n, m, wp, wv, wc, v, inL, inR), (n, m, rp, tv, tc), (label, v, vb)


def single_witness(ctx, it):
    """bpg_witness_eval of one item -> (a_L, a_R, a_O) bytes"""
    n, m, wp, wv, wc, v, inL, inR = it
    aL, aR, aO = C.create_string_buffer(bytes(inL), 32 * max(1, n)), C.create_string_buffer(bytes(inR), 32 * max(1, n)), C.create_string_buffer(32 * max(1, n))
    ctx.check(ctx.lib.bpg_witness_eval(ctx.h, n, m, (C.c_uint32 * max(1, len(wp)))(*wp), (C.c_uint32 * max(1, len(wv)))(*wv), bytes(wc), v, aL, aR, aO))
    return aL.raw[:32 * n], aR.raw[:32 * n], aO.raw[:32 * n]


def check_witness_batch(ctx, items, provers=None):
    got = ctx.witness_eval_batch(items)
    assert len(got) == len(items)
    for k, it in enumerate(items):
        assert got[k] == single_witness(ctx, it), "entry %d of %d differs from bpg_witness_eval" % (k, len(items))
        if provers is not None and provers[k] is not None:
            assert got[k] == tuple(enc(x) for x in host_witness(provers[k])), "entry %d differs from the big-integer evaluation" % k
    return got


def test_witness_batch_reference_fixtures(ctx):
    """all 13 fixtures in one batch; example (14 988 multipliers) and the other large ones take the delegated path"""
    ps = [fixture_prover(ctx, nm) for nm in FIXTURES]
    check_witness_batch(ctx, [p._witness_args() for p in ps], ps)


def test_witness_batch_config5(ctx):
    check_witness_batch(ctx, [cfg5_item(k, valid=(k % 13 != 5))[0] for k in range(200)])


def edge_provers(ctx):
    import bulletproofs_gadgets_b200 as bpg
    rnd = random.Random(11)
    out = []
    p = bpg.Prover.new(b"empty", ctx=ctx)           # n = 0 (one commitment)
    p.commit(5, 1)
    out.append(p)
    p = bpg.Prover.new(b"assigned", ctx=ctx)        # only assigned multipliers
    for _ in range(7):
        p.allocate_multiplier((rnd.randrange(L), rnd.randrange(L)))
    out.append(p)
    p = bpg.Prover.new(b"pending", ctx=ctx)         # a half-allocated multiplier: a_R still zero
    p.allocate_multiplier((L - 1, L - 1))
    p.allocate(7)
    out.append(p)
    p = bpg.Prover.new(b"chain", ctx=ctx)           # a 300-deep chain
    _, v0 = p.commit(rnd.randrange(L), 1)
    x = p.allocate(7)
    p.allocate(9)
    cur = [(x, 3), (v0, L - 2), (bpg.api.ONE, rnd.randrange(L))]
    for _ in range(300):
        _, r, o = p.multiply(cur, cur + [(bpg.api.ONE, 1)])
        cur = [(o, rnd.randrange(L)), (r, 5), (v0, 1)]
    out.append(p)
    p = bpg.Prover.new(b"wide", ctx=ctx)            # level 1 holds 600 multipliers: wider than the 256-thread block
    a, b, o = p.allocate_multiplier((3, 4))
    _, v1 = p.commit(rnd.randrange(L), 1)
    for k in range(600):
        p.multiply([(a, k + 1), (v1, 2)], [(o, rnd.randrange(L)), (b, 1), (bpg.api.ONE, k)])
    out.append(p)
    return out


def unreduced(it):
    """the same statement with every caller input (a_L, a_R, v, coefficients) given as x + l >= l"""
    n, m, wp, wv, wc, v, inL, inR = it
    up = lambda b: b"".join((int.from_bytes(b[i:i + 32], "little") + L).to_bytes(32, "little") for i in range(0, len(b), 32))
    return (n, m, wp, wv, up(wc), up(v), up(inL), up(inR))


def test_witness_batch_edge_statements(ctx):
    ps = edge_provers(ctx)
    items = [p._witness_args() for p in ps]
    items += [unreduced(it) for it in items]
    got = check_witness_batch(ctx, items, ps + ps)
    assert got[0] == (b"", b"", b"")
    assert got[2][2] == enc([1, 0])


def tiny_item(k):
    """two multipliers: an assigned one and one multiply() of it"""
    rnd = random.Random(k)
    a, b, c = rnd.randrange(L), rnd.randrange(L), rnd.randrange(L)
    return (2, 1, [0, 0, 0, 1, 3], [0 << 29, 2 << 29, 3 << 29], enc([c, 1, k]), enc([b]), enc([a, 0]), enc([b, 0]))


def test_witness_batch_above_one_pass(ctx):
    """1 100 statements: more than the 1 024 of one pass"""
    check_witness_batch(ctx, [tiny_item(k) for k in range(1100)])


def raw_witness_batch(ctx, items, **over):
    """bpg_witness_eval_batch with sentinel-filled outputs -> (rc, [(aL, aR, aO) raw buffers]); `over` replaces an argument array"""
    k = len(items)
    bufs = [[C.create_string_buffer(bytes(it[6 + j]) if j < 2 else b"", 32 * max(1, it[0])) for j in range(3)] for it in items]
    for b in bufs:
        for x in b:
            C.memset(x, 0xA5, len(x))
    keep = [[(C.c_uint32 * max(1, len(it[j])))(*it[j]) for it in items] for j in (2, 3)]
    arg = dict(n=(C.c_size_t * k)(*[it[0] for it in items]), m=(C.c_size_t * k)(*[it[1] for it in items]),
               lc_ptr=(C.POINTER(C.c_uint32) * k)(*[C.cast(x, C.POINTER(C.c_uint32)) for x in keep[0]]),
               term_var=(C.POINTER(C.c_uint32) * k)(*[C.cast(x, C.POINTER(C.c_uint32)) for x in keep[1]]),
               term_coeff=(C.c_char_p * k)(*[bytes(it[4]) for it in items]), v=(C.c_char_p * k)(*[bytes(it[5]) for it in items]),
               aL=(C.c_void_p * k)(*[C.addressof(b[0]) for b in bufs]), aR=(C.c_void_p * k)(*[C.addressof(b[1]) for b in bufs]),
               aO=(C.c_void_p * k)(*[C.addressof(b[2]) for b in bufs]))
    arg.update(over)
    rc = ctx.lib.bpg_witness_eval_batch(ctx.h, k, arg["n"], arg["m"], arg["lc_ptr"], arg["term_var"], arg["term_coeff"], arg["v"], arg["aL"],
                                        arg["aR"], arg["aO"])
    return rc, [[x.raw for x in b] for b in bufs]


def test_witness_batch_bad_arguments_write_nothing(ctx):
    items = [tiny_item(k) for k in range(10)]
    _, before = raw_witness_batch(ctx, items, n=(C.c_size_t * 10)(*([0] * 10)))  # n = 0 everywhere: nothing evaluated, nothing written
    fwd = list(items[5])
    fwd[3] = [0 << 29, 2 << 29, 0 << 29 | 1]     # multiplier 1 references a_L[1]: itself, not an earlier multiplier
    bad = items[:5] + [tuple(fwd)] + items[6:]
    rc, after = raw_witness_batch(ctx, bad)
    assert rc == E_ARG and after == before
    rc, after = raw_witness_batch(ctx, items, aL=None)
    assert rc == E_ARG and after == before
    rc, after = raw_witness_batch(ctx, items, lc_ptr=None)
    assert rc == E_ARG and after == before
    big_n = lambda k: (C.c_size_t * k)(*[1 << 22 if i == 3 else 2 for i in range(k)])  # checked before lc_ptr is read
    rc, after = raw_witness_batch(ctx, items, n=big_n(10))
    assert rc == E_SIZE and after == before
    # the first failing entry decides the code
    rc, _ = raw_witness_batch(ctx, items[:2] + [tuple(fwd)] + items[3:4], n=big_n(4))
    assert rc == E_ARG
    rc, _ = raw_witness_batch(ctx, items[:4] + [tuple(fwd)], n=big_n(5))
    assert rc == E_SIZE
    assert ctx.lib.bpg_witness_eval_batch(ctx.h, 0, None, None, None, None, None, None, None, None, None) == 0


def test_witness_batch_is_one_launch_per_pass(ctx):
    items = [cfg5_item(k)[0] for k in range(256)]
    ctx.witness_eval_batch(items[:4])  # scratch sized outside the count
    l0 = ctx.launch_count()
    ctx.witness_eval_batch(items)
    assert ctx.launch_count() - l0 <= 2


# ---------------------------------------------------------------- circuits
def single_circuit(ctx, csr):
    n, m, rp, tv, tc = csr
    h = C.c_void_p()
    ctx.check(ctx.lib.bpg_circuit_create(ctx.h, n, m, len(rp) - 1, (C.c_uint32 * len(rp))(*rp), (C.c_uint32 * max(1, len(tv)))(*tv), tc, C.byref(h)))
    return h


def prove_one(ctx, h, st, w, k, flags=0):
    label, v, vb = st
    m = len(v) // 32
    proof, V = C.create_string_buffer(CAP), C.create_string_buffer(32 * max(1, m))
    rc = ctx.lib.bpg_r1cs_prove(ctx.h, h, label, len(label), w[0], w[1], w[2], v, vb, ext_of(k), flags, V, proof, CAP)
    ctx.check(rc)
    return proof.raw[:rc], V.raw[:32 * m]


def verify_one(ctx, h, label, V, proof):
    acc = C.c_int(0)
    ctx.check(ctx.lib.bpg_r1cs_verify(ctx.h, h, label, len(label), V, proof, len(proof), os.urandom(32), 0, C.byref(acc)))
    return bool(acc.value)


def ext_of(k):
    return hashlib.sha256(b"batch setup ext %d" % k).digest()


def statements(ctx, count):
    """configs[4] statements plus two fixtures of other shapes -> (witness items, CSR entries, (label, v, blinding))"""
    wit, csr, st = [], [], []
    for k in range(count):
        a, b, c = cfg5_item(k)
        wit.append(a); csr.append(b); st.append(c)
    for nm in ("or3", "bounds_check"):
        p = fixture_prover(ctx, nm)
        wit.append(p._witness_args()); csr.append(p._circuit_args(len(p.v))); st.append((p.label, enc(p.v), enc(p.v_blinding)))
    return wit, csr, st


def test_circuit_batch_proves_and_verifies_like_single_handles(ctx):
    wit, csr, st = statements(ctx, 24)
    ws = ctx.witness_eval_batch(wit)
    hb = ctx.circuit_create_batch(csr)
    hs = [single_circuit(ctx, c) for c in csr]
    try:
        for flags in (0, FLAG_LEGACY):
            want = [prove_one(ctx, h, s, w, k, flags) for k, (h, s, w) in enumerate(zip(hs, st, ws))]
            assert [prove_one(ctx, h, s, w, k, flags) for k, (h, s, w) in enumerate(zip(hb, st, ws))] == want
            mk = lambda hh: [(h, s[0], w[0], w[1], w[2], s[1], s[2], ext_of(k)) for k, (h, s, w) in enumerate(zip(hh, st, ws))]
            assert ctx.prove_batch(mk(hb), flags) == want
            assert ctx.prove_batch(mk(hs), flags) == want
        want = [prove_one(ctx, h, s, w, k) for k, (h, s, w) in enumerate(zip(hs, st, ws))]
        assert all(verify_one(ctx, h, s[0], V, proof) for h, s, (proof, V) in zip(hb, st, want))
        assert ctx.verify_batch([(h, s[0], V, proof, os.urandom(32)) for h, s, (proof, V) in zip(hb, st, want)]) == [True] * len(hb)
    finally:
        for h in hb + hs:
            ctx.lib.bpg_circuit_destroy(h)


def test_circuit_batch_handles_outlive_each_other(ctx):
    wit, csr, st = statements(ctx, 16)
    ws = ctx.witness_eval_batch(wit)
    hs = [single_circuit(ctx, c) for c in csr]
    want = [prove_one(ctx, h, s, w, k) for k, (h, s, w) in enumerate(zip(hs, st, ws))]
    hb = ctx.circuit_create_batch(csr)
    order = list(range(len(hb)))
    random.Random(3).shuffle(order)
    gone, alive = order[:len(order) // 2], order[len(order) // 2:]
    for i in gone:
        ctx.lib.bpg_circuit_destroy(hb[i])
    for i in alive:
        assert prove_one(ctx, hb[i], st[i], ws[i], i) == want[i]
    items = [(hb[i], st[i][0], ws[i][0], ws[i][1], ws[i][2], st[i][1], st[i][2], ext_of(i)) for i in alive]
    assert ctx.prove_batch(items) == [want[i] for i in alive]
    for i in alive:
        ctx.lib.bpg_circuit_destroy(hb[i])
    for h in hs:
        ctx.lib.bpg_circuit_destroy(h)


def raw_circuit_batch(ctx, csr):
    k = len(csr)
    out = (C.c_void_p * k)(*([0x1234] * k))
    keep = [[(C.c_uint32 * max(1, len(c[j])))(*c[j]) for c in csr] for j in (2, 3)]
    u32pp = lambda xs: (C.POINTER(C.c_uint32) * k)(*[C.cast(x, C.POINTER(C.c_uint32)) for x in xs])
    rc = ctx.lib.bpg_circuit_create_batch(ctx.h, k, (C.c_size_t * k)(*[c[0] for c in csr]), (C.c_size_t * k)(*[c[1] for c in csr]),
                                          (C.c_size_t * k)(*[len(c[2]) - 1 for c in csr]), u32pp(keep[0]), u32pp(keep[1]),
                                          (C.c_char_p * k)(*[bytes(c[4]) for c in csr]), out)
    return rc, list(out)


def test_circuit_batch_bad_term_fails_whole(ctx):
    _, csr, _ = statements(ctx, 6)
    for bad_var in ((0 << 29) | csr[3][0], 5 << 29):   # a_L index = n, kind 5
        tv = list(csr[3][3])
        tv[1] = bad_var
        bad = csr[:3] + [csr[3][:3] + (tv,) + csr[3][4:]] + csr[4:]
        rc, out = raw_circuit_batch(ctx, bad)
        assert rc == E_ARG and out == [None] * len(bad)
    n = (C.c_size_t * 1)(1 << 22)
    out = (C.c_void_p * 1)(0x1234)
    rp = (C.c_uint32 * 1)(0)
    assert ctx.lib.bpg_circuit_create_batch(ctx.h, 1, n, (C.c_size_t * 1)(0), (C.c_size_t * 1)(0), (C.POINTER(C.c_uint32) * 1)(rp), None, None, out) == E_SIZE
    assert list(out) == [None]
    assert ctx.lib.bpg_circuit_create_batch(ctx.h, 0, None, None, None, None, None, None, None) == 0


def test_circuit_batch_without_constraints_or_terms(ctx):
    """q = 0 (no constraints) and T = 0 (constraints with no terms) next to an ordinary circuit"""
    rnd = random.Random(4)
    aL, aR = [rnd.randrange(L) for _ in range(3)], [rnd.randrange(L) for _ in range(3)]
    w = (enc(aL), enc(aR), enc([a * b % L for a, b in zip(aL, aR)]))
    wit, csr, st = statements(ctx, 1)
    ws = ctx.witness_eval_batch(wit)
    entries = [(3, 0, [0], [], b""), (3, 0, [0, 0, 0], [], b""), csr[0]]
    sts = [(b"q0", b"", b""), (b"t0", b"", b""), st[0]]
    wits = [w, w, ws[0]]
    hb = ctx.circuit_create_batch(entries)
    hs = [single_circuit(ctx, c) for c in entries]
    try:
        for k in range(3):
            proof, V = prove_one(ctx, hb[k], sts[k], wits[k], k)
            assert (proof, V) == prove_one(ctx, hs[k], sts[k], wits[k], k)
            assert verify_one(ctx, hb[k], sts[k][0], V, proof)
    finally:
        for h in hb + hs:
            ctx.lib.bpg_circuit_destroy(h)


# ---------------------------------------------------------------- Python API
def test_api_verify_batch_matches_verifier_verify(ctx):
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import frontend as fe
    rnd = random.Random(9)
    cases = []
    for k in range(12):
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        if k % 4 == 1:
            a, b = b, a                                                  # a false statement
        cases.append(("LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b)))
    cases.append(("SET_MEMBER W0 I0 I1\n", "I0 = 0x11\nI1 = 0x64\n", "W0 = 0x64\n"))
    runs = [fe.ProverRun(b"vb-%d" % k, g, i, w, test_seed=k, ctx=ctx) for k, (g, i, w) in enumerate(cases)]
    gens = bpg.BulletproofGens.new(4096, 1, ctx=ctx)
    out = bpg.api.prove_batch([r.prover for r in runs], gens, [ext_of(k) for k in range(len(runs))])
    verifiers, proofs = [], []
    for k, (r, (g, i, _), (proof, V)) in enumerate(zip(runs, cases, out)):
        coms = "".join("%s = 0x%s\n" % (nm, c.hex()) for nm, c in zip(r.coms_names, V))
        verifiers.append(fe.VerifierRun(b"vb-%d" % k, g, i, coms, ctx=ctx).verifier)
        proofs.append(proof if k != 6 else proof[:40] + bytes([proof[40] ^ 1]) + proof[41:])  # a tampered proof
    got = bpg.api.verify_batch(verifiers, proofs)
    want = []
    for v, pf in zip(verifiers, proofs):
        try:
            v.verify(pf)
            want.append(True)
        except bpg.R1CSError:
            want.append(False)
    assert got == want
    assert True in want and False in want
    assert bpg.api.verify_batch([], []) == []
    with pytest.raises(ValueError):
        bpg.api.verify_batch(verifiers, proofs[:-1])


def test_api_prove_batch_uses_cached_and_batched_witnesses(ctx):
    """prove_batch fills each prover's witness cache from one batched evaluation; a prover whose witness is already cached,
    or that appears twice, gives the same bytes as Prover.prove"""
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import frontend as fe
    rnd = random.Random(21)
    runs = []
    for k in range(5):
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        runs.append(fe.ProverRun(b"pb-%d" % k, "LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b), test_seed=k, ctx=ctx))
    provers = [r.prover for r in runs]
    provers[1].witness_bytes()
    gens = bpg.BulletproofGens.new(4096, 1, ctx=ctx)
    batch = provers + [provers[2]]
    exts = [ext_of(k) for k in range(len(batch))]
    got = bpg.api.prove_batch(batch, gens, exts)
    assert all(p._witness_cached() for p in provers)
    assert [p.witness() for p in provers] == [host_witness(p) for p in provers]
    assert got == [p.prove(gens, ext_rng32=e) for p, e in zip(batch, exts)]
