"""Batched proving (bpg_r1cs_prove_batch): every proof of a batch must be byte-identical to bpg_r1cs_prove with the same
arguments -- for the config-5 shapes, the reference fixtures, edge circuits, mixed sizes that leave the inner-product lockstep
at different rounds, batches above the internal pass size, a delegated large proof and the legacy framing -- verify, match
the CPU oracle, and fail whole (nothing written) on bad arguments."""
import ctypes as C
import hashlib
import os
import random

import pytest

import circuits
import oracle_lib as ol
from oracle import pyref as pr

pytestmark = pytest.mark.gpu

FX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures")
CAP = 1 + 32 * (14 + 64 + 2)
E_SIZE, E_ARG = -2, -4
FLAG_LEGACY, FLAG_FAST, FLAG_WOD, FLAG_NO_LATE, FLAG_FORCE_LATE = 1, 2, 4, 8, 16


@pytest.fixture(scope="module")
def ctx():
    import bulletproofs_gadgets_b200 as bpg
    c = bpg.Context(0)
    c.gens_ensure(16384)
    yield c
    c.close()


def ext_of(k):
    return hashlib.sha256(b"prove batch ext %d" % k).digest()


def circuit(ctx, n, m, csr):
    rp, tv, tc = csr
    h = C.c_void_p()
    ctx.check(ctx.lib.bpg_circuit_create(ctx.h, n, m, len(rp) - 1, (C.c_uint32 * len(rp))(*rp), (C.c_uint32 * max(1, len(tv)))(*tv), tc, C.byref(h)))
    return h


def item_of_instance(ctx, inst, k):
    """(item for Context.prove_batch, CSR) of a tests/circuits.py instance"""
    m = len(inst["vals"]) // 32
    return (circuit(ctx, inst["n"], m, inst["csr"]), inst["label"], inst["aL"], inst["aR"], inst["aO"], inst["vals"], inst["blinds"], ext_of(k)), inst["csr"]


def item_of_run(ctx, run, k):
    p = run.prover
    enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
    aL, aR, aO = p.witness_bytes()
    return (p._circuit(len(p.v)), p.label, aL, aR, aO, enc(p.v), enc(p.v_blinding), ext_of(k)), p.csr()


def no_commitment_instance(n, seed):
    """m = 0: allocate_multiplier gates tied to constants (L_i - aL_i = 0)"""
    rnd = random.Random(seed)
    aL = [rnd.randrange(pr.L) for _ in range(n)]
    aR = [rnd.randrange(pr.L) for _ in range(n)]
    aO = [a * b % pr.L for a, b in zip(aL, aR)]
    rows = [[(("L", i), 1), (("1", 0), (-aL[i]) % pr.L)] for i in range(n)]
    enc = lambda xs: b"".join(pr.sc_bytes(a) for a in xs)
    return dict(label=b"nocommit", n=n, vals=b"", blinds=b"", aL=enc(aL), aR=enc(aR), aO=enc(aO), csr=circuits.to_csr(rows))


def single(ctx, it, flags=0):
    m = len(it[5]) // 32
    proof, V = C.create_string_buffer(CAP), C.create_string_buffer(32 * max(1, m))
    rc = ctx.lib.bpg_r1cs_prove(ctx.h, it[0], it[1], len(it[1]), it[2], it[3], it[4], it[5], it[6], it[7], flags, V, proof, CAP)
    ctx.check(rc)
    return proof.raw[:rc], V.raw[:32 * m]


def check_equal(ctx, items, flags=0):
    got = ctx.prove_batch(items, flags)
    want = [single(ctx, it, flags) for it in items]
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert g == w, "proof %d of %d differs from bpg_r1cs_prove" % (k, len(items))
    return got


def destroy(ctx, items):
    for it in items:
        ctx.lib.bpg_circuit_destroy(it[0])


def raw_call(ctx, items, flags=0, caps=None, null_circuit_at=None):
    """bpg_r1cs_prove_batch with pre-filled outputs -> (rc, proofs, Vs, lens)"""
    n = len(items)
    proofs = [C.create_string_buffer(CAP) for _ in range(n)]
    Vs = [C.create_string_buffer(32 * 8) for _ in range(n)]
    lens = (C.c_size_t * n)(*([12345] * n))
    circs = [None if k == null_circuit_at else it[0] for k, it in enumerate(items)]
    arr = lambda j: (C.c_char_p * n)(*[it[j] for it in items])
    rc = ctx.lib.bpg_r1cs_prove_batch(ctx.h, n, (C.c_void_p * n)(*circs), arr(1), (C.c_size_t * n)(*[len(it[1]) for it in items]), arr(2), arr(3), arr(4),
                                      arr(5), arr(6), b"".join(it[7] for it in items), flags, (C.c_void_p * n)(*[C.addressof(b) for b in Vs]),
                                      (C.c_void_p * n)(*[C.addressof(b) for b in proofs]), (C.c_size_t * n)(*(caps or [CAP] * n)), lens)
    return rc, [p.raw for p in proofs], [v.raw for v in Vs], list(lens)


def cfg5_run(ctx, k):
    """the SET_MEMBER / LESS_THAN shapes of BASELINE configs[4], assembled by the front-end as bench._cfg5_assemble does"""
    from bulletproofs_gadgets_b200 import frontend as fe
    rnd = random.Random(60000 + k)
    label = b"cfg5-%d" % k
    if k % 2:
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        return fe.ProverRun(label, "LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b), test_seed=k, ctx=ctx)
    vals = rnd.sample(range(1 << 40), 5)
    inst = "".join("I%d = 0x%010x\n" % (i, vals[1 + i]) for i in (0, 1, 2))
    wt = "W0 = 0x%010x\nW1 = 0x%010x\n" % (vals[1 + k % 4], vals[4])
    return fe.ProverRun(label, "SET_MEMBER W0 I0 W1 I1 I2\n", inst, wt, test_seed=k, ctx=ctx)


@pytest.fixture(scope="module")
def cfg5(ctx):
    items = [item_of_run(ctx, cfg5_run(ctx, k), k)[0] for k in range(128)]
    yield items
    destroy(ctx, items)


def test_config5_shapes_byte_equal(ctx, cfg5):
    got = check_equal(ctx, cfg5)
    # and they verify, batched
    assert ctx.verify_batch([(it[0], it[1], V, proof, os.urandom(32)) for it, (proof, V) in zip(cfg5, got)]) == [True] * len(cfg5)


def test_reference_fixtures_in_one_batch(ctx):
    from bulletproofs_gadgets_b200 import frontend as fe
    rd = lambda nm: open(os.path.join(FX, nm)).read()
    items = []
    for k, name in enumerate(["bounds_check", "equality", "inequality", "less_than", "or3"]):  # every fixture with N <= 4096
        run = fe.ProverRun(b"fixtures/" + name.encode(), rd(name + ".gadgets"), rd(name + ".inst"), rd(name + ".wtns"), test_seed=7, ctx=ctx)
        items.append(item_of_run(ctx, run, k)[0])
    check_equal(ctx, items)
    destroy(ctx, items)


def test_edge_circuits(ctx):
    insts = [circuits.chain_instance(0, 11), circuits.chain_instance(1, 12), no_commitment_instance(5, 13), no_commitment_instance(0, 14),
             circuits.chain_instance(13, 15), circuits.chain_instance(100, 16)]
    items = [item_of_instance(ctx, inst, k)[0] for k, inst in enumerate(insts)]
    check_equal(ctx, items)
    destroy(ctx, items)


def test_mixed_sizes_leave_the_lockstep_at_different_rounds(ctx):
    insts = [circuits.chain_instance(n, 20 + k) for k, n in enumerate([1, 8, 512, 4096, 300, 2, 4000])]
    items = [item_of_instance(ctx, inst, k)[0] for k, inst in enumerate(insts)]
    got = check_equal(ctx, items)
    # CPU oracle parity on a handful of them
    for k in (0, 1, 2, 5):
        rp, tv, tc = insts[k]["csr"]
        assert ol.r1cs_prove(insts[k]["label"], 512, insts[k]["aL"], insts[k]["aR"], insts[k]["aO"], insts[k]["vals"], insts[k]["blinds"], rp, tv, tc,
                             ext_of(k)) == got[k]
    destroy(ctx, items)


def test_count_one_and_count_above_the_pass_size(ctx):
    it = item_of_instance(ctx, circuits.chain_instance(37, 30), 0)[0]
    check_equal(ctx, [it])
    destroy(ctx, [it])
    # 2^17 padded elements per pass: 34 proofs of N = 4096 plus small ones take two passes
    insts = [circuits.random_dense_instance(4000, 40 + k) for k in range(34)] + [circuits.chain_instance(9, 90), circuits.chain_instance(70, 91)]
    items = [item_of_instance(ctx, inst, k)[0] for k, inst in enumerate(insts)]
    check_equal(ctx, items)
    destroy(ctx, items)


def test_more_proofs_than_one_pass_holds(ctx):
    """1 100 tiny statements (N = 1 and N = 2) exceed the 1 024 proofs of one pass; each must still equal bpg_r1cs_prove"""
    base = [item_of_instance(ctx, circuits.chain_instance(n, 110 + n), 0)[0] for n in (1, 2)]
    items = [base[k % 2][:7] + (ext_of(1000 + k),) for k in range(1100)]
    check_equal(ctx, items)
    destroy(ctx, base)


def test_large_proof_is_delegated(ctx):
    from bulletproofs_gadgets_b200 import frontend as fe
    rd = lambda nm: open(os.path.join(FX, nm)).read()
    run = fe.ProverRun(b"fixtures/example", rd("example.gadgets"), rd("example.inst"), rd("example.wtns"), test_seed=3, ctx=ctx)
    big = item_of_run(ctx, run, 0)[0]
    assert run.prover.num_vars > 8192  # N = 2^14
    small = [item_of_instance(ctx, circuits.chain_instance(n, 50 + n), 1 + k)[0] for k, n in enumerate([3, 200])]
    check_equal(ctx, [small[0], big, small[1]])
    destroy(ctx, [big] + small)


def test_legacy_framing(ctx):
    items = [item_of_instance(ctx, circuits.chain_instance(n, 60 + n), n)[0] for n in (4, 33, 0)]
    got = check_equal(ctx, items, FLAG_LEGACY)
    assert all(len(p) % 32 == 0 for p, _ in got)
    got2 = check_equal(ctx, items, FLAG_NO_LATE)  # a no-op at these sizes
    assert [p[0] for p, _ in got2] == [0, 0, 0]
    destroy(ctx, items)


def test_wrong_witness_is_rejected(ctx):
    insts = [circuits.chain_instance(20, 70), circuits.chain_instance(20, 71, wrong=True), circuits.chain_instance(64, 72)]
    items = [item_of_instance(ctx, inst, k)[0] for k, inst in enumerate(insts)]
    got = check_equal(ctx, items)
    verdicts = ctx.verify_batch([(it[0], it[1], V, proof, os.urandom(32)) for it, (proof, V) in zip(items, got)])
    assert verdicts == [True, False, True]
    # the single path's proof of the wrong witness is the same bytes and is rejected as well
    acc = C.c_int(-1)
    proof, V = single(ctx, items[1])
    ctx.check(ctx.lib.bpg_r1cs_verify(ctx.h, items[1][0], items[1][1], len(items[1][1]), V, proof, len(proof), os.urandom(32), 0, C.byref(acc)))
    assert acc.value == 0
    destroy(ctx, items)


def _nothing_written(res, n):
    rc, proofs, Vs, lens = res
    assert lens == [0] * n
    assert all(p == bytes(CAP) for p in proofs) and all(v == bytes(len(v)) for v in Vs)
    return rc


def test_bad_arguments_fail_whole_and_write_nothing(ctx):
    items = [item_of_instance(ctx, circuits.chain_instance(n, 80 + n), n)[0] for n in (3, 40, 7)]
    n = len(items)
    assert _nothing_written(raw_call(ctx, items, null_circuit_at=1), n) == E_ARG
    caps = [CAP, 1 + 32 * (11 + 2 * 6 + 2) - 1, CAP]  # proof 1 (N = 64) needs 1 + 32 * 25 bytes
    assert _nothing_written(raw_call(ctx, items, caps=caps), n) == E_SIZE
    caps[1] += 1
    rc, _, _, lens = raw_call(ctx, items, caps=caps)
    assert rc == 0 and lens[1] == caps[1]
    for flag in (FLAG_FAST, FLAG_WOD, FLAG_FORCE_LATE):
        assert _nothing_written(raw_call(ctx, items, flags=flag), n) == E_ARG
    assert ctx.lib.bpg_r1cs_prove_batch(ctx.h, 0, None, None, None, None, None, None, None, None, None, 0, None, None, None, None) == 0
    # generator capacity (16384) below N of the middle proof (2^15)
    mid = [item_of_instance(ctx, circuits.chain_instance(n, 85), n)[0] for n in (3, 16385, 7)]
    assert _nothing_written(raw_call(ctx, mid), n) == E_SIZE
    destroy(ctx, mid + items)


def test_sharded_context_is_rejected(ctx):
    import bulletproofs_gadgets_b200 as bpg
    sh = bpg.Context(0)
    sh.gens_ensure(64)
    send, recv = sh.dev_alloc(1 << 18), sh.dev_alloc(2 << 18)
    CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t)
    calls = []
    cb = CB(lambda user, nbytes: calls.append(nbytes) or 1)
    try:
        sh.check(sh.lib.bpg_ctx_set_shard(sh.h, 0, 2, send, recv, 1 << 18, C.cast(cb, C.c_void_p), None))
        items = [item_of_instance(sh, circuits.chain_instance(n, 95 + n), n)[0] for n in (3, 9)]
        assert _nothing_written(raw_call(sh, items), 2) == E_ARG
        assert calls == []
        destroy(sh, items)
        sh.check(sh.lib.bpg_ctx_set_shard(sh.h, 0, 1, None, None, 0, None, None))
    finally:
        sh.dev_free(send)
        sh.dev_free(recv)
        sh.close()


def test_launches_stay_below_three_single_proofs(ctx, cfg5):
    batch = cfg5[:64]
    l0 = ctx.launch_count()
    ctx.prove_batch(batch)
    l1 = ctx.launch_count()
    largest = max(batch, key=lambda it: len(it[2]))
    single(ctx, largest)
    l2 = ctx.launch_count()
    assert (l1 - l0) < 3 * (l2 - l1), (l1 - l0, l2 - l1)


def test_api_prove_batch_matches_prover_prove(ctx):
    from bulletproofs_gadgets_b200 import api
    gens = api.BulletproofGens(4096, ctx=ctx)
    runs = [cfg5_run(ctx, k) for k in range(6)]
    exts = [ext_of(100 + k) for k in range(6)]
    got = api.prove_batch([r.prover for r in runs], gens, exts)
    assert got == [r.prover.prove(gens, ext_rng32=e) for r, e in zip(runs, exts)]
    with pytest.raises(ValueError):
        api.prove_batch([r.prover for r in runs], gens, exts[:-1])
