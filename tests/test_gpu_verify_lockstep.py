"""Batch verification with lockstep preparation: bpg_r1cs_verify_batch prepares every replayed proof with padded N <= 4096 in
passes of one set of launches for all of them, and sums the G/H scalars of a checked set in one launch.  Every verdict must
equal bpg_r1cs_verify of that proof alone and the CPU oracle's, for every failure kind, edge shapes, mixed sizes (a proof of
N = 2^13 taking the per-proof path in the same call), a shared circuit handle, the legacy framing, a proof beyond the
generator capacity, calls above the per-pass proof and element limits and the front-end's configs[4] statements; the
launches of a call must not grow with its proof count."""
import ctypes as C
import hashlib
import random

import pytest

import circuits
import oracle_lib as ol
from test_gpu_batch_verify import make_items
from test_gpu_prove_batch import item_of_instance, no_commitment_instance

pytestmark = pytest.mark.gpu
FLAG_LEGACY = 1
# Preparing one proof at a time took 6-7 launches per proof before the first check (at least 384 for 64 proofs), and every
# combined check of a set took one more launch per proof in it; in lockstep the call below takes under 200.
LAUNCH_BOUND_ONE_BAD_OF_64 = 384


@pytest.fixture(scope="module")
def ctx():
    import bulletproofs_gadgets_b200 as bpg
    c = bpg.Context(0)
    c.gens_ensure(16384)
    yield c
    c.close()


def ext_of(k):
    return hashlib.sha256(b"verify lockstep ext %d" % k).digest()


def single(ctx, it, flags=0):
    acc = C.c_int(-1)
    ctx.check(ctx.lib.bpg_r1cs_verify(ctx.h, it[0], it[1], len(it[1]), it[2], it[3], len(it[3]), it[4], flags, C.byref(acc)))
    return bool(acc.value)


def flip(proof, pos):
    b = bytearray(proof)
    b[pos] ^= 1
    return bytes(b)


def pow2(n):
    N = 1
    while N < n:
        N *= 2
    return N


class Case:
    """verify items (handle, label, V, proof, ext) with what the oracle needs to check each one"""

    def __init__(self, ctx):
        self.ctx, self.items, self.oracle, self.handles = ctx, [], [], []

    def prove(self, insts, flags=0, tamper=None):
        """proves tests/circuits.py instances on the GPU and adds them; tamper(k, proof) may alter proof k"""
        made = [item_of_instance(self.ctx, inst, len(self.items) + k) for k, inst in enumerate(insts)]
        got = self.ctx.prove_batch([it for it, _ in made], flags)
        for k, ((it, csr), (proof, V), inst) in enumerate(zip(made, got, insts)):
            if tamper:
                proof = tamper(k, proof)
            self.add((it[0], it[1], V, proof, ext_of(len(self.items))), inst["n"], csr)
            self.handles.append(it[0])

    def add(self, item, n, csr, cap=None):
        self.items.append(item)
        self.oracle.append((n, csr, cap or max(8, pow2(n))))

    def check(self, flags=0, expect=None):
        got = self.ctx.verify_batch(self.items, flags)
        assert got == [single(self.ctx, it, flags) for it in self.items]
        want = [ol.r1cs_verify(it[1], cap, n, it[2], csr[0], csr[1], csr[2], it[3], bytes(32), flags) for it, (n, csr, cap) in zip(self.items, self.oracle)]
        assert got == want
        if expect is not None:
            assert got == expect
        return got

    def destroy(self):
        for h in self.handles:
            self.ctx.lib.bpg_circuit_destroy(h)


def test_every_failure_kind_mixed_with_valid_proofs(ctx):
    good, want_g = make_items(ctx, 40, 501, 0)
    bad, want_b = make_items(ctx, 48, 502, 1)  # every item one of the six failure kinds
    order = list(range(len(good) + len(bad)))
    random.Random(3).shuffle(order)
    items, want = [(good + bad)[k] for k in order], [(want_g + want_b)[k] for k in order]
    got = ctx.verify_batch(items)
    assert got == want
    assert [single(ctx, it) for it in items] == want
    for it in good + bad:
        ctx.lib.bpg_circuit_destroy(it[0])


def test_edge_shapes(ctx):
    case = Case(ctx)
    insts = [circuits.chain_instance(0, 11), circuits.chain_instance(1, 12), no_commitment_instance(5, 13), no_commitment_instance(0, 14),
             circuits.chain_instance(13, 15), circuits.chain_instance(100, 16), circuits.chain_instance(3, 17, wrong=True)]
    case.prove(insts, tamper=lambda k, p: flip(p, len(p) - 40) if k == 4 else p)
    assert case.check() == [True, True, True, True, False, True, False]
    case.destroy()


def test_mixed_sizes_and_a_proof_on_the_per_proof_path(ctx):
    case = Case(ctx)
    sizes = [8, 4096, 30, 5000, 200, 1000, 3, 2048, 4000]  # 5000: N = 2^13 > 4096
    insts = [circuits.chain_instance(n, 200 + k) for k, n in enumerate(sizes)]
    case.prove(insts)
    assert case.check() == [True] * len(sizes)
    # the same proofs with the large one and a lockstep one tampered: bisection runs through both paths
    for k in (1, 3):
        h, label, V, proof, ext = case.items[k]
        case.items[k] = (h, label, V, flip(proof, 1 + 32 * 3 + 5), ext)
    assert case.check() == [k not in (1, 3) for k in range(len(sizes))]
    case.destroy()


def test_one_circuit_handle_shared_by_many_proofs(ctx):
    inst = circuits.chain_instance(57, 300)
    it, csr = item_of_instance(ctx, inst, 0)
    exts = [ext_of(3000 + k) for k in range(40)]
    got = ctx.prove_batch([it[:7] + (e,) for e in exts])
    case = Case(ctx)
    for k, (proof, V) in enumerate(got):
        case.add((it[0], it[1], V, flip(proof, len(proof) - 70) if k % 13 == 5 else proof, ext_of(k)), inst["n"], csr)
    case.handles.append(it[0])
    assert case.check() == [k % 13 != 5 for k in range(40)]
    case.destroy()


def test_legacy_framing(ctx):
    case = Case(ctx)
    case.prove([circuits.chain_instance(n, 400 + n) for n in (4, 33, 0, 260)], flags=FLAG_LEGACY,
               tamper=lambda k, p: flip(p, 200) if k == 1 else p)
    assert all(len(it[3]) % 32 == 0 for it in case.items)
    assert case.check(FLAG_LEGACY) == [True, False, True, True]
    case.destroy()


def test_proof_beyond_the_generator_capacity_is_rejected(ctx):
    """a circuit whose padded N exceeds the generators the device holds: the replay rejects its proof (no device work), the
    lockstep proofs of the same call are unaffected"""
    cap = ctx.gens_capacity()
    case = Case(ctx)
    case.prove([no_commitment_instance(5, 520), circuits.chain_instance(40, 521)])
    h = C.c_void_p()
    ctx.check(ctx.lib.bpg_circuit_create(ctx.h, cap + 1, 0, 0, (C.c_uint32 * 1)(0), (C.c_uint32 * 1)(), b"", C.byref(h)))
    case.handles.append(h)
    _, label, V, proof, _ = case.items[0]  # a valid proof of m = 0 whose statement now claims cap + 1 multipliers
    case.add((h, label, V, proof, ext_of(99)), cap + 1, ([0], [], b""), cap=cap)
    assert case.check() == [True, True, False]
    case.destroy()


def test_more_proofs_than_one_pass_holds(ctx):
    """1 100 tiny proofs (N = 1, 2) exceed the 1 024 proofs of one pass"""
    base = [item_of_instance(ctx, circuits.chain_instance(n, 600 + n), 0) for n in (1, 2)]
    got = ctx.prove_batch([base[k % 2][0][:7] + (ext_of(5000 + k),) for k in range(1100)])
    case = Case(ctx)
    for k, (proof, V) in enumerate(got):
        it, csr = base[k % 2]
        case.add((it[0], it[1], V, flip(proof, 40) if k in (3, 1030) else proof, ext_of(k)), k % 2 + 1, csr)
    case.handles += [it[0] for it, _ in base]
    assert case.check() == [k not in (3, 1030) for k in range(1100)]
    case.destroy()


def test_more_padded_elements_than_one_pass_holds(ctx):
    """33 proofs of N = 4096 and small ones: more than the 2^17 padded elements of one pass"""
    case = Case(ctx)
    insts = [circuits.random_dense_instance(4000, 700 + k) for k in range(33)] + [circuits.chain_instance(9, 790), circuits.chain_instance(70, 791)]
    case.prove(insts, tamper=lambda k, p: flip(p, len(p) - 3) if k in (0, 34) else p)
    assert case.check() == [k not in (0, 34) for k in range(35)]
    case.destroy()


def cfg5_item(ctx, k):
    """a BASELINE configs[4] statement as bench._cfg5_assemble builds it (statement k % 100 == 37 false), proved on the GPU"""
    from bulletproofs_gadgets_b200 import frontend as fe
    valid = k % 100 != 37
    rnd = random.Random(60000 + k)
    label = b"cfg5-%d" % k
    if k % 2:
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        if not valid:
            a, b = b, a
        run = fe.ProverRun(label, "LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b), test_seed=k, ctx=ctx)
    else:
        vals = rnd.sample(range(1 << 40), 5)
        member = vals[1 + k % 4] if valid else vals[0]
        inst = "".join("I%d = 0x%010x\n" % (i, vals[1 + i]) for i in (0, 1, 2))
        wt = "W0 = 0x%010x\nW1 = 0x%010x\n" % (member, vals[4])
        run = fe.ProverRun(label, "SET_MEMBER W0 I0 W1 I1 I2\n", inst, wt, test_seed=k, ctx=ctx)
    p = run.prover
    enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
    aL, aR, aO = p.witness_bytes()
    return (p._circuit(len(p.v)), label, aL, aR, aO, enc(p.v), enc(p.v_blinding), ext_of(k)), p.csr(), p.num_vars, valid


@pytest.fixture(scope="module")
def cfg5(ctx):
    made = [cfg5_item(ctx, k) for k in range(300)]
    got = ctx.prove_batch([m[0] for m in made])
    yield [((it[0], it[1], V, proof, ext_of(k)), csr, n, valid) for k, ((it, csr, n, valid), (proof, V)) in enumerate(zip(made, got))]
    for m in made:
        ctx.lib.bpg_circuit_destroy(m[0][0])


def test_config5_statements_with_false_ones(ctx, cfg5):
    case = Case(ctx)
    for item, csr, n, valid in cfg5:
        case.add(item, n, csr)
    want = [valid for _, _, _, valid in cfg5]
    assert want.count(False) == 3
    assert case.check(expect=want) == want
    for b0 in range(0, len(cfg5), 64):  # the batch size of bench.py's configs[4] extra
        assert ctx.verify_batch(case.items[b0:b0 + 64]) == want[b0:b0 + 64]


def launches(ctx, items):
    l0 = ctx.launch_count()
    got = ctx.verify_batch(items)
    return ctx.launch_count() - l0, got


def test_launches_do_not_grow_with_the_proof_count(ctx, cfg5):
    valid = [item for item, _, _, v in cfg5 if v]
    l16, got16 = launches(ctx, valid[:16])
    l256, got256 = launches(ctx, valid[:256])  # one pass: 128 x 8 + 128 x 512 padded elements
    assert got16 == [True] * 16 and got256 == [True] * 256
    # the preparation is the same launches for both; the check's variable-base MSM over all proofs' own points sums its
    # per-block partials in a tree one level deeper for 16 x the terms
    assert l256 <= l16 + 2, (l16, l256)


def test_one_bad_proof_among_64_is_cheap(ctx, cfg5):
    items = [item for item, _, _, v in cfg5 if v][:64]
    items[21] = items[21][:3] + (flip(items[21][3], 40),) + items[21][4:]
    n, got = launches(ctx, items)
    assert got == [k != 21 for k in range(64)]
    # preparing one at a time took 6 launches per proof before any check
    assert n < LAUNCH_BOUND_ONE_BAD_OF_64, n
