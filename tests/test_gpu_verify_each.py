"""Per-proof verification in one call (bpg_r1cs_verify_each): every verdict must equal bpg_r1cs_verify of that proof alone and
the CPU oracle's, for every failure kind, an undecodable point inside a lockstep pass (only its own proof is rejected), edge
shapes, mixed sizes with a proof on the per-proof path, a shared circuit handle, the legacy framing, a proof beyond the
generator capacity, calls above the per-pass limits (proofs, padded elements, own points) and the configs[4] statements.  The
launches of a call depend on the proofs' shapes only, and bpg_r1cs_verify_batch isolates false proofs with one per-proof
check instead of bisection."""
import ctypes as C
import random

import pytest

import circuits
import oracle_lib as ol
from oracle import pyref as pr
from test_gpu_batch_verify import make_items
from test_gpu_prove_batch import item_of_instance, no_commitment_instance
from test_gpu_verify_lockstep import Case, cfg5_item, ext_of, flip, single
from test_oracle import BAD_ENCODINGS

pytestmark = pytest.mark.gpu
FLAG_LEGACY = 1
E_ARG = -4


@pytest.fixture(scope="module")
def ctx():
    import bulletproofs_gadgets_b200 as bpg
    c = bpg.Context(0)
    c.gens_ensure(16384)
    yield c
    c.close()


class EachCase(Case):
    def check(self, flags=0, expect=None):
        got = self.ctx.verify_each(self.items, flags)
        assert got == [single(self.ctx, it, flags) for it in self.items]
        want = [ol.r1cs_verify(it[1], cap, n, it[2], csr[0], csr[1], csr[2], it[3], bytes(32), flags) for it, (n, csr, cap) in zip(self.items, self.oracle)]
        assert got == want
        if expect is not None:
            assert got == expect
        return got


def launches(ctx, fn, items):
    l0 = ctx.launch_count()
    got = fn(items)
    return ctx.launch_count() - l0, got


def test_every_failure_kind_mixed_with_valid_proofs(ctx):
    good, want_g = make_items(ctx, 40, 801, 0)
    bad, want_b = make_items(ctx, 48, 802, 1)  # every item one of the six failure kinds
    order = list(range(len(good) + len(bad)))
    random.Random(5).shuffle(order)
    items, want = [(good + bad)[k] for k in order], [(want_g + want_b)[k] for k in order]
    assert ctx.verify_each(items) == want
    assert [single(ctx, it) for it in items] == want
    for it in good + bad:
        ctx.lib.bpg_circuit_destroy(it[0])


@pytest.mark.parametrize("where", ["V", "L"])
def test_an_undecodable_point_rejects_only_its_own_proof(ctx, where):
    """one proof of a lockstep pass carries an RFC 9496 bad encoding as a V commitment or as its first L point: the replay
    accepts the bytes, the device decode fails for that proof alone"""
    case = EachCase(ctx)
    case.prove([circuits.chain_instance(n, 900 + n) for n in (3, 20, 8, 64, 5)])
    bad = bytes.fromhex(BAD_ENCODINGS[2])
    h, label, V, proof, ext = case.items[2]
    if where == "V":
        V = V[:32] + bad + V[64:]
    else:  # version byte, 3 (version 0) or 6 (version 1) A points, T_1, T_3..T_6, t_x, t_x~, e~, then L_0
        off = 1 + 32 * ((6 if proof[0] == 1 else 3) + 5 + 3)
        proof = proof[:off] + bad + proof[off + 32:]
    case.items[2] = (h, label, V, proof, ext)
    assert case.check() == [k != 2 for k in range(5)]
    case.destroy()


def test_edge_shapes_and_arguments(ctx):
    case = EachCase(ctx)
    insts = [circuits.chain_instance(0, 11), circuits.chain_instance(1, 12), no_commitment_instance(5, 13), no_commitment_instance(0, 14),
             circuits.chain_instance(13, 15), circuits.chain_instance(100, 16), circuits.chain_instance(3, 17, wrong=True)]
    case.prove(insts, tamper=lambda k, p: flip(p, len(p) - 40) if k == 4 else p)
    assert case.check() == [True, True, True, True, False, True, False]
    for k in range(len(insts)):  # a single proof per call
        assert ctx.verify_each(case.items[k:k + 1]) == [single(ctx, case.items[k])]
    assert ctx.verify_each([]) == []
    lib, n = ctx.lib, 2
    it = case.items[:n]
    circs = (C.c_void_p * n)(*[x[0] for x in it])
    labels = (C.c_char_p * n)(*[x[1] for x in it])
    lens = (C.c_size_t * n)(*[len(x[1]) for x in it])
    Vs = (C.c_char_p * n)(*[x[2] for x in it])
    proofs = (C.c_char_p * n)(*[x[3] for x in it])
    plens = (C.c_size_t * n)(*[len(x[3]) for x in it])
    ext = b"".join(x[4] for x in it)
    acc = (C.c_int * n)(7, 7)
    assert lib.bpg_r1cs_verify_each(ctx.h, 0, None, None, None, None, None, None, None, 0, None) == 0
    assert lib.bpg_r1cs_verify_each(ctx.h, n, None, labels, lens, Vs, proofs, plens, ext, 0, acc) == E_ARG
    assert list(acc) == [0, 0]
    acc = (C.c_int * n)(7, 7)
    nulls = (C.c_void_p * n)(it[0][0], None)
    assert lib.bpg_r1cs_verify_each(ctx.h, n, nulls, labels, lens, Vs, proofs, plens, ext, 0, acc) == E_ARG
    assert list(acc) == [0, 0]
    case.destroy()


def test_mixed_sizes_and_proofs_on_the_per_proof_path(ctx):
    case = EachCase(ctx)
    sizes = [8, 4096, 30, 5000, 200, 1000, 3, 2048, 4000]  # 5000: N = 2^13 > 4096
    case.prove([circuits.chain_instance(n, 200 + k) for k, n in enumerate(sizes)])
    assert case.check() == [True] * len(sizes)
    for k in (1, 3):  # a lockstep proof and the large one tampered
        h, label, V, proof, ext = case.items[k]
        case.items[k] = (h, label, V, flip(proof, 1 + 32 * 3 + 5), ext)
    assert case.check() == [k not in (1, 3) for k in range(len(sizes))]
    case.destroy()


def test_one_circuit_handle_shared_by_many_proofs(ctx):
    inst = circuits.chain_instance(57, 300)
    it, csr = item_of_instance(ctx, inst, 0)
    got = ctx.prove_batch([it[:7] + (ext_of(3000 + k),) for k in range(40)])
    case = EachCase(ctx)
    for k, (proof, V) in enumerate(got):
        case.add((it[0], it[1], V, flip(proof, len(proof) - 70) if k % 13 == 5 else proof, ext_of(k)), inst["n"], csr)
    case.handles.append(it[0])
    assert case.check() == [k % 13 != 5 for k in range(40)]
    case.destroy()


def test_legacy_framing(ctx):
    case = EachCase(ctx)
    case.prove([circuits.chain_instance(n, 400 + n) for n in (4, 33, 0, 260)], flags=FLAG_LEGACY,
               tamper=lambda k, p: flip(p, 200) if k == 1 else p)
    assert case.check(FLAG_LEGACY) == [True, False, True, True]
    case.destroy()


def test_proof_beyond_the_generator_capacity_is_rejected(ctx):
    cap = ctx.gens_capacity()
    case = EachCase(ctx)
    case.prove([no_commitment_instance(5, 520), circuits.chain_instance(40, 521)])
    h = C.c_void_p()
    ctx.check(ctx.lib.bpg_circuit_create(ctx.h, cap + 1, 0, 0, (C.c_uint32 * 1)(0), (C.c_uint32 * 1)(), b"", C.byref(h)))
    case.handles.append(h)
    _, label, V, proof, _ = case.items[0]
    case.add((h, label, V, proof, ext_of(99)), cap + 1, ([0], [], b""), cap=cap)
    assert case.check() == [True, True, False]
    case.destroy()


def test_more_proofs_than_one_pass_holds(ctx):
    """1 100 tiny proofs (N = 1, 2) exceed the 1 024 proofs of one pass"""
    base = [item_of_instance(ctx, circuits.chain_instance(n, 600 + n), 0) for n in (1, 2)]
    got = ctx.prove_batch([base[k % 2][0][:7] + (ext_of(5000 + k),) for k in range(1100)])
    case = EachCase(ctx)
    for k, (proof, V) in enumerate(got):
        it, csr = base[k % 2]
        case.add((it[0], it[1], V, flip(proof, 40) if k in (3, 1030) else proof, ext_of(k)), k % 2 + 1, csr)
    case.handles += [it[0] for it, _ in base]
    assert case.check() == [k not in (3, 1030) for k in range(1100)]
    case.destroy()


def test_more_padded_elements_than_one_pass_holds(ctx):
    """33 proofs of N = 4096 and small ones: more than the 2^17 padded elements of one pass"""
    case = EachCase(ctx)
    insts = [circuits.random_dense_instance(4000, 700 + k) for k in range(33)] + [circuits.chain_instance(9, 790), circuits.chain_instance(70, 791)]
    case.prove(insts, tamper=lambda k, p: flip(p, len(p) - 3) if k in (0, 34) else p)
    assert case.check() == [k not in (0, 34) for k in range(35)]
    case.destroy()


def many_commitments_instance(m, seed):
    """one multiplier and m commitments, each tied to its value (V_i - v_i = 0)"""
    rnd = random.Random(seed)
    a, b = rnd.randrange(pr.L), rnd.randrange(pr.L)
    vals = [rnd.randrange(pr.L) for _ in range(m)]
    rows = [[(("L", 0), 1), (("1", 0), (-a) % pr.L)]] + [[(("V", i), 1), (("1", 0), (-v) % pr.L)] for i, v in enumerate(vals)]
    enc = lambda xs: b"".join(pr.sc_bytes(x) for x in xs)
    return dict(label=b"manycom", n=1, vals=enc(vals), blinds=enc([rnd.randrange(pr.L) for _ in vals]), aL=enc([a]), aR=enc([b]),
                aO=enc([a * b % pr.L]), csr=circuits.to_csr(rows))


def test_a_proof_with_thousands_of_commitments(ctx):
    """m = 9 000: bpg_r1cs_verify takes the variable-base bucket engine for it, bpg_r1cs_verify_each the per-term kernel"""
    case = EachCase(ctx)
    case.prove([circuits.chain_instance(6, 950), many_commitments_instance(9000, 951), many_commitments_instance(9000, 952), circuits.chain_instance(2, 953)],
               tamper=lambda k, p: flip(p, len(p) - 90) if k == 2 else p)
    assert case.check() == [True, True, False, True]
    case.destroy()


@pytest.fixture(scope="module")
def cfg5(ctx):
    made = [cfg5_item(ctx, k) for k in range(300)]
    got = ctx.prove_batch([m[0] for m in made])
    yield [((it[0], it[1], V, proof, ext_of(k)), csr, n, valid) for k, ((it, csr, n, valid), (proof, V)) in enumerate(zip(made, got))]
    for m in made:
        ctx.lib.bpg_circuit_destroy(m[0][0])


def test_config5_statements(ctx, cfg5):
    case = EachCase(ctx)
    for item, csr, n, valid in cfg5:
        case.add(item, n, csr)
    want = [valid for _, _, _, valid in cfg5]
    assert want.count(False) == 3
    assert case.check(expect=want) == want
    for b0 in range(0, len(cfg5), 64):
        assert ctx.verify_each(case.items[b0:b0 + 64]) == want[b0:b0 + 64]


def wrong_witness_pair(ctx):
    """64 chain proofs and the same shapes with every other one proved from a witness that breaks its last constraint"""
    sizes = [(k * 37) % 300 for k in range(64)]
    good, half = EachCase(ctx), EachCase(ctx)
    good.prove([circuits.chain_instance(n, 1200 + k) for k, n in enumerate(sizes)])
    half.prove([circuits.chain_instance(n, 1200 + k, wrong=k % 2 == 1) for k, n in enumerate(sizes)])
    return good, half


def test_launches_do_not_depend_on_which_proofs_are_false(ctx, cfg5):
    good, half = wrong_witness_pair(ctx)
    lg, got_g = launches(ctx, ctx.verify_each, good.items)
    lh, got_h = launches(ctx, ctx.verify_each, half.items)
    assert got_g == [True] * 64 and got_h == [k % 2 == 0 for k in range(64)]
    assert lg == lh, (lg, lh)
    good.destroy()
    half.destroy()
    valid = [item for item, _, _, v in cfg5 if v]
    l16, got16 = launches(ctx, ctx.verify_each, valid[:16])
    l256, got256 = launches(ctx, ctx.verify_each, valid[:256])
    assert got16 == [True] * 16 and got256 == [True] * 256
    assert l256 <= l16 + 2, (l16, l256)


def test_batch_verification_isolates_false_proofs_without_bisection(ctx):
    """a failing combined check is followed by ONE per-proof check of the call: bisection took dozens of checks here"""
    good, half = wrong_witness_pair(ctx)
    want = [k % 2 == 0 for k in range(64)]
    l_batch_good, got = launches(ctx, ctx.verify_batch, good.items)
    assert got == [True] * 64
    l_each, got = launches(ctx, ctx.verify_each, half.items)
    assert got == want
    l_batch_half, got = launches(ctx, ctx.verify_batch, half.items)
    assert got == want
    assert got == [single(ctx, it) for it in half.items]
    assert l_batch_half <= l_batch_good + l_each, (l_batch_half, l_batch_good, l_each)
    good.destroy()
    half.destroy()


def test_api_verify_each_matches_verifier_verify(ctx):
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import frontend as fe
    rnd = random.Random(19)
    cases = []
    for k in range(10):
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        if k % 3 == 1:
            a, b = b, a  # a false statement
        cases.append(("LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b)))
    cases.append(("SET_MEMBER W0 I0 I1\n", "I0 = 0x11\nI1 = 0x64\n", "W0 = 0x64\n"))
    runs = [fe.ProverRun(b"ve-%d" % k, g, i, w, test_seed=k, ctx=ctx) for k, (g, i, w) in enumerate(cases)]
    gens = bpg.BulletproofGens.new(4096, 1, ctx=ctx)
    out = bpg.api.prove_batch([r.prover for r in runs], gens, [ext_of(k) for k in range(len(runs))])
    verifiers, proofs = [], []
    for k, (r, (g, i, _), (proof, V)) in enumerate(zip(runs, cases, out)):
        coms = "".join("%s = 0x%s\n" % (nm, c.hex()) for nm, c in zip(r.coms_names, V))
        verifiers.append(fe.VerifierRun(b"ve-%d" % k, g, i, coms, ctx=ctx).verifier)
        proofs.append(proof if k != 5 else flip(proof, 40))
    got = bpg.api.verify_each(verifiers, proofs)
    want = []
    for v, pf in zip(verifiers, proofs):
        try:
            v.verify(pf)
            want.append(True)
        except bpg.R1CSError:
            want.append(False)
    assert got == want
    assert True in want and False in want
    assert bpg.api.verify_each([], []) == []
    with pytest.raises(ValueError):
        bpg.api.verify_each(verifiers, proofs[:-1])
    other = bpg.Context(0)
    try:
        stranger = fe.VerifierRun(b"ve-x", cases[0][0], cases[0][1], "".join("%s = 0x%s\n" % (nm, c.hex()) for nm, c in zip(runs[0].coms_names, out[0][1])),
                                  ctx=other).verifier
        with pytest.raises(ValueError):
            bpg.api.verify_each(verifiers[:1] + [stranger], proofs[:2])
    finally:
        other.close()
