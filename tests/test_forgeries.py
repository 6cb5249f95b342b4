"""Forged proofs that are valid except for one encoding, scalar or identity check (tests/forgeries.py) must be rejected on
every verification path: bpg_r1cs_verify (both decode kernels), bpg_r1cs_verify_batch alone and mixed with valid proofs
(combined check, then the per-proof fallback), bpg_r1cs_verify_each and the Python API, with the CPU oracle's verdict
proof by proof.  The CPU tests pin the forging prover to the reference prover and show that every forgery is rejected by
the strict big-integer verifier and accepted by the lax one it names: each is a relaxation a device check could make.
The last tests compare the decode of every MSM entry point with the oracle on non-canonical and invalid encodings."""
import random

import pytest

import circuits
import forgeries as fg
import oracle_lib as ol
from forgeries import FLAG_LEGACY, corpus, ol_verify, pr_verify
from oracle import pyref as pr
from test_oracle import BAD_ENCODINGS, RISTRETTO_MULTIPLES

L, P = pr.L, pr.P
E_DECOMPRESS = -3


# ----------------------------------------------------------------------------- CPU: the forging prover and the corpus
@pytest.mark.parametrize("n", [0, 1, 3, 8, 13])
def test_forge_prove_without_hooks_is_the_reference_prover(n):
    seed = 100 + n
    inst = circuits.chain_instance(n, seed)
    cs = pr.ConstraintSystem(pr.Transcript(inst["label"]), True)
    Vv = [cs.commit(v, b)[1] for v, b in zip(inst["ivals"], inst["iblinds"])]
    circuits.chain_wire(cs, Vv, seed + 1000, n)
    want, _ = pr.r1cs_prove(cs, 64, fg.EXT)
    rp, tv, tc = inst["csr"]
    want_c, V = ol.r1cs_prove(inst["label"], 64, inst["aL"], inst["aR"], inst["aO"], inst["vals"], inst["blinds"], rp, tv, tc, fg.EXT)
    st = fg.chain(n, seed)
    assert st.csr == inst["csr"]
    assert st.prove() == (want, V) == (want_c, V)
    assert V == b"".join(cs.V)
    for framing, flags in (("v1", 0), ("legacy", FLAG_LEGACY)):
        proof, V1 = st.prove(framing=framing)
        assert V1 == V
        assert proof == (b"\x01" + want[1:97] + bytes(96) + want[97:] if framing == "v1" else want[1:97] + bytes(96) + want[97:])
        assert ol_verify(st, V, proof, flags)
    if n <= 3:
        assert pr_verify(st, V, st.prove(framing="legacy")[0], FLAG_LEGACY)


def test_every_forgery_is_rejected_strictly_and_accepted_by_its_lax_verifier():
    fs = corpus()
    assert len({f.name for f in fs}) == len(fs)
    assert {f.lax for f in fs} == {"reduce_scalars", "mask_scalars", "mask_decode", "reduce_decode", "no_identity", "drop_phase2", "skip_zero"}
    assert {f.st.n for f in fs} >= set(fg.SIZES)
    for f in fs:
        assert f.proof != f.twin[0] or f.V != f.twin[1], f
        assert ol_verify(f.st, f.twin[1], f.twin[0], f.flags), f
        assert not ol_verify(f.st, f.V, f.proof, f.flags), f
        assert not pr_verify(f.st, f.V, f.proof, f.flags), f
        with fg.lax(f.lax):
            assert pr_verify(f.st, f.V, f.proof, f.flags), f
    # the honest twins of every class are accepted by the big-integer verifier too
    for f in {f.lax: f for f in fs if f.st.n <= 3}.values():
        assert pr_verify(f.st, f.twin[1], f.twin[0], f.flags), f


def test_the_identity_forgeries_hold_exactly_one_identity():
    for f in corpus():
        if f.lax == "no_identity":
            pts = [f.proof[1 + 32 * i:33 + 32 * i] for i in range(8)]  # A_I1, A_O1, S1, T_1, T_3 .. T_6
            assert pts.count(fg.IDENTITY) == 1 and fg.IDENTITY not in [f.twin[0][1 + 32 * i:33 + 32 * i] for i in range(8)], f


def test_a_cancelling_pair_sums_to_the_identity_under_equal_weights():
    st = fg.chain(3, 43)
    proof, V = st.prove()
    P1, P2 = (fg.verification_point(st, V, p) for p in fg.cancelling_pair(proof))
    assert pr.pt_eq(fg.verification_point(st, V, proof), pr.IDENT)
    assert not pr.pt_eq(P1, pr.IDENT) and not pr.pt_eq(P2, pr.IDENT)
    assert pr.pt_eq(pr.pt_add(P1, P2), pr.IDENT)
    for p in fg.cancelling_pair(proof):
        assert not ol_verify(st, V, p) and not pr_verify(st, V, p)


def encoding_corpus():
    """RFC 9496 bad encodings, p + j, 2^255 - 1, valid multiples of B and each of them with bit 255 set"""
    good = [bytes.fromhex(h) for h in RISTRETTO_MULTIPLES]
    return ([bytes.fromhex(h) for h in BAD_ENCODINGS] + [(P + j).to_bytes(32, "little") for j in range(19)] + [((1 << 255) - 1).to_bytes(32, "little")]
            + good + [fg.high_bit(e) for e in good])


def test_encoding_corpus_decodes_as_rfc_9496():
    for e in encoding_corpus():
        ok = pr.ristretto_decode(e) is not None
        assert ok == bool(ol.lib().bpo_point_decode_ok(e)), e.hex()
        assert ok == (e in [bytes.fromhex(h) for h in RISTRETTO_MULTIPLES]), e.hex()
        # the oracle's MSM decodes a point whose scalar is 0
        assert (ol.msm(bytes(32) + pr.sc_bytes(3), e + bytes.fromhex(RISTRETTO_MULTIPLES[1])) is not None) == ok, e.hex()


# ----------------------------------------------------------------------------- GPU: every forgery through every path
@pytest.fixture(scope="module")
def ctx():
    import bulletproofs_gadgets_b200 as bpg
    c = bpg.Context(0)
    c.gens_ensure(16384)
    yield c
    c.close()


def ext_of(k):
    return bytes([k % 251 + 1]) * 32


def circuit(ctx, st):
    from test_gpu_prove_batch import circuit as make
    return make(ctx, st.n, st.m, st.csr)


@pytest.fixture(scope="module")
def forged(ctx):
    """[(forgery, its verify item, its twin's verify item)]"""
    out = []
    for k, f in enumerate(corpus()):
        h = circuit(ctx, f.st)
        out.append((f, (h, f.st.label, f.V, f.proof, ext_of(k)), (h, f.st.label, f.twin[1], f.twin[0], ext_of(k + 1))))
    yield out
    for _, it, _ in out:
        ctx.lib.bpg_circuit_destroy(it[0])


@pytest.fixture(scope="module")
def valid(ctx):
    """eight valid proofs from the GPU prover per framing flag (0 and legacy), with their oracle cases"""
    from test_gpu_verify_lockstep import Case
    pools = {}
    for flags in (0, FLAG_LEGACY):
        case = Case(ctx)
        case.prove([circuits.chain_instance(n, 3000 + 10 * flags + k) for k, n in enumerate((0, 1, 2, 3, 5, 8, 13, 40))], flags)
        pools[flags] = case
    yield pools
    for case in pools.values():
        case.destroy()


def single(ctx, it, flags):
    from test_gpu_verify_lockstep import single as verify
    return verify(ctx, it, flags)


def oracle_of(st, it, flags):
    return ol_verify(st, it[2], it[3], flags)


@pytest.mark.gpu
def test_single_verify_rejects_every_forgery(ctx, forged):
    for f, it, tw in forged:
        assert oracle_of(f.st, it, f.flags) is False and oracle_of(f.st, tw, f.flags) is True, f
        assert single(ctx, it, f.flags) is False, f
        assert single(ctx, tw, f.flags) is True, f


@pytest.mark.gpu
def test_batch_of_one_rejects_every_forgery(ctx, forged):
    """a lone proof is checked with weight 1 and no fallback"""
    for f, it, tw in forged:
        assert ctx.verify_batch([it], f.flags) == [False], f
        assert ctx.verify_batch([tw], f.flags) == [True], f


@pytest.mark.gpu
def test_batch_rejects_every_forgery_among_valid_proofs(ctx, forged, valid):
    for f, it, tw in forged:
        pool = valid[f.flags].items
        assert ctx.verify_batch(pool[:4] + [it] + pool[4:], f.flags) == [True] * 4 + [False] + [True] * 4, f
        assert ctx.verify_batch(pool[:3] + [tw] + pool[3:], f.flags) == [True] * 9, f
    for flags in (0, FLAG_LEGACY):  # all forgeries and twins of a framing in one call
        group = [(it, tw) for f, it, tw in forged if f.flags == flags]
        items = [x for pair in group for x in pair] + valid[flags].items
        want = [k % 2 == 1 for k in range(2 * len(group))] + [True] * 8
        assert ctx.verify_batch(items, flags) == want


@pytest.mark.gpu
def test_verify_each_rejects_every_forgery(ctx, forged, valid):
    for f, it, tw in forged:
        assert ctx.verify_each([it, tw], f.flags) == [False, True], f
    for flags in (0, FLAG_LEGACY):
        group = [(it, tw) for f, it, tw in forged if f.flags == flags]
        items = valid[flags].items[:4] + [x for pair in group for x in pair] + valid[flags].items[4:]
        assert ctx.verify_each(items, flags) == [True] * 4 + [k % 2 == 1 for k in range(2 * len(group))] + [True] * 4


def api_verifier(ctx, st, V):
    import bulletproofs_gadgets_b200 as bpg
    v = bpg.Verifier(st.label, ctx)
    for i in range(st.m):
        v.commit(V[32 * i:32 * i + 32])
    v.num_vars = st.n
    rp, tv, tc = st.csr
    v.row_ptr, v.term_var, v.term_coeff = list(rp), list(tv), bytearray(tc)
    return v


@pytest.mark.gpu
def test_api_rejects_every_forgery(ctx, forged):
    import bulletproofs_gadgets_b200 as bpg
    for flags in (0, FLAG_LEGACY):
        fs = [f for f, _, _ in forged if f.flags == flags]
        for f in fs:
            with pytest.raises(bpg.R1CSError):
                api_verifier(ctx, f.st, f.V).verify(f.proof, flags=flags)
            api_verifier(ctx, f.st, f.twin[1]).verify(f.twin[0], flags=flags)
        verifiers = [api_verifier(ctx, f.st, V) for f in fs for V in (f.V, f.twin[1])]
        proofs = [p for f in fs for p in (f.proof, f.twin[0])]
        assert bpg.api.verify_each(verifiers, proofs, flags=flags) == [k % 2 == 1 for k in range(len(proofs))]
        assert bpg.api.verify_batch(verifiers, proofs, flags=flags) == [k % 2 == 1 for k in range(len(proofs))]


@pytest.mark.gpu
def test_forged_own_points_on_the_bucket_decode_path(ctx, valid):
    """m = 8 200 commitments (and one no constraint references): bpg_r1cs_verify decodes the proof's own points with
    k_decompress_an_kernel for the bucket engine, bpg_r1cs_verify_each with its per-term kernel"""
    from test_gpu_verify_each import many_commitments_instance
    st = fg.from_instance(many_commitments_instance(8200, 1300))
    st.add_commitment(5, 6)
    twin = st.prove()
    forgeries = [("high bit V_4000", st.prove(enc=fg.on("V", 4000, fg.high_bit))),
                 ("unused V_8200 = bad encoding 7", st.prove(enc=fg.on("V", 8200, lambda e: bytes.fromhex(BAD_ENCODINGS[7]))))]
    h = circuit(ctx, st)
    try:
        items = [(h, st.label, twin[1], twin[0], ext_of(0))] + [(h, st.label, V, proof, ext_of(k + 1)) for k, (_, (proof, V)) in enumerate(forgeries)]
        want = [True, False, False]
        assert [oracle_of(st, it, 0) for it in items] == want
        assert [single(ctx, it, 0) for it in items] == want
        pool = valid[0].items
        assert ctx.verify_each(pool[:2] + items + pool[2:4], 0) == [True] * 2 + want + [True] * 2
        assert ctx.verify_batch(pool[:2] + items + pool[2:4], 0) == [True] * 2 + want + [True] * 2
    finally:
        ctx.lib.bpg_circuit_destroy(h)


@pytest.mark.gpu
def test_scalar_forgeries_of_a_proof_on_the_per_proof_path(ctx, valid):
    """n = 5 000 (N = 8 192 > 4 096): the batch calls check this proof with the single-proof finish"""
    from test_gpu_verify_lockstep import Case
    case = Case(ctx)
    case.prove([circuits.chain_instance(5000, 1400)])
    big = case.items[0]
    assert case.check() == [True]
    forged = [(name, big[:3] + (proof,) + big[4:]) for name, proof, _ in fg.scalar_forgeries(big[3])]
    assert len(forged) == 15
    pool = valid[0].items
    items = pool[:4] + [it for _, it in forged] + [big] + pool[4:]
    want = [True] * 4 + [False] * len(forged) + [True] * 5
    rp, tv, tc = case.oracle[0][1]
    assert [ol.r1cs_verify(it[1], 8192, 5000, it[2], rp, tv, tc, it[3], bytes(32)) for _, it in forged] == [False] * len(forged)
    assert ctx.verify_batch(items) == want
    assert ctx.verify_each(items) == want
    for name, it in forged:
        assert single(ctx, it, 0) is False, name
        assert ctx.verify_batch([it, big]) == [False, True], name
    case.destroy()


@pytest.mark.gpu
def test_batch_rejects_both_proofs_of_a_cancelling_pair(ctx, valid):
    pool = valid[0]
    for k in (2, 5):  # n = 2 and n = 8
        it = pool.items[k]
        pair = [it[:3] + (p,) + it[4:] for p in fg.cancelling_pair(it[3])]
        n, csr, cap = pool.oracle[k]
        assert [ol.r1cs_verify(x[1], cap, n, x[2], *csr, x[3], bytes(32)) for x in pair] == [False, False]
        items = pool.items[:3] + [pair[0]] + pool.items[3:6] + [pair[1]] + pool.items[6:]
        want = [True] * 3 + [False] + [True] * 3 + [False] + [True] * 2
        assert ctx.verify_batch(items) == want
        assert ctx.verify_each(items) == want
        assert ctx.verify_batch(pair) == [False, False]
        assert [single(ctx, x, 0) for x in pair] == [False, False]


@pytest.mark.gpu
def test_an_all_valid_batch_passes_the_combined_check(ctx):
    """64 valid proofs take fewer launches than the same batch with one false proof, whose failing combined check is
    followed by the per-proof check: the combined check accepts an all-valid batch without the fallback"""
    from test_gpu_verify_lockstep import Case
    case = Case(ctx)
    case.prove([circuits.chain_instance((k * 37) % 300, 1500 + k) for k in range(64)])
    items = list(case.items)
    bad = list(items)
    bad[17] = items[17][:3] + (fg.cancelling_pair(items[17][3])[0],) + items[17][4:]
    l0 = ctx.launch_count()
    assert ctx.verify_batch(items) == [True] * 64
    l1 = ctx.launch_count()
    assert ctx.verify_batch(bad) == [k != 17 for k in range(64)]
    l2 = ctx.launch_count()
    assert l1 - l0 < l2 - l1, (l1 - l0, l2 - l1)
    case.destroy()


# ----------------------------------------------------------------------------- GPU: decode parity of the MSM entry points
def outcome(fn, *args):
    from bulletproofs_gadgets_b200 import BpgError
    try:
        return fn(*args)
    except BpgError as e:
        return e.code


def want_of(res):
    return E_DECOMPRESS if res is None else res


@pytest.mark.gpu
@pytest.mark.parametrize("n", [100, 8192])
def test_msm_decode_matches_the_oracle(ctx, n):
    """bpg_msm below (k_decompress_kernel) and at (k_decompress_an_kernel) the bucket threshold: each encoding at one
    position among valid points, with scalar 0 there"""
    rnd = random.Random(n)
    G, _ = ol.gens(0, n)
    scalars = bytearray(b"".join(pr.sc_bytes(rnd.randrange(L)) for _ in range(n)))
    for j, e in enumerate(encoding_corpus()):
        pos = (j * 7919) % n
        sc = bytes(scalars[:32 * pos]) + bytes(32) + bytes(scalars[32 * pos + 32:])
        pts = G[:32 * pos] + e + G[32 * pos + 32:]
        assert outcome(ctx.msm, sc, pts) == want_of(ol.msm(sc, pts)), (n, pos, e.hex())


@pytest.mark.gpu
def test_msm_gens_extras_decode_matches_the_oracle(ctx):
    rnd = random.Random(17)
    n = 64
    sG = b"".join(pr.sc_bytes(rnd.randrange(L)) for _ in range(n))
    sH = b"".join(pr.sc_bytes(rnd.randrange(L)) for _ in range(n))
    good = [bytes.fromhex(h) for h in RISTRETTO_MULTIPLES[1:]]
    for j, e in enumerate(encoding_corpus()):
        pos = j % (len(good) + 1)
        pts = good[:pos] + [e] + good[pos:]
        es = b"".join(bytes(32) if p is e else pr.sc_bytes(rnd.randrange(L)) for p in pts)
        got = outcome(ctx.msm_gens, sG, sH, n, 3, es, b"".join(pts))
        assert got == want_of(ol.msm_gens(sG, sH, n, 3, es, b"".join(pts))), (pos, e.hex())


@pytest.mark.gpu
def test_fold_points_decode_matches_the_oracle(ctx):
    rnd = random.Random(18)
    n = 16
    G, H = ol.gens(0, n)
    sl, sr = pr.sc_bytes(rnd.randrange(L)), pr.sc_bytes(rnd.randrange(L))
    for j, e in enumerate(encoding_corpus()):
        pos = (5 * j) % n
        PL, PR = (G, H[:32 * pos] + e + H[32 * pos + 32:]) if j % 2 else (G[:32 * pos] + e + G[32 * pos + 32:], H)
        assert outcome(ctx.fold_points, sl, sr, PL, PR) == want_of(ol.fold_points(sl, sr, PL, PR)), (pos, e.hex())
