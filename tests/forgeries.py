"""Forged R1CS proofs for the verifier tests: a prover that can substitute point encodings, override its random draws and
send non-identity phase-2 points, the statements it proves, lax variants of the big-integer verifier, and a corpus of
forgeries that are valid except for one encoding, scalar or identity check.

Every forgery is rejected by a strict verifier and accepted by the lax verifier it names, so a device verifier that made
the same relaxation would accept it (tests/test_forgeries.py)."""
import contextlib
import functools
import random

import circuits
import oracle_lib as ol
from oracle import pyref as pr
from test_oracle import BAD_ENCODINGS, RISTRETTO_MULTIPLES

L, P = pr.L, pr.P
FLAG_LEGACY = 1
IDENTITY = bytes(32)
HIGH_IDENTITY = bytes(31) + b"\x80"  # the identity's encoding with bit 255 set
P_ENC = P.to_bytes(32, "little")  # edff..ff7f: s = p, which reduces to the identity's s = 0
EXT = bytes(range(32))
SIZES = (0, 1, 3, 8)


def _sc(xs):
    return b"".join(pr.sc_bytes(x % L) for x in xs)


def _msm(scalars, points):
    """C-oracle MSM of big-integer scalars and 32-byte encodings -> encoding"""
    return ol.msm(_sc(scalars), b"".join(points))


def high_bit(enc):
    return enc[:31] + bytes([enc[31] | 0x80])


def forge_prove(cs, cap, ext, enc=None, draw=None, phase2=None, framing="v0"):
    """pyref.r1cs_prove of a ConstraintSystem whose commitments were recorded lazily (circuits._lazy_commit: nothing appended
    to the transcript yet) -> (proof bytes, V bytes).  Without hooks the proof is byte-equal to pyref.r1cs_prove's.

    enc(label, index, encoding) -> bytes replaces every point the prover appends to the transcript (V, A_I1 .. S2, T_1 ..
    T_6, L, R); the replacement is what is appended and serialised, and the prover carries on from that transcript.
    draw(name, index, value) -> value overrides a TranscriptRng draw (ib, ob, sb, sL, sR, tb1, tb3 .. tb6).
    phase2 = (A_I2, A_O2, S2) encodings are sent in place of the identity.  framing: "v0", "v1" or "legacy"."""
    enc = enc or (lambda label, i, e: e)
    draw = draw or (lambda name, i, v: v)
    assert framing in ("v0", "v1", "legacy")
    t = cs.t
    m = len(cs.v)
    honest_V = ol.pedersen_commit(_sc(cs.v), _sc(cs.v_blinding)) if m else b""
    V = []
    for i in range(m):
        e = enc("V", i, honest_V[32 * i:32 * i + 32])
        t.append_point(b"V", e)
        V.append(e)
    t.append_u64(b"m", m)
    rng = t.build_rng([pr.sc_bytes(x) for x in cs.v_blinding], ext)
    n = n1 = len(cs.aL)
    N = pr.next_pow2(n)
    if cap < N:
        raise ValueError("InvalidGeneratorsLength")
    Genc, Henc = ol.gens(0, N)
    G = [Genc[32 * i:32 * i + 32] for i in range(N)]
    H = [Henc[32 * i:32 * i + 32] for i in range(N)]
    B, Bb = ol.pedersen_gens()
    ib, ob, sb = (draw(name, 0, rng.scalar()) for name in ("ib", "ob", "sb"))
    sL = [draw("sL", i, rng.scalar()) for i in range(n)]
    sR = [draw("sR", i, rng.scalar()) for i in range(n)]
    A_I = enc("A_I1", 0, _msm([ib] + cs.aL + cs.aR, [Bb] + G[:n] + H[:n]))
    A_O = enc("A_O1", 0, _msm([ob] + cs.aO, [Bb] + G[:n]))
    S = enc("S1", 0, _msm([sb] + sL + sR, [Bb] + G[:n] + H[:n]))
    t.append_point(b"A_I1", A_I)
    t.append_point(b"A_O1", A_O)
    t.append_point(b"S1", S)
    t.append_message(b"dom-sep", b"r1cs-1phase")
    A2 = [enc(lab, 0, p) for lab, p in zip(("A_I2", "A_O2", "S2"), phase2 or (IDENTITY,) * 3)]
    if framing == "v0":
        assert A2 == [IDENTITY] * 3, "version-0 framing carries no phase-2 points"
    for lab, p in zip((b"A_I2", b"A_O2", b"S2"), A2):
        t.append_point(lab, p)
    y = t.challenge_scalar(b"y")
    z = t.challenge_scalar(b"z")
    wL, wR, wO, wV, _ = cs.flatten(z, n, m)
    yinv = pr.sc_inv(y)
    ypow = [pow(y, i, L) for i in range(N)]
    yipow = [pow(yinv, i, L) for i in range(N)]
    l1 = [(cs.aL[i] + yipow[i] * wR[i]) % L for i in range(n)]
    l2 = list(cs.aO)
    l3 = list(sL)
    r0 = [(wO[i] - ypow[i]) % L for i in range(n)]
    r1 = [(ypow[i] * cs.aR[i] + wL[i]) % L for i in range(n)]
    r3 = [ypow[i] * sR[i] % L for i in range(n)]
    ip = pr._ip
    t1 = ip(l1, r0)
    t2 = (ip(l1, r1) + ip(l2, r0)) % L
    t3 = (ip(l2, r1) + ip(l3, r0)) % L
    t4 = (ip(l1, r3) + ip(l3, r1)) % L
    t5 = ip(l2, r3)
    t6 = ip(l3, r3)
    tb1, tb3, tb4, tb5, tb6 = (draw(name, 0, rng.scalar()) for name in ("tb1", "tb3", "tb4", "tb5", "tb6"))
    Tc = ol.pedersen_commit(_sc([t1, t3, t4, t5, t6]), _sc([tb1, tb3, tb4, tb5, tb6]))
    Ts = []
    for k, lab in enumerate(("T_1", "T_3", "T_4", "T_5", "T_6")):
        Ts.append(enc(lab, 0, Tc[32 * k:32 * k + 32]))
        t.append_point(lab.encode(), Ts[-1])
    u = t.challenge_scalar(b"u")
    x = t.challenge_scalar(b"x")
    tb2 = ip(wV, cs.v_blinding)
    tx = txb = 0
    for k, (tc, tbc) in enumerate(((t1, tb1), (t2, tb2), (t3, tb3), (t4, tb4), (t5, tb5), (t6, tb6)), 1):
        tx = (tx + tc * pow(x, k, L)) % L
        txb = (txb + tbc * pow(x, k, L)) % L
    x2, x3 = x * x % L, x * x % L * x % L
    a = [(x * l1[i] + x2 * l2[i] + x3 * l3[i]) % L for i in range(n)] + [0] * (N - n)
    b = [(r0[i] + x * r1[i] + x3 * r3[i]) % L for i in range(n)] + [(-ypow[i]) % L for i in range(n, N)]
    eb = x * (ib + x * (ob + x * sb)) % L
    t.append_scalar(b"t_x", tx)
    t.append_scalar(b"t_x_blinding", txb)
    t.append_scalar(b"e_blinding", eb)
    w = t.challenge_scalar(b"w")
    Q = ol.point_mul(pr.sc_bytes(w), B)
    # InnerProductProof::create; the first round carries the factors u^-1 (G beyond n) and y^-i (H) of pyref.ipp_create
    Gf = [1] * n1 + [u] * (N - n1)
    Hf = [yipow[i] * Gf[i] % L for i in range(N)]
    t.append_message(b"dom-sep", b"ipp v1")
    t.append_u64(b"n", N)
    Ls, Rs = [], []
    k = N
    while k != 1:
        k //= 2
        aL, aR, bL, bR = a[:k], a[k:], b[:k], b[k:]
        GL, GR, HL, HR = G[:k], G[k:], H[:k], H[k:]
        gL, gR, hL, hR = Gf[:k], Gf[k:], Hf[:k], Hf[k:]
        cL, cR = ip(aL, bR), ip(aR, bL)
        Lp = _msm([p * f for p, f in zip(aL, gR)] + [q * f for q, f in zip(bR, hL)] + [cL], GR + HL + [Q])
        Rp = _msm([p * f for p, f in zip(aR, gL)] + [q * f for q, f in zip(bL, hR)] + [cR], GL + HR + [Q])
        Ls.append(enc("L", len(Ls), Lp))
        Rs.append(enc("R", len(Rs), Rp))
        t.append_point(b"L", Ls[-1])
        t.append_point(b"R", Rs[-1])
        uj = t.challenge_scalar(b"u")
        ui = pr.sc_inv(uj)
        a = [(p * uj + ui * q) % L for p, q in zip(aL, aR)]
        b = [(p * ui + uj * q) % L for p, q in zip(bL, bR)]
        G = [_msm([ui * gL[i], uj * gR[i]], [GL[i], GR[i]]) for i in range(k)]
        H = [_msm([uj * hL[i], ui * hR[i]], [HL[i], HR[i]]) for i in range(k)]
        Gf, Hf = [1] * k, [1] * k
    out = bytearray()
    if framing == "legacy":
        out += A_I + A_O + S + b"".join(A2)
    elif framing == "v1":
        out += b"\x01" + A_I + A_O + S + b"".join(A2)
    else:
        out += b"\x00" + A_I + A_O + S
    out += b"".join(Ts) + _sc([tx, txb, eb])
    for Le, Re in zip(Ls, Rs):
        out += Le + Re
    out += _sc([a[0], b[0]])
    return bytes(out), b"".join(V)


# ----------------------------------------------------------------------------- statements
class Statement:
    """an R1CS statement (label, n multipliers, m commitments, CSR constraints) with the witness of a prover for it"""

    def __init__(self, label, rows, aL, aR, vals, blinds):
        self.label, self.rows = label, list(rows)
        self.aL, self.aR = [x % L for x in aL], [x % L for x in aR]
        self.vals, self.blinds = list(vals), list(blinds)
        self.n, self.m = len(self.aL), len(self.vals)
        self.csr = circuits.to_csr(self.rows)

    def add_commitment(self, v, r, row=None):
        """one more commitment, referenced by the constraint `row` if one is given"""
        self.vals.append(v)
        self.blinds.append(r)
        self.m += 1
        if row:
            self.rows.append(row)
            self.csr = circuits.to_csr(self.rows)

    def prover_cs(self):
        cs = pr.ConstraintSystem(pr.Transcript(self.label), True)
        for v, b in zip(self.vals, self.blinds):
            circuits._lazy_commit(cs, v, b)
        cs.aL, cs.aR = list(self.aL), list(self.aR)
        cs.aO = [p * q % L for p, q in zip(self.aL, self.aR)]
        cs.num_vars = self.n
        cs.constraints = list(self.rows)
        return cs

    def verifier_cs(self, V):
        cs = pr.ConstraintSystem(pr.Transcript(self.label), False)
        for i in range(len(V) // 32):
            cs.commit_verifier(V[32 * i:32 * i + 32])
        cs.num_vars = self.n
        cs.constraints = list(self.rows)
        return cs

    def cap(self):
        return max(8, pr.next_pow2(self.n))

    def prove(self, **hooks):
        return forge_prove(self.prover_cs(), self.cap(), EXT, **hooks)


_KINDS = {k: name for name, k in circuits.KIND.items()}


def from_instance(inst):
    """the Statement of a tests/circuits.py-style instance dict (label, CSR, witness and openings as 32-byte strings)"""
    dec = lambda b: [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]
    rp, tv, tc = inst["csr"]
    coeff = dec(tc)
    rows = [[((_KINDS[tv[t] >> 29], tv[t] & 0x1FFFFFFF), coeff[t]) for t in range(rp[r], rp[r + 1])] for r in range(len(rp) - 1)]
    return Statement(inst["label"], rows, dec(inst["aL"]), dec(inst["aR"]), dec(inst["vals"]), dec(inst["blinds"]))


def chain(n, seed, extra=None):
    """circuits.chain_instance(n, seed), and with extra = "unused" one more commitment no constraint references, with
    extra = "zero" one more commitment to (v, r) = (0, 0) constrained to V_3 = 0"""
    st = from_instance(circuits.chain_instance(n, seed))
    if extra == "unused":
        rnd = random.Random(seed + 77)
        st.add_commitment(rnd.randrange(L), rnd.randrange(L))
    elif extra == "zero":
        st.add_commitment(0, 0, [(("V", 3), 1)])
    return st


def zero_witness(n):
    """n multipliers whose inputs are all 0 (L_i = 0, R_i = 0), no commitment"""
    rows = [r for i in range(n) for r in ([(("L", i), 1)], [(("R", i), 1)])]
    return Statement(b"zero witness", rows, [0] * n, [0] * n, [], [])


# ----------------------------------------------------------------------------- verifiers
def ol_verify(st, V, proof, flags=0):
    rp, tv, tc = st.csr
    return ol.r1cs_verify(st.label, st.cap(), st.n, V, rp, tv, tc, proof, bytes(32), flags)


def pr_verify(st, V, proof, flags=0):
    return pr.r1cs_verify(st.verifier_cs(V), proof, st.cap(), bytes(32), legacy_framing=bool(flags & FLAG_LEGACY))


def _edit_scalars(buf, legacy, f):
    """applies f to the five scalars (t_x, t_x_blinding, e_blinding, a, b) of a serialised proof"""
    head = 0 if legacy else 1
    npts = 6 if legacy or buf[:1] == b"\x01" else 3
    if len(buf) < head + 32 * (npts + 10):
        return buf
    out = bytearray(buf)
    t0 = head + 32 * (npts + 5)
    for off in (t0, t0 + 32, t0 + 64, len(buf) - 64, len(buf) - 32):
        out[off:off + 32] = f(int.from_bytes(buf[off:off + 32], "little")).to_bytes(32, "little")
    return bytes(out)


_BAD = object()  # an encoding that failed to decode, kept for the lax MSM to look at


@contextlib.contextmanager
def lax(kind):
    """pyref.r1cs_verify with one check relaxed, as a kernel or host check could relax it:
    reduce_scalars  R1CSProof::from_bytes reduces the five proof scalars mod l instead of rejecting them when >= l
    mask_scalars    ... clears bit 255 of them instead
    mask_decode     ristretto decode clears bit 255 of the encoding first (fe_frombytes without the canonical check)
    reduce_decode   ristretto decode reduces s mod p before its checks
    no_identity     validate_and_append_point appends the identity instead of rejecting it
    drop_phase2     the verification MSM leaves out A_I2, A_O2, S2
    skip_zero       the verification MSM drops terms whose scalar is 0 before their points are decoded"""
    saved = pr.proof_from_bytes, pr.ristretto_decode, pr.msm, pr.Transcript.validate_and_append_point
    pfb, dec, msm = saved[:3]
    if kind in ("reduce_scalars", "mask_scalars"):
        f = (lambda x: x % L) if kind == "reduce_scalars" else (lambda x: x & ((1 << 255) - 1))
        pr.proof_from_bytes = lambda buf, legacy_framing=False: pfb(_edit_scalars(buf, legacy_framing, f), legacy_framing)
    elif kind == "mask_decode":
        pr.ristretto_decode = lambda e: dec(e[:31] + bytes([e[31] & 0x7F]))
    elif kind == "reduce_decode":
        pr.ristretto_decode = lambda e: dec((int.from_bytes(e, "little") % P).to_bytes(32, "little"))
    elif kind == "no_identity":
        pr.Transcript.validate_and_append_point = pr.Transcript.append_point
    elif kind == "drop_phase2":  # r1cs_verify calls msm once: scalars 3..5 weight A_I2, A_O2, S2
        pr.msm = lambda s, p: msm(s[:3] + [0, 0, 0] + s[6:], p)
    elif kind == "skip_zero":
        pr.ristretto_decode = lambda e: _BAD if dec(e) is None else dec(e)
        pr.msm = lambda s, p: pr.BASEPOINT if any(q is _BAD and x % L for x, q in zip(s, p)) else \
            msm([x for x, q in zip(s, p) if q is not _BAD], [q for q in p if q is not _BAD])
    else:
        raise ValueError(kind)
    try:
        yield
    finally:
        pr.proof_from_bytes, pr.ristretto_decode, pr.msm, pr.Transcript.validate_and_append_point = saved


def verification_point(st, V, proof, flags=0):
    """the point pyref.r1cs_verify compares with the identity (None if it rejects before its MSM)"""
    got, msm = [], pr.msm
    pr.msm = lambda s, p: got.append(msm(s, p)) or got[-1]
    try:
        pr_verify(st, V, proof, flags)
    finally:
        pr.msm = msm
    return got[-1] if got else None


# ----------------------------------------------------------------------------- the corpus
class Forgery:
    """a forged proof of a statement and its honest twin (the same hooks without the forging change)"""

    def __init__(self, name, st, proof, V, twin, lax_kind, flags=0):
        self.name, self.st, self.proof, self.V, self.twin, self.lax, self.flags = name, st, proof, V, twin, lax_kind, flags

    def __repr__(self):
        return self.name


def _framing_flags(framing):
    return FLAG_LEGACY if framing == "legacy" else 0


def on(label, index, f):
    return lambda lab, i, e: f(e) if (lab, i) == (label, index) else e


def zero_draws(*names):
    return lambda name, i, v: 0 if name in names else v


def scalar_offsets(proof, flags=0):
    """byte offsets of t_x, t_x_blinding, e_blinding, a, b in a serialised proof"""
    head = 0 if flags & FLAG_LEGACY else 1
    npts = 6 if flags & FLAG_LEGACY or proof[0] == 1 else 3
    t0 = head + 32 * (npts + 5)
    return dict(t_x=t0, t_x_blinding=t0 + 32, e_blinding=t0 + 64, a=len(proof) - 64, b=len(proof) - 32)


def scalar_variants(x):
    """(name, forged value, lax verifier that accepts it) of a canonical scalar x"""
    k = ((1 << 256) - 1 - x) // L
    return [("+l", x + L, "reduce_scalars"), ("+%dl" % k, x + k * L, "reduce_scalars"), ("+2^255", x + (1 << 255), "mask_scalars")]


def scalar_forgeries(proof, flags=0):
    """-> [(name, forged proof bytes, lax kind)]: each proof scalar in turn as x + l, x + k l (largest k below 2^256), x + 2^255"""
    out = []
    for field, off in scalar_offsets(proof, flags).items():
        x = int.from_bytes(proof[off:off + 32], "little")
        for vname, val, kind in scalar_variants(x):
            out.append(("%s%s" % (field, vname), proof[:off] + val.to_bytes(32, "little") + proof[off + 32:], kind))
    return out


FIVE_B = bytes.fromhex(RISTRETTO_MULTIPLES[5])  # a valid point that is not the identity


@functools.lru_cache(maxsize=None)
def corpus():
    """every forgery class of the verifier tests, at n in SIZES (lg N = 0, 0, 2, 3), seeded and deterministic"""
    out = []
    honest = {}

    def twin_of(st, key, **hooks):
        if key not in honest:
            honest[key] = st.prove(**hooks)
        return honest[key]

    def add(name, st, key, lax_kind, framing="v0", **hooks):
        base = {k: v for k, v in hooks.items() if k.startswith("twin_")}
        forged = {k: v for k, v in hooks.items() if not k.startswith("twin_")}
        tw = {k[5:]: v for k, v in base.items()}
        twin = twin_of(st, key, framing=framing, **tw)
        proof, V = st.prove(framing=framing, **{**tw, **forged})
        out.append(Forgery(name, st, proof, V, twin, lax_kind, _framing_flags(framing)))

    chains = {n: chain(n, 40 + n) for n in SIZES}
    # scalars >= l or with bit 255 set: byte edits of honest proofs
    for j, n in enumerate(SIZES):
        st = chains[n]
        proof, V = twin_of(st, ("chain", n, "v0"), framing="v0")
        for name, forged, kind in scalar_forgeries(proof)[j::len(SIZES)]:
            out.append(Forgery("n%d %s" % (n, name), st, forged, V, (proof, V), kind))
    # bit 255 set on each own point in turn
    for j, (lab, idx) in enumerate([("V", 0), ("V", 2), ("A_I1", 0), ("A_O1", 0), ("S1", 0), ("T_1", 0), ("T_3", 0), ("T_4", 0),
                                    ("T_5", 0), ("T_6", 0)]):
        n = SIZES[j % len(SIZES)]
        add("n%d high bit %s_%d" % (n, lab, idx), chains[n], ("chain", n, "v0"), "mask_decode", enc=on(lab, idx, high_bit))
    for n in (3, 8):
        lg = pr.next_pow2(n).bit_length() - 1
        for lab in ("L", "R"):
            for idx in sorted({0, lg - 1}):
                add("n%d high bit %s_%d" % (n, lab, idx), chains[n], ("chain", n, "v0"), "mask_decode", enc=on(lab, idx, high_bit))
    for j, framing in enumerate(("v1", "legacy")):
        for lab in ("A_I2", "A_O2", "S2"):
            n = SIZES[(j + len(lab)) % len(SIZES)]
            add("n%d %s high bit %s" % (n, framing, lab), chains[n], ("chain", n, framing), "mask_decode", framing=framing,
                enc=on(lab, 0, lambda e: HIGH_IDENTITY))
    # the identity encoded as s = p
    add("n1 v1 A_I2 = p", chains[1], ("chain", 1, "v1"), "reduce_decode", framing="v1", enc=on("A_I2", 0, lambda e: P_ENC))
    zc = chain(3, 60, extra="zero")
    add("n3 V_3 = (0, 0) encoded as p", zc, ("zero V", 3), "reduce_decode", enc=on("V", 3, lambda e: P_ENC))
    # one own point equal to the identity, everything else honest
    for n in (3, 8):
        st = chains[n]
        add("n%d S1 = identity" % n, st, ("sLR", n), "no_identity", draw=zero_draws("sb", "sL", "sR"), twin_draw=zero_draws("sL", "sR"))
        add("n%d T_4 = identity" % n, st, ("sLR", n), "no_identity", draw=zero_draws("sL", "sR", "tb4"), twin_draw=zero_draws("sL", "sR"))
        add("n%d T_5 = identity" % n, st, ("sR", n), "no_identity", draw=zero_draws("sR", "tb5"), twin_draw=zero_draws("sR"))
        add("n%d T_6 = identity" % n, st, ("sR", n), "no_identity", draw=zero_draws("sR", "tb6"), twin_draw=zero_draws("sR"))
    for n in (0, 3):
        st = zero_witness(n)
        add("zero witness n%d A_I1 = identity" % n, st, ("zero", n), "no_identity", draw=zero_draws("ib"))
        add("zero witness n%d A_O1 = identity" % n, st, ("zero", n), "no_identity", draw=zero_draws("ob"))
    # a valid phase-2 point that is not the identity
    for j, framing in enumerate(("v1", "legacy")):
        for k, lab in enumerate(("A_I2", "A_O2", "S2")):
            n = SIZES[(j + k) % len(SIZES)]
            p2 = [IDENTITY] * 3
            p2[k] = FIVE_B
            add("n%d %s %s = 5 B" % (n, framing, lab), chains[n], ("chain", n, framing), "drop_phase2", framing=framing, phase2=tuple(p2))
    # a commitment no constraint references (scalar 0), encoded as each RFC 9496 bad encoding
    for j, h in enumerate(BAD_ENCODINGS):
        n = SIZES[j % len(SIZES)]
        st = chain(n, 80 + n, extra="unused")
        add("n%d unused V_3 = bad encoding %d" % (n, j), st, ("unused", n), "skip_zero", enc=on("V", 3, lambda e, h=h: bytes.fromhex(h)))
    return out


def cancelling_pair(proof, delta=1):
    """two copies of a proof with a + delta and a - delta (both canonical): their errors cancel under equal weights"""
    off = len(proof) - 64
    a = int.from_bytes(proof[off:off + 32], "little")
    assert delta <= a < L - delta
    return tuple(proof[:off] + pr.sc_bytes(a + s * delta) + proof[off + 32:] for s in (1, -1))
