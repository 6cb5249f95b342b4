"""Host-side mirror of the reference's operator interface for the hot path, over libbpg's C ABI.

Names follow the bulletproofs fork as the reference calls it (SURVEY.md section 8b):
  PedersenGens.default().commit(v, r)            gadget.rs:31  commitments.rs:27,39  cs_buffer.rs:39
  BulletproofGens.new(capacity, 1)                prover.rs:92  verifier.rs:89
  Prover.new / commit / multiply / allocate_multiplier / allocate / constrain / prove      prover.rs:54,93
  Verifier.new / commit / ... / verify                                                      verifier.rs:53,90
  mimc_hash(bytes)                                src/mimc_hash/mimc.rs:61
Scalars are Python ints or 32-byte LE bytes; points are 32-byte compressed ristretto255.
"""
import array
import ctypes as C
import json
import os

from . import _lib
from ._lib import BpgError

L_ORDER = 2 ** 252 + 27742317777372353535851937790883648493


class R1CSError(Exception):
    """bulletproofs::r1cs::R1CSError (VerificationError, FormatError, InvalidGeneratorsLength, ...)."""


def _sb(x):
    if isinstance(x, (bytes, bytearray)):
        assert len(x) == 32
        return bytes(x)
    return int(x % L_ORDER).to_bytes(32, "little")


def _u32_array(xs):
    """ctypes uint32 array holding xs (at least one element, so that an empty list still gives a valid pointer)"""
    a = array.array("I", xs or [0])
    return (C.c_uint32 * len(a)).from_buffer(a)


class Context:
    """One CUDA device + stream + resident generator tables (bpg_ctx)."""
    _default = None

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.bpg_ctx_create(device, C.byref(h))
        if rc != 0:
            raise BpgError(rc, (self.lib.bpg_last_error(None) or b"").decode() or self.lib.bpg_strerror(rc).decode())
        self.h = h
        self.device = device
        self._mimc_ready = False

    @classmethod
    def default(cls):
        if cls._default is None:
            cls._default = cls(int(os.environ.get("LOCAL_RANK", "0")))
        return cls._default

    def check(self, rc):
        if rc < 0:
            raise BpgError(rc, (self.lib.bpg_last_error(self.h) or b"").decode() if rc == _lib.E_CUDA else self.lib.bpg_strerror(rc).decode())
        return rc

    def close(self):
        if self.h:
            self.lib.bpg_ctx_destroy(self.h)
            self.h = None

    # ---- generators
    def gens_ensure(self, capacity):
        self.check(self.lib.bpg_gens_ensure(self.h, capacity))

    def gens_capacity(self):
        return self.lib.bpg_gens_capacity(self.h)

    def gens_export(self, i0, n):
        g, h = C.create_string_buffer(32 * n), C.create_string_buffer(32 * n)
        self.check(self.lib.bpg_gens_export(self.h, i0, n, g, h))
        return g.raw, h.raw

    def pedersen_gens(self):
        a, b = C.create_string_buffer(32), C.create_string_buffer(32)
        self.check(self.lib.bpg_pedersen_gens(self.h, a, b))
        return a.raw, b.raw

    # ---- group operations
    def pedersen_commit(self, v, r):
        n = len(v) // 32
        out = C.create_string_buffer(32 * max(n, 1))
        self.check(self.lib.bpg_pedersen_commit(self.h, v, r, n, out))
        return out.raw[:32 * n]

    def msm(self, scalars, points, n=None):
        """variable-base MSM; scalars / points: bytes, or host pointers (e.g. from host_alloc) with n given"""
        out = C.create_string_buffer(32)
        self.check(self.lib.bpg_msm(self.h, scalars, points, len(scalars) // 32 if n is None else n, out))
        return out.raw

    def msm_gens(self, sG, sH, n, offset=0, extra_scalars=b"", extra_points=b""):
        out = C.create_string_buffer(32)
        k = len(extra_scalars) // 32
        self.check(self.lib.bpg_msm_gens(self.h, sG, sH, n, offset, extra_scalars or None, extra_points or None, k, out))
        return out.raw

    def msm_gens_dev(self, d_sG, d_sH, n, offset=0):
        out = C.create_string_buffer(32)
        self.check(self.lib.bpg_msm_gens_dev(self.h, d_sG, d_sH, n, offset, out))
        return out.raw

    def msm_gens_partial_dev(self, d_sG, d_sH, n, offset=0):
        out = C.create_string_buffer(128)
        self.check(self.lib.bpg_msm_gens_partial_dev(self.h, d_sG, d_sH, n, offset, out))
        return out.raw

    def msm_gens_partial_to_dev(self, d_sG, d_sH, n, offset, d_out128):
        self.check(self.lib.bpg_msm_gens_partial_to_dev(self.h, d_sG, d_sH, n, offset, d_out128))

    def points_sum_compress_dev(self, d_ext128, n):
        out = C.create_string_buffer(32)
        self.check(self.lib.bpg_points_sum_compress_dev(self.h, d_ext128, n, out))
        return out.raw

    def points_sum_compress(self, ext128):
        out = C.create_string_buffer(32)
        self.check(self.lib.bpg_points_sum_compress(self.h, ext128, len(ext128) // 128, out))
        return out.raw

    def fold_points(self, sl, sr, PL, PR):
        n = len(PL) // 32
        out = C.create_string_buffer(32 * max(n, 1))
        self.check(self.lib.bpg_fold_points(self.h, _sb(sl), _sb(sr), PL, PR, n, out))
        return out.raw[:32 * n]

    # ---- MiMC
    def _mimc_init(self):
        if not self._mimc_ready:
            p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "mimc_consts.json")
            with open(p) as f:
                consts = b"".join(bytes.fromhex(h) for h in json.load(f))
            self.check(self.lib.bpg_mimc_set_constants(self.h, consts))
            self._mimc_ready = True

    def mimc_hash_batch(self, preimages):
        self._mimc_init()
        n = len(preimages)
        offs = [0]
        for p in preimages:
            offs.append(offs[-1] + len(p))
        out = C.create_string_buffer(32 * max(n, 1))
        self.check(self.lib.bpg_mimc_hash_batch(self.h, b"".join(preimages), (C.c_uint64 * (n + 1))(*offs), n, out))
        raw = out.raw  # (.raw copies the whole buffer: take it once)
        return [raw[32 * i:32 * i + 32] for i in range(n)]

    def mimc_sponge_batch(self, block_lists, trace=False):
        """block_lists: list of lists of 32-byte LE blocks -> (digests, trace bytes or None)."""
        self._mimc_init()
        n = len(block_lists)
        offs = [0]
        for b in block_lists:
            offs.append(offs[-1] + len(b))
        flat = b"".join(b"".join(bl) for bl in block_lists)
        out = C.create_string_buffer(32 * max(n, 1))
        tr = C.create_string_buffer(offs[-1] * 972 * 96) if trace else None
        self.check(self.lib.bpg_mimc_sponge_batch(self.h, flat, (C.c_uint32 * (n + 1))(*offs), n, out, tr))
        raw = out.raw  # (.raw copies the whole buffer: take it once)
        return [raw[32 * i:32 * i + 32] for i in range(n)], (tr.raw if trace else None)

    # ---- batched set-up
    def circuit_create_batch(self, csrs):
        """csrs: list of (n, m, row_ptr, term_var, term_coeff bytes) -> list of circuit handles (c_void_p), handle i behaving as
        the one bpg_circuit_create makes for csrs[i].  All handles share one device allocation; release each with
        bpg_circuit_destroy, in any order."""
        k = len(csrs)
        if k == 0:
            return []
        rps, tvs = [_u32_array(c[2]) for c in csrs], [_u32_array(c[3]) for c in csrs]
        u32pp = lambda xs: (C.POINTER(C.c_uint32) * k)(*[C.cast(x, C.POINTER(C.c_uint32)) for x in xs])
        sizes = lambda j: (C.c_size_t * k)(*[c[j] for c in csrs])
        out = (C.c_void_p * k)()
        self.check(self.lib.bpg_circuit_create_batch(self.h, k, sizes(0), sizes(1), (C.c_size_t * k)(*[len(c[2]) - 1 for c in csrs]), u32pp(rps), u32pp(tvs),
                                                     (C.c_char_p * k)(*[bytes(c[4]) for c in csrs]), out))
        return [C.c_void_p(h) for h in out]

    def witness_eval_batch(self, items):
        """items: list of (n, m, lc_ptr, term_var, term_coeff bytes, v bytes, a_L inputs, a_R inputs (n x 32 bytes or shorter,
        zero-padded)) -> list of (a_L, a_R, a_O) bytes, entry i being what bpg_witness_eval computes for items[i]"""
        k = len(items)
        if k == 0:
            return []
        bufs = [[C.create_string_buffer(bytes(it[6]), 32 * max(1, it[0])), C.create_string_buffer(bytes(it[7]), 32 * max(1, it[0])),
                 C.create_string_buffer(32 * max(1, it[0]))] for it in items]
        ptrs, tvs = [_u32_array(it[2]) for it in items], [_u32_array(it[3]) for it in items]
        u32pp = lambda xs: (C.POINTER(C.c_uint32) * k)(*[C.cast(x, C.POINTER(C.c_uint32)) for x in xs])
        sizes = lambda j: (C.c_size_t * k)(*[it[j] for it in items])
        bytes_pp = lambda j: (C.c_char_p * k)(*[bytes(it[j]) for it in items])
        out_pp = lambda j: (C.c_void_p * k)(*[C.addressof(b[j]) for b in bufs])
        self.check(self.lib.bpg_witness_eval_batch(self.h, k, sizes(0), sizes(1), u32pp(ptrs), u32pp(tvs), bytes_pp(4), bytes_pp(5),
                                                   out_pp(0), out_pp(1), out_pp(2)))
        return [tuple(b[j].raw[:32 * it[0]] for j in range(3)) for b, it in zip(bufs, items)]

    # ---- batched proving
    def prove_batch(self, items, flags=0):
        """items: list of (circuit handle (c_void_p), label bytes, aL, aR, aO, v, v_blinding (n or m x 32 bytes each), ext_rng32)
        -> list of (proof bytes, V bytes), entry i being exactly what bpg_r1cs_prove returns for item i"""
        n = len(items)
        if n == 0:
            return []
        ms = [len(it[5] or b"") // 32 for it in items]
        cap = 1 + 32 * (14 + 64 + 2)
        ptr = lambda xs: (C.c_char_p * n)(*xs)
        proofs = [C.create_string_buffer(cap) for _ in range(n)]
        Vs = [C.create_string_buffer(32 * max(1, m)) for m in ms]
        lens = (C.c_size_t * n)()
        self.check(self.lib.bpg_r1cs_prove_batch(
            self.h, n, (C.c_void_p * n)(*[it[0] for it in items]), ptr([it[1] for it in items]), (C.c_size_t * n)(*[len(it[1]) for it in items]),
            ptr([it[2] for it in items]), ptr([it[3] for it in items]), ptr([it[4] for it in items]), ptr([it[5] for it in items]),
            ptr([it[6] for it in items]), b"".join(it[7] for it in items), flags, (C.c_void_p * n)(*[C.addressof(b) for b in Vs]),
            (C.c_void_p * n)(*[C.addressof(b) for b in proofs]), (C.c_size_t * n)(*([cap] * n)), lens))
        return [(proofs[i].raw[:lens[i]], Vs[i].raw[:32 * ms[i]]) for i in range(n)]

    # ---- batch verification
    def verify_batch(self, items, flags=0):
        """items: list of (circuit handle (c_void_p), label bytes, V bytes, proof bytes, ext_rng32) -> list of bool,
        verdict i being exactly what bpg_r1cs_verify returns for item i (one combined check with random weights; if it fails,
        one check per proof)"""
        return self._verify_many(self.lib.bpg_r1cs_verify_batch, items, flags)

    def verify_each(self, items, flags=0):
        """items as for verify_batch -> list of bool, verdict i being exactly what bpg_r1cs_verify returns for item i: every
        proof is checked against its own verification equation (bpg_r1cs_verify_each), whatever the other proofs are"""
        return self._verify_many(self.lib.bpg_r1cs_verify_each, items, flags)

    def _verify_many(self, fn, items, flags):
        n = len(items)
        if n == 0:
            return []
        circs = (C.c_void_p * n)(*[it[0] for it in items])
        labels = (C.c_char_p * n)(*[it[1] for it in items])
        lens = (C.c_size_t * n)(*[len(it[1]) for it in items])
        Vs = (C.c_char_p * n)(*[it[2] if it[2] else b"\0" for it in items])
        proofs = (C.c_char_p * n)(*[it[3] if it[3] else b"\0" for it in items])
        plens = (C.c_size_t * n)(*[len(it[3]) for it in items])
        ext = b"".join(it[4] for it in items)
        acc = (C.c_int * n)()
        self.check(fn(self.h, n, circs, labels, lens, Vs, proofs, plens, ext, flags, acc))
        return [bool(a) for a in acc]

    # ---- misc
    def launch_count(self):
        return self.lib.bpg_launch_count(self.h)

    def event_record(self, slot):
        self.check(self.lib.bpg_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = C.c_float()
        self.check(self.lib.bpg_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def prof_enable(self, on=True):
        self.check(self.lib.bpg_prof_enable(self.h, 1 if on else 0))

    def prof_read(self):
        n, ms, pairs = C.c_uint64(), C.c_double(), C.c_uint64()
        self.check(self.lib.bpg_prof_read(self.h, C.byref(n), C.byref(ms), C.byref(pairs)))
        return n.value, ms.value, pairs.value

    def prof_read_launches(self, cap=64):
        """[(ms, pairs)] of every timed k_msm_accumulate launch since prof_enable(True)"""
        ms, pairs = (C.c_float * cap)(), (C.c_uint32 * cap)()
        n = self.lib.bpg_prof_read_launches(self.h, ms, pairs, cap)
        if n < 0:
            self.check(n)
        return [(ms[i], pairs[i]) for i in range(n)]

    def sync(self):
        self.check(self.lib.bpg_sync(self.h))

    def bench_latency(self, iters=200):
        out = (C.c_double * 8)()
        self.check(self.lib.bpg_bench_latency(self.h, iters, out))
        names = ["fe_mul", "ge_add", "ge_add_ilp", "ge_dbl", "ge_dbl_ilp", "ge_madd", "ge_madd_ilp", "fe_mul4"]
        return dict(zip(names, [round(x, 1) for x in out]))

    def bench_imad(self, iters):
        ms, mac = C.c_float(), C.c_double()
        self.check(self.lib.bpg_bench_imad(self.h, iters, C.byref(ms), C.byref(mac)))
        return ms.value, mac.value

    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.bpg_dev_alloc(self.h, nbytes, C.byref(p)))
        return p

    def host_alloc(self, data):
        """page-locked host copy of `data` (bpg_host_alloc); returns (pointer usable wherever a host buffer is expected, handle
        for host_free)"""
        p = C.c_void_p()
        self.check(self.lib.bpg_host_alloc(self.h, len(data), C.byref(p)))
        C.memmove(p, data, len(data))
        return C.cast(p, C.c_char_p), p

    def host_free(self, p):
        self.check(self.lib.bpg_host_free(self.h, p))

    def dev_free(self, p):
        self.check(self.lib.bpg_dev_free(self.h, p))

    def dev_upload(self, d, data):
        self.check(self.lib.bpg_dev_upload(self.h, d, data, len(data)))

    def dev_download(self, d, nbytes):
        out = C.create_string_buffer(nbytes)
        self.check(self.lib.bpg_dev_download(self.h, out, d, nbytes))
        return out.raw


class Transcript:
    """merlin::Transcript (host)."""

    def __init__(self, label):
        self.lib = _lib.load()
        self.label = bytes(label)
        self.h = self.lib.bpg_transcript_new(self.label, len(self.label))

    def append_message(self, label, msg):
        self.lib.bpg_transcript_append(self.h, label, len(label), msg, len(msg))

    def challenge_bytes(self, label, n):
        out = C.create_string_buffer(n)
        self.lib.bpg_transcript_challenge(self.h, label, len(label), out, n)
        return out.raw

    def __del__(self):
        try:
            self.lib.bpg_transcript_free(self.h)
        except Exception:
            pass


class PedersenGens:
    def __init__(self, ctx=None):
        self.ctx = ctx or Context.default()
        if self.ctx.gens_capacity() == 0:
            self.ctx.gens_ensure(64)
        self.B, self.B_blinding = self.ctx.pedersen_gens()

    @classmethod
    def default(cls, ctx=None):
        return cls(ctx)

    def commit(self, value, blinding):
        return self.ctx.pedersen_commit(_sb(value), _sb(blinding))

    def commit_batch(self, values, blindings):
        out = self.ctx.pedersen_commit(b"".join(_sb(v) for v in values), b"".join(_sb(b) for b in blindings))
        return [out[32 * i:32 * i + 32] for i in range(len(values))]


class BulletproofGens:
    def __init__(self, gens_capacity, party_capacity=1, ctx=None):
        if party_capacity != 1:
            raise ValueError("the reference only ever uses party_capacity = 1 (prover.rs:92, verifier.rs:89)")
        self.ctx = ctx or Context.default()
        self.gens_capacity = gens_capacity
        self.ctx.gens_ensure(max(gens_capacity, 1))

    @classmethod
    def new(cls, gens_capacity, party_capacity=1, ctx=None):
        return cls(gens_capacity, party_capacity, ctx)

    def G(self, n, i0=0):
        g, _ = self.ctx.gens_export(i0, n)
        return [g[32 * i:32 * i + 32] for i in range(n)]

    def H(self, n, i0=0):
        _, h = self.ctx.gens_export(i0, n)
        return [h[32 * i:32 * i + 32] for i in range(n)]


# Variables / linear combinations: ("L"|"R"|"O"|"V", index) or ("1", 0); an LC is a list of (variable, coeff).
_KIND = {"L": 0, "R": 1, "O": 2, "V": 3, "1": 4}
ONE = ("1", 0)


class _ConstraintSystem:
    """Shared recorder of r1cs::Prover / r1cs::Verifier: the 5-method ConstraintSystem trait the reference's gadgets
    use (cs_buffer.rs:89-113): multiply, allocate, allocate_multiplier, constrain (+ the transcript label)."""

    def __init__(self, label, ctx, prover):
        self._ctx = ctx  # resolved lazily: recording constraints needs no device
        self.label = bytes(label)
        self.is_prover = prover
        self.row_ptr, self.term_var, self.term_coeff = [0], [], bytearray()
        # prover side: caller-assigned a_L, a_R (allocate / allocate_multiplier) and, for multiply(), the pair of linear
        # combinations per multiplier; the assignment itself is computed on the device at prove() (bpg_witness_eval)
        self._in_L, self._in_R = [], []
        self._w_ptr, self._w_var, self._w_coeff = [0], [], bytearray()
        self._witness = None
        self.v, self.v_blinding, self.V = [], [], []
        self.num_vars = 0
        self._pending = None

    @property
    def ctx(self):
        if self._ctx is None:
            self._ctx = Context.default()
        return self._ctx

    def csr(self):
        """(row_ptr, term_var, term_coeff bytes) of the recorded constraints"""
        return list(self.row_ptr), list(self.term_var), bytes(self.term_coeff)

    # -- the prover's assignment (Prover::eval of every multiply(), cs_buffer.rs:94-97 / prover.rs:102-117) is evaluated on
    # the device, level by level of the dependency graph, in ONE call when it is first needed
    def _push_witness_lc(self, lc):
        for (k, i), c in lc:
            self._w_var.append((_KIND[k] << 29) | i)
            self._w_coeff += int(c % L_ORDER).to_bytes(32, "little")
        self._w_ptr.append(len(self._w_var))

    def _witness_cached(self):
        return self._witness is not None and self._witness[0] == (self.num_vars, len(self.v))

    def _witness_args(self):
        """the arguments of bpg_witness_eval as one item of Context.witness_eval_batch"""
        enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
        return (self.num_vars, len(self.v), self._w_ptr, self._w_var, bytes(self._w_coeff), enc(self.v), enc(self._in_L), enc(self._in_R))

    def witness_bytes(self):
        """(a_L, a_R, a_O) as n x 32-byte LE strings, computed by bpg_witness_eval (cached until the system grows)"""
        n, m = self.num_vars, len(self.v)
        if self._witness_cached():
            return self._witness[1]
        enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
        aL, aR = C.create_string_buffer(enc(self._in_L), 32 * max(1, n)), C.create_string_buffer(enc(self._in_R), 32 * max(1, n))
        aO = C.create_string_buffer(32 * max(1, n))
        ptr = (C.c_uint32 * (2 * n + 1))(*self._w_ptr)
        tv = (C.c_uint32 * max(1, len(self._w_var)))(*self._w_var)
        self.ctx.check(self.ctx.lib.bpg_witness_eval(self.ctx.h, n, m, ptr, tv, bytes(self._w_coeff), enc(self.v), aL, aR, aO))
        self._witness = ((n, m), (aL.raw[:32 * n], aR.raw[:32 * n], aO.raw[:32 * n]))
        return self._witness[1]

    def witness(self):
        """(a_L, a_R, a_O) as lists of integers"""
        dec = lambda b: [int.from_bytes(b[32 * i:32 * i + 32], "little") for i in range(len(b) // 32)]
        return tuple(dec(b) for b in self.witness_bytes())

    def _push_row(self, lc):
        for (k, i), c in lc:
            self.term_var.append((_KIND[k] << 29) | i)
            self.term_coeff += int(c % L_ORDER).to_bytes(32, "little")
        self.row_ptr.append(len(self.term_var))

    def multiply(self, left, right):
        i = self.num_vars
        self.num_vars += 1
        if self.is_prover:
            self._in_L.append(0); self._in_R.append(0)
            self._push_witness_lc(left); self._push_witness_lc(right)
        self._push_row(list(left) + [(("L", i), L_ORDER - 1)])
        self._push_row(list(right) + [(("R", i), L_ORDER - 1)])
        return ("L", i), ("R", i), ("O", i)

    def allocate_multiplier(self, input_assignments=None):
        if self.is_prover and input_assignments is None:
            raise R1CSError("MissingAssignment")
        i = self.num_vars
        self.num_vars += 1
        if self.is_prover:
            l, r = input_assignments
            self._in_L.append(l % L_ORDER); self._in_R.append(r % L_ORDER)
            self._w_ptr += [len(self._w_var)] * 2
        return ("L", i), ("R", i), ("O", i)

    def allocate(self, assignment=None):
        if self.is_prover and assignment is None:
            raise R1CSError("MissingAssignment")
        if self._pending is None:
            i = self.num_vars
            self.num_vars += 1
            self._pending = i
            if self.is_prover:
                self._in_L.append(assignment % L_ORDER); self._in_R.append(0)
                self._w_ptr += [len(self._w_var)] * 2
            return ("L", i)
        i, self._pending = self._pending, None
        if self.is_prover:
            self._in_R[i] = assignment % L_ORDER
        return ("R", i)

    def constrain(self, lc):
        self._push_row(lc)

    def num_constraints(self):
        return len(self.row_ptr) - 1

    def get_num_multiplications(self):
        return self.num_vars

    get_num_vars = get_num_multiplications

    def _circuit_args(self, m):
        """the arguments of bpg_circuit_create as one entry of Context.circuit_create_batch"""
        return self.num_vars, m, self.row_ptr, self.term_var, bytes(self.term_coeff)

    def _circuit(self, m):
        lib, h = self.ctx.lib, C.c_void_p()
        q = len(self.row_ptr) - 1
        rp = (C.c_uint32 * (q + 1))(*self.row_ptr)
        tv = (C.c_uint32 * max(1, len(self.term_var)))(*self.term_var)
        self.ctx.check(lib.bpg_circuit_create(self.ctx.h, self.num_vars, m, q, rp, tv, bytes(self.term_coeff), C.byref(h)))
        return h


class Prover(_ConstraintSystem):
    def __init__(self, label, ctx=None):
        super().__init__(label, ctx, True)

    @classmethod
    def new(cls, label, ctx=None):
        return cls(label, ctx)

    def commit(self, v, v_blinding):
        """-> (CompressedRistretto, Variable).  The group operation is deferred to prove(), which commits all
        openings in one batched launch; call commitments() for the bytes before proving."""
        self.v.append(v % L_ORDER)
        self.v_blinding.append(v_blinding % L_ORDER)
        return None, ("V", len(self.v) - 1)

    def commitments(self):
        out = self.ctx.pedersen_commit(b"".join(_sb(x) for x in self.v), b"".join(_sb(x) for x in self.v_blinding))
        return [out[32 * i:32 * i + 32] for i in range(len(self.v))]

    def prove(self, bp_gens, ext_rng32=None, flags=0):
        """Prover::prove(&bp_gens) -> (proof bytes, [V commitments]).  ext_rng32 stands for the 32 bytes the
        reference draws from thread_rng (os.urandom if omitted)."""
        n, m = self.num_vars, len(self.v)
        npad = 1
        while npad < n:
            npad *= 2
        if bp_gens.gens_capacity < npad:
            raise R1CSError("InvalidGeneratorsLength")
        ext = ext_rng32 if ext_rng32 is not None else os.urandom(32)
        circ = self._circuit(m)
        try:
            enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
            cap = 1 + 32 * (14 + 64 + 2)
            proof, V = C.create_string_buffer(cap), C.create_string_buffer(32 * max(1, m))
            aL, aR, aO = self.witness_bytes()
            rc = self.ctx.lib.bpg_r1cs_prove(self.ctx.h, circ, self.label, len(self.label), aL, aR, aO,
                                             enc(self.v), enc(self.v_blinding), ext, flags, V, proof, cap)
            if rc < 0:
                self.ctx.check(rc)
            return proof.raw[:rc], [V.raw[32 * i:32 * i + 32] for i in range(m)]
        finally:
            self.ctx.lib.bpg_circuit_destroy(circ)


def prove_batch(provers, bp_gens, ext_rngs=None, flags=0):
    """Prover::prove(&bp_gens) of many provers in ONE call (bpg_r1cs_prove_batch) -> list of (proof bytes, [V commitments]),
    entry i being what provers[i].prove(bp_gens, ext_rngs[i], flags) returns.  The provers share one context; ext_rngs
    (one 32-byte string per prover) default to os.urandom."""
    if not provers:
        return []
    ctx = provers[0].ctx
    if any(p.ctx is not ctx for p in provers):
        raise ValueError("prove_batch: every prover must use the same Context")
    for p in provers:
        npad = 1
        while npad < p.num_vars:
            npad *= 2
        if bp_gens.gens_capacity < npad:
            raise R1CSError("InvalidGeneratorsLength")
    exts = list(ext_rngs) if ext_rngs is not None else [os.urandom(32) for _ in provers]
    if len(exts) != len(provers):
        raise ValueError("prove_batch: %d ext_rngs for %d provers" % (len(exts), len(provers)))
    enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
    # set-up in two calls: every witness not yet cached (bpg_witness_eval_batch), every circuit (bpg_circuit_create_batch)
    stale = list({id(p): p for p in provers if not p._witness_cached()}.values())
    for p, w in zip(stale, ctx.witness_eval_batch([p._witness_args() for p in stale])):
        p._witness = ((p.num_vars, len(p.v)), w)
    circs = ctx.circuit_create_batch([p._circuit_args(len(p.v)) for p in provers])
    try:
        items = [(c, p.label, *p.witness_bytes(), enc(p.v), enc(p.v_blinding), ext) for c, p, ext in zip(circs, provers, exts)]
        out = ctx.prove_batch(items, flags)
    finally:
        for c in circs:
            ctx.lib.bpg_circuit_destroy(c)
    return [(proof, [V[32 * i:32 * i + 32] for i in range(len(p.v))]) for (proof, V), p in zip(out, provers)]


class Verifier(_ConstraintSystem):
    def __init__(self, label, ctx=None):
        super().__init__(label, ctx, False)

    @classmethod
    def new(cls, label, ctx=None):
        return cls(label, ctx)

    def commit(self, commitment):
        self.V.append(bytes(commitment))
        return ("V", len(self.V) - 1)

    def verify(self, proof, pc_gens=None, bp_gens=None, ext_rng32=None, flags=0):
        """Verifier::verify -> None on success, raises R1CSError('VerificationError') otherwise."""
        n = self.num_vars
        npad = 1
        while npad < n:
            npad *= 2
        if bp_gens is not None and bp_gens.gens_capacity < npad:
            raise R1CSError("InvalidGeneratorsLength")
        ext = ext_rng32 if ext_rng32 is not None else os.urandom(32)
        circ = self._circuit(len(self.V))
        try:
            acc = C.c_int(0)
            self.ctx.check(self.ctx.lib.bpg_r1cs_verify(self.ctx.h, circ, self.label, len(self.label), b"".join(self.V), proof, len(proof), ext,
                                                        flags, C.byref(acc)))
        finally:
            self.ctx.lib.bpg_circuit_destroy(circ)
        if not acc.value:
            raise R1CSError("VerificationError")


def verify_batch(verifiers, proofs, ext_rngs=None, flags=0):
    """Verifier::verify of many statements in ONE call (bpg_r1cs_verify_batch) -> list of bool, entry i being whether
    verifiers[i].verify(proofs[i], ext_rng32=ext_rngs[i], flags=flags) succeeds.  The verifiers share one context; their
    circuits are made by one bpg_circuit_create_batch.  ext_rngs (one 32-byte string per verifier) default to os.urandom."""
    return _verify_many("verify_batch", verifiers, proofs, ext_rngs, flags)


def verify_each(verifiers, proofs, ext_rngs=None, flags=0):
    """As verify_batch, through bpg_r1cs_verify_each: every proof is checked against its own verification equation, so entry i
    is exactly verifiers[i].verify(proofs[i], ext_rng32=ext_rngs[i], flags=flags)'s outcome whatever the other proofs are,
    at a cost that does not depend on how many of them are false."""
    return _verify_many("verify_each", verifiers, proofs, ext_rngs, flags)


def _verify_many(name, verifiers, proofs, ext_rngs, flags):
    if len(proofs) != len(verifiers):
        raise ValueError("%s: %d proofs for %d verifiers" % (name, len(proofs), len(verifiers)))
    if not verifiers:
        return []
    ctx = verifiers[0].ctx
    if any(v.ctx is not ctx for v in verifiers):
        raise ValueError("%s: every verifier must use the same Context" % name)
    exts = list(ext_rngs) if ext_rngs is not None else [os.urandom(32) for _ in verifiers]
    if len(exts) != len(verifiers):
        raise ValueError("%s: %d ext_rngs for %d verifiers" % (name, len(exts), len(verifiers)))
    circs = ctx.circuit_create_batch([v._circuit_args(len(v.V)) for v in verifiers])
    try:
        return getattr(ctx, name)([(c, v.label, b"".join(v.V), bytes(pf), ext) for c, v, pf, ext in zip(circs, verifiers, proofs, exts)], flags)
    finally:
        for c in circs:
            ctx.lib.bpg_circuit_destroy(c)


def mimc_hash(preimage, ctx=None):
    """mimc_hash(&Vec<u8>) -> Scalar bytes (32 B LE)   [src/mimc_hash/mimc.rs:61]"""
    return (ctx or Context.default()).mimc_hash_batch([bytes(preimage)])[0]


def mimc_hash_batch(preimages, ctx=None):
    return (ctx or Context.default()).mimc_hash_batch([bytes(p) for p in preimages])


def merkle_node_batch(pairs, ctx=None):
    """hash!(left, right) of merkle_tree_gadget.rs:7-12 for many (left, right) 32-byte LE pairs."""
    return (ctx or Context.default()).mimc_sponge_batch([[l, r] for l, r in pairs])[0]
