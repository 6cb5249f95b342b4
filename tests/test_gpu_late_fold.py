"""Late fold at every fold point (BPG_LATE_FOLD_LG: n' = 2^lg folded generators per vector, read once per process, so each
value runs in a subprocess of its own): on mid-size Merkle circuits of the benchmark's family (N = 2^15, 2^16, 2^17) and on a
bit-valued BoundsCheck witness (N = 2^15: the digits of many outputs fall into few buckets), every proof forced through the
late fold at n' = N/4 ... N/256 must equal, byte for byte, the proof without the late fold and the CPU oracle's."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EXT = b"\x5a" * 32
CAP = 1 << 17
# (name, lg N): Merkle trees of 16 / 32 / 64 leaves (29 160 / 60 264 / 122 472 multipliers), 256 BoundsChecks of 8 bytes
CIRCUITS = [("merkle16", 15), ("merkle32", 16), ("merkle64", 17), ("bounds256", 15)]
LGS = sorted({lgN - k for _, lgN in CIRCUITS for k in range(2, 9)})


def make_instance(name, ctx):
    from bulletproofs_gadgets_b200 import gadgets
    if name.startswith("merkle"):
        return gadgets.merkle_tree_instances(int(name[6:]), [100 + int(name[6:])], ctx=ctx)[0]
    return gadgets.bounds_check_batch_instance(256, 8, seed=9)


def prove_all(lg, flags):
    """proofs (hex) of every circuit whose fold point n' = 2^lg lies in N/4 ... N/256 (all circuits if lg is None)"""
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import gadgets
    ctx = bpg.Context(0)
    ctx.gens_ensure(CAP)
    out = {}
    for name, lgN in CIRCUITS:
        if lg is not None and not (lgN - 8 <= lg <= lgN - 2):
            continue
        inst = make_instance(name, ctx)
        circ = gadgets.Circuit(ctx, inst["n"], inst["m"], inst["csr"])
        proof, V = circ.prove(inst, EXT, flags)
        assert circ.verify(inst["label"], V, proof)
        circ.close()
        out[name] = (proof + V).hex()
    ctx.close()
    return out


@pytest.fixture(scope="module")
def reference():
    """GPU proofs without the late fold, checked against the CPU oracle"""
    import bulletproofs_gadgets_b200 as bpg
    import oracle_lib as ol
    ref = prove_all(None, bpg._lib.FLAG_NO_LATE_FOLD)
    ctx = bpg.Context(0)
    ol.lib().bpo_set_threads(os.cpu_count() or 1)
    try:
        for name, _ in CIRCUITS:
            inst = make_instance(name, ctx)
            rp, tv, tc = inst["csr"]
            want, Vw = ol.r1cs_prove(inst["label"], CAP, inst["aL"], inst["aR"], inst["aO"], inst["vals"], inst["blinds"], rp, tv, tc.tobytes(), EXT)
            assert ref[name] == (want + Vw).hex(), name
    finally:
        ol.lib().bpo_set_threads(1)
        ctx.close()
    return ref


@pytest.mark.parametrize("lg", LGS)
def test_forced_late_fold_at_every_fold_point_matches_oracle(reference, lg):
    env = dict(os.environ, BPG_LATE_FOLD_LG=str(lg))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(lg)], env=env, capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got, "no circuit has a fold point at n' = 2^%d" % lg
    for name, hexproof in got.items():
        assert hexproof == reference[name], "%s: fold point 2^%d changed the proof bytes" % (name, lg)


if __name__ == "__main__":
    for p in (ROOT, HERE):
        sys.path.insert(0, p)
    import bulletproofs_gadgets_b200 as _bpg
    print(json.dumps(prove_all(int(sys.argv[1]), _bpg._lib.FLAG_FORCE_LATE_FOLD)))
