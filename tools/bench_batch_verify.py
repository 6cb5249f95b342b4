#!/usr/bin/env python3
"""Batch verification on the BASELINE configs[4] mix: SET_MEMBER / LESS_THAN statements assembled as
bench.batch_verify_config5 does and proved on the GPU (bpg_r1cs_prove_batch), then verified by `--contexts` contexts in threads,
`--per-call` proofs per call, through each `--entry`: `batch` (bpg_r1cs_verify_batch: one combined check, then one per-proof
check if it fails) and `each` (bpg_r1cs_verify_each: every proof against its own equation).  Every entry and per-call size runs
on mixes of `--total` statements with each `--invalid` percentage of false statements (false statements are proved from
witnesses that do not satisfy them, as configs[4]'s 1 % are), spread evenly over the mix.  Reports verifications/s,
launches and host CPU per verification and whether every verdict equals the expected one, with a digest of the verdicts of
each mix (equal digests: equal verdicts, e.g. across library versions and entries).  Prints one JSON line (and writes it to
--out if given).

    python tools/bench_batch_verify.py [--total 8192] [--contexts 8] [--per-call 64,256] [--entry batch,each]
                                       [--invalid 0,1,10,50] [--repeat 3] [--cache path] [--out path]

--cache keeps the assembled statements (front-end output, no proofs) in a pickle, so alternating runs of two library
versions verify the same statements without assembling them again.  A library without bpg_r1cs_verify_each runs the `batch`
entry only."""
import argparse
import hashlib
import json
import multiprocessing as mp
import os
import pickle
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    """(card name, power limit) of device 0 as nvidia-smi reports them, ("unknown", "unknown") if it cannot say"""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "unknown", "unknown"
    fields = [x.strip() for x in q.stdout.strip().split(",")]
    if q.returncode != 0 or len(fields) != 2:
        return "unknown", "unknown"
    return fields[0], fields[1]


def assemble(total, cache):
    """`total` valid statements (k < total) and total / 2 false ones (k >= total)"""
    import bench
    nfalse = total // 2
    if cache and os.path.exists(cache):
        with open(cache, "rb") as f:
            built = pickle.load(f)
        if len(built) == total + nfalse:
            return built
    jobs = [("sm" if k % 2 == 0 else "lt", k, k < total) for k in range(total + nfalse)]
    with mp.get_context("spawn").Pool(max(1, min(16, os.cpu_count() or 1))) as pool:
        built = pool.map(bench._cfg5_assemble, jobs, chunksize=32)
    if cache:
        with open(cache, "wb") as f:
            pickle.dump(built, f)
    return built


def mix(total, pct):
    """statement indices of a mix of `total` with pct % false ones at evenly spaced positions"""
    nbad = total * pct // 100
    bad = {(j * total) // nbad for j in range(nbad)} if nbad else set()
    out, nv, nf = [], 0, 0
    for pos in range(total):
        if pos in bad:
            out.append(total + nf); nf += 1
        else:
            out.append(nv); nv += 1
    return out


def main():
    import bulletproofs_gadgets_b200 as bpg
    ap = argparse.ArgumentParser()
    ap.add_argument("--total", type=int, default=8192)
    ap.add_argument("--contexts", type=int, default=8)
    ap.add_argument("--per-call", default="64,256")
    ap.add_argument("--entry", default="batch,each")
    ap.add_argument("--invalid", default="0,1,10,50")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--cache", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    built = assemble(args.total, args.cache)
    NCTX = args.contexts
    ctxs = [bpg.Context(0) for _ in range(NCTX)]
    for c in ctxs:
        c.gens_ensure(512)
    # circuits and proofs on context 0 (verification only needs the device: any context of it will do)
    c0 = ctxs[0]
    wit = [(n, m, wp, wv, wc, v, inL, inR) for (k, label, n, m, rp, tv, tc, (inL, inR, wp, wv, wc), v, vb, valid) in built]
    handles = c0.circuit_create_batch([(n, m, rp, tv, tc) for (k, label, n, m, rp, tv, tc, _, v, vb, valid) in built])
    items, expected = [], []
    for b0 in range(0, len(built), 256):
        chunk = range(b0, min(len(built), b0 + 256))
        ws = c0.witness_eval_batch([wit[i] for i in chunk])
        got = c0.prove_batch([(handles[i], built[i][1], w[0], w[1], w[2], built[i][8], built[i][9], hashlib.sha256(b"cfg5 ext %d" % built[i][0]).digest())
                              for i, w in zip(chunk, ws)])
        for i, (proof, V) in zip(chunk, got):
            items.append((handles[i], built[i][1], V, proof, hashlib.sha256(b"cfg5 verify ext %d" % built[i][0]).digest()))
            expected.append(built[i][10])

    def timed(idx_set, B, entry):
        calls = [idx_set[b:b + B] for b in range(0, len(idx_set), B)]
        out = {}

        def lane(ci):
            c = ctxs[ci]
            for chunk in calls[ci::NCTX]:
                for i, acc in zip(chunk, getattr(c, "verify_" + entry)([items[i] for i in chunk])):
                    out[i] = acc
        for c in ctxs:
            c.sync()
        l0 = sum(c.launch_count() for c in ctxs)
        cpu0, t0 = time.process_time(), time.perf_counter()
        with ThreadPoolExecutor(NCTX) as tp:
            list(tp.map(lane, range(NCTX)))
        for c in ctxs:
            c.sync()
        dt, cpu = time.perf_counter() - t0, time.process_time() - cpu0
        n = len(idx_set)
        return out, {"verifications_per_sec": n / dt, "seconds": dt, "launches_per_verification": (sum(c.launch_count() for c in ctxs) - l0) / n,
                     "host_cpu_ms_per_verification": 1e3 * cpu / n}

    entries = [e for e in args.entry.split(",") if e == "batch" or hasattr(bpg.Context, "verify_" + e)]
    runs, digests = {}, {}
    for pct in [int(x) for x in args.invalid.split(",")]:
        idx_set = mix(args.total, pct)
        for entry in entries:
            for B in [int(x) for x in args.per_call.split(",")]:
                timed(idx_set, B, entry)  # warm-up at this shape (the first call of a shape grows the scratch buffers)
                reps = [timed(idx_set, B, entry) for _ in range(args.repeat)]
                got = reps[-1][0]
                rates = sorted(r[1]["verifications_per_sec"] for r in reps)
                digest = hashlib.sha256(bytes(int(got[i]) for i in idx_set)).hexdigest()
                runs["%s_per_call_%d_invalid_%dpct" % (entry, B, pct)] = {
                    "verifications": len(idx_set), "invalid": sum(1 for i in idx_set if not expected[i]),
                    "median_verifications_per_sec": rates[len(rates) // 2], "runs": [r[1] for r in reps],
                    "verdicts_match_expected": all(got[i] == expected[i] for i in idx_set), "verdict_digest": digest}
                digests.setdefault("invalid_%dpct" % pct, set()).add(digest)
    result = {"gpu": name, "power_limit": power, "statements": args.total, "contexts": NCTX, "entries": entries, "runs": runs,
              "verdict_digests": {k: sorted(v) for k, v in digests.items()},
              "digests_equal_across_entries_and_sizes": all(len(v) == 1 for v in digests.values())}
    for h in handles:
        c0.lib.bpg_circuit_destroy(h)
    for c in ctxs:
        c.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
