#!/usr/bin/env python3
"""End-to-end proving pipeline on the BASELINE configs[4] mix: `total` SET_MEMBER / LESS_THAN statements (1 % false), assembled
as bench.batch_verify_config5 does, proved on 8 contexts in threads, `--per-call` statements per bpg_r1cs_prove_batch call.
Each timed window covers the set-up of a chunk (witness evaluation and circuit upload), its proofs and the destruction of
its circuits:
  (a) per-statement set-up: one bpg_witness_eval and one bpg_circuit_create per statement
  (b) batched set-up: one bpg_witness_eval_batch and one bpg_circuit_create_batch per chunk
Both variants pass the same host arrays to the library, so they differ only in the native calls.  Reports proofs/s, the
set-up time, launches and host CPU per proof, and whether the proofs of (a) and (b) are byte-identical.  Prints one JSON line
(and writes it to --out if given).

    python tools/bench_prove_pipeline.py [--total 8192] [--per-call 256] [--out path]"""
import argparse
import ctypes as C
import hashlib
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
NCTX = 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split(",")]
    return name, power


def main():
    import bench
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200.api import _u32_array
    ap = argparse.ArgumentParser()
    ap.add_argument("--total", type=int, default=8192)
    ap.add_argument("--per-call", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B = args.per_call
    name, power = gpu_info()
    jobs = [("sm" if k % 2 == 0 else "lt", k, (k % 100) != 37) for k in range(args.total)]
    with mp.get_context("spawn").Pool(max(1, min(16, os.cpu_count() or 1))) as pool:
        built = pool.map(bench._cfg5_assemble, jobs, chunksize=32)
    # host arrays of every statement, shared by both variants: witness item and CSR entry as the Context batch calls take them
    wit = [(n, m, wp, wv, wc, v, inL, inR) for (k, label, n, m, rp, tv, tc, (inL, inR, wp, wv, wc), v, vb, valid) in built]
    csr = [(n, m, rp, tv, tc) for (k, label, n, m, rp, tv, tc, _, v, vb, valid) in built]
    tail = [(label, v, vb, hashlib.sha256(b"cfg5 ext %d" % k).digest()) for (k, label, n, m, rp, tv, tc, _, v, vb, valid) in built]
    ctxs = [bpg.Context(0) for _ in range(NCTX)]
    for c in ctxs:
        c.gens_ensure(512)

    def setup_per_statement(c, chunk):
        out = []
        for idx in chunk:
            n, m, wp, wv, wc, v, inL, inR = wit[idx]
            aL, aR, aO = C.create_string_buffer(inL, 32 * max(1, n)), C.create_string_buffer(inR, 32 * max(1, n)), C.create_string_buffer(32 * max(1, n))
            c.check(c.lib.bpg_witness_eval(c.h, n, m, _u32_array(wp), _u32_array(wv), wc, v, aL, aR, aO))
            _, _, rp, tv, tc = csr[idx]
            h = C.c_void_p()
            c.check(c.lib.bpg_circuit_create(c.h, n, m, len(rp) - 1, _u32_array(rp), _u32_array(tv), tc, C.byref(h)))
            out.append((h, (aL.raw[:32 * n], aR.raw[:32 * n], aO.raw[:32 * n])))
        return out

    def setup_batched(c, chunk):
        ws = c.witness_eval_batch([wit[i] for i in chunk])
        return list(zip(c.circuit_create_batch([csr[i] for i in chunk]), ws))

    def variant(setup):
        def run(ci, idxs, out, setup_s):
            c = ctxs[ci]
            for b0 in range(0, len(idxs), B):
                chunk = idxs[b0:b0 + B]
                t0 = time.perf_counter()
                hw = setup(c, chunk)
                setup_s[ci] += time.perf_counter() - t0
                items = [(h, tail[i][0], w[0], w[1], w[2], tail[i][1], tail[i][2], tail[i][3]) for i, (h, w) in zip(chunk, hw)]
                try:
                    for i, r in zip(chunk, c.prove_batch(items)):
                        out[i] = r
                finally:
                    for h, _ in hw:
                        c.lib.bpg_circuit_destroy(h)
        return run

    def timed(fn, idx_set):
        out, setup_s = {}, [0.0] * NCTX
        slices = [[i for i in idx_set if i % NCTX == ci] for ci in range(NCTX)]
        for c in ctxs:
            c.sync()
        l0 = sum(c.launch_count() for c in ctxs)
        cpu0, t0 = time.process_time(), time.perf_counter()
        with ThreadPoolExecutor(NCTX) as tp:
            list(tp.map(lambda ci: fn(ci, slices[ci], out, setup_s), range(NCTX)))
        for c in ctxs:
            c.sync()
        dt, cpu = time.perf_counter() - t0, time.process_time() - cpu0
        launches = sum(c.launch_count() for c in ctxs) - l0
        n = len(idx_set)
        return out, {"proofs_per_sec": n / dt, "seconds": dt, "setup_seconds_per_context": sum(setup_s) / NCTX,
                     "setup_share": sum(setup_s) / NCTX / dt, "launches_per_proof": launches / n, "host_cpu_ms_per_proof": 1e3 * cpu / n}

    per_statement, batched = variant(setup_per_statement), variant(setup_batched)
    # each variant is warmed at its own per-call shape: the first call of a shape grows the scratch buffers (cudaFree / cudaMalloc
    # synchronise the device shared by all contexts)
    warm = list(range(min(len(built), NCTX * B)))
    timed(per_statement, warm)
    timed(batched, warm)
    everything = list(range(len(built)))
    ref, ra = timed(per_statement, everything)
    got, rb = timed(batched, everything)
    ra["cuda_malloc_and_free_per_statement"] = 2          # bpg_circuit_create: one allocation per circuit, freed by bpg_circuit_destroy
    rb["cuda_malloc_and_free_per_statement"] = 2.0 / B    # bpg_circuit_create_batch: one allocation per chunk
    result = {"gpu": name, "power_limit": power, "proofs": len(built), "invalid_statements": sum(1 for j in jobs if not j[2]), "contexts": NCTX,
              "per_call": B, "per_statement_setup": ra, "batched_setup": rb,
              "batched_over_per_statement": rb["proofs_per_sec"] / ra["proofs_per_sec"],
              "proof_bytes_equal": all(got[i] == ref[i] for i in everything)}
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
