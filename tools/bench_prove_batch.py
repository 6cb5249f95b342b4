#!/usr/bin/env python3
"""Proving throughput on the BASELINE configs[4] mix: `total` SET_MEMBER / LESS_THAN proofs (1 % false statements), assembled
as bench.batch_verify_config5 does, proved on 8 contexts in threads (a) one bpg_r1cs_prove per proof, as bench.py does, and
(b) with bpg_r1cs_prove_batch in batches of 16 / 64 / 256 per call.  Every batched proof is compared with the per-proof bytes.
Prints one JSON line (and writes it to --out if given).

    python tools/bench_prove_batch.py [--total 8192] [--out path]"""
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
CAP = 1 + 32 * (14 + 64 + 2)
NCTX = 8
BATCHES = (16, 64, 256)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split(",")]
    return name, power


def main():
    import bench
    import bulletproofs_gadgets_b200 as bpg
    ap = argparse.ArgumentParser()
    ap.add_argument("--total", type=int, default=8192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    jobs = [("sm" if k % 2 == 0 else "lt", k, (k % 100) != 37) for k in range(args.total)]
    with mp.get_context("spawn").Pool(max(1, min(16, os.cpu_count() or 1))) as pool:
        built = pool.map(bench._cfg5_assemble, jobs, chunksize=32)
    ctxs = [bpg.Context(0) for _ in range(NCTX)]
    for c in ctxs:
        c.gens_ensure(512)
    # witness (bpg_witness_eval) and circuit of every proof on the context that proves it; untimed
    items = [None] * len(built)

    def setup(ci):
        c = ctxs[ci]
        for idx in range(ci, len(built), NCTX):
            k, label, n, m, rp, tv, tc, (inL, inR, wp, wv, wc), v, vb, valid = built[idx]
            aL, aR, aO = C.create_string_buffer(inL, 32 * n), C.create_string_buffer(inR, 32 * n), C.create_string_buffer(32 * n)
            c.check(c.lib.bpg_witness_eval(c.h, n, m, (C.c_uint32 * len(wp))(*wp), (C.c_uint32 * max(1, len(wv)))(*wv), wc, v, aL, aR, aO))
            h = C.c_void_p()
            c.check(c.lib.bpg_circuit_create(c.h, n, m, len(rp) - 1, (C.c_uint32 * len(rp))(*rp), (C.c_uint32 * max(1, len(tv)))(*tv), tc, C.byref(h)))
            items[idx] = (h, label, aL.raw[:32 * n], aR.raw[:32 * n], aO.raw[:32 * n], v, vb, hashlib.sha256(b"cfg5 ext %d" % k).digest())

    with ThreadPoolExecutor(NCTX) as tp:
        list(tp.map(setup, range(NCTX)))

    def per_proof(ci, idxs, out):
        c = ctxs[ci]
        for idx in idxs:
            it = items[idx]
            m = len(it[5]) // 32
            proof, V = C.create_string_buffer(CAP), C.create_string_buffer(32 * max(1, m))
            rc = c.lib.bpg_r1cs_prove(c.h, it[0], it[1], len(it[1]), it[2], it[3], it[4], it[5], it[6], it[7], 0, V, proof, CAP)
            c.check(rc)
            out[idx] = (proof.raw[:rc], V.raw[:32 * m])

    def batched(B):
        def run(ci, idxs, out):
            c = ctxs[ci]
            for b0 in range(0, len(idxs), B):
                chunk = idxs[b0:b0 + B]
                for idx, r in zip(chunk, c.prove_batch([items[i] for i in chunk])):
                    out[idx] = r
        return run

    def timed(fn, idx_set):
        out = {}
        slices = [[i for i in idx_set if i % NCTX == ci] for ci in range(NCTX)]
        for c in ctxs:
            c.sync()
        l0 = sum(c.launch_count() for c in ctxs)
        cpu0, t0 = time.process_time(), time.perf_counter()
        with ThreadPoolExecutor(NCTX) as tp:
            list(tp.map(lambda ci: fn(ci, slices[ci], out), range(NCTX)))
        for c in ctxs:
            c.sync()
        dt, cpu = time.perf_counter() - t0, time.process_time() - cpu0
        launches = sum(c.launch_count() for c in ctxs) - l0
        n = len(idx_set)
        return out, {"proofs_per_sec": n / dt, "seconds": dt, "launches_per_proof": launches / n, "host_cpu_ms_per_proof": 1e3 * cpu / n}

    # every variant is warmed at its own per-call shape: the first call of a shape grows the scratch buffers (cudaFree / cudaMalloc
    # synchronise the device shared by all contexts)
    warm = list(range(min(len(items), NCTX * max(BATCHES))))
    timed(per_proof, warm)
    for B in BATCHES:
        timed(batched(B), warm)
    everything = list(range(len(items)))
    ref, res_single = timed(per_proof, everything)
    result = {"gpu": name, "power_limit": power, "proofs": len(items), "invalid_statements": sum(1 for j in jobs if not j[2]), "contexts": NCTX,
              "per_proof": res_single, "batched": {}}
    for B in BATCHES:
        got, r = timed(batched(B), everything)
        r["bytes_equal_per_proof_path"] = all(got[i] == ref[i] for i in everything)
        r["speedup_vs_per_proof"] = r["proofs_per_sec"] / res_single["proofs_per_sec"]
        result["batched"][str(B)] = r
    result["all_batched_bytes_equal"] = all(r["bytes_equal_per_proof_path"] for r in result["batched"].values())
    for it in items:
        ctxs[0].lib.bpg_circuit_destroy(it[0])
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
