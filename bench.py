#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native Bulletproofs R1CS hot path.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W

Metric (BASELINE.json): R1CS proofs/sec (and MSM Mpoints/sec in the `msm*` sweeps) on BASELINE configs[3], the size
north_star's target sentence names: "synthetic R1CS circuit 2^20 multipliers (MSM ~2^21 points, IPP 20 rounds)" --
993 384 multipliers (the reference's own largest circuit, merkle_tree_gadget.rs:473-545), N = 2^20, byte-exact proofs.
The circuit is the reference's test_merkle_tree_gadget_512: MerkleTree256 over 512 committed leaves (511 two-block MiMC nodes).
A proof = 512 Pedersen commits, 3 commitment MSMs of 2n+1 / n+1 / 2n+1 points, polynomial phase, 20 IPP rounds.
A step = P proofs, one per concurrent prover of the GPU (own host thread + bpg_ctx + witness each; P is in `config`);
every prover runs through its `steps` proofs of the timed region without waiting for the others, so the sequential host-side Merlin
TranscriptRng of one proof (2n draws, ~0.7 s of one core at this size; the streams of concurrent provers share SIMD
lanes) overlaps the device work of the others.  Every rank runs its own provers (weak scaling, no data-path collective).

  value         proofs/s, witness vectors already resident in HBM (BPG_FLAG_WITNESS_ON_DEVICE)
  e2e           proofs/s through the C ABI with HOST buffers: witness H2D, proof + commitments D2H inside the timed region
  roofline      the dominant kernel k_msm_accumulate against what binds it, the integer-multiply pipe (measured MAC32/s of a
                dependent field-multiply chain); the HBM view (100 B per (term, window) pair) is listed beside it
  cpu_baseline  the C oracle (oracle/bpo.c, a restatement of dalek's algorithms) on the host cores, same circuit, and the
                GPU's proof bytes are compared with the oracle's
Extras: MSM sweeps 2^16..2^22 with the oracle's Mpoints/s beside every point, MiMC, BASELINE configs[1] and [4]
(batch verification of 8192 set_membership / less_than proofs, sharded by rank, verdicts == oracle), and for N > 1 the
oracle-parity checks of the sharded MSM and the sharded prover.

--dump-outputs DIR: after the run, DIR/proofs.npy and DIR/commitments.npy hold what the timed region (`value`; for
`--impl reference` its oracle proofs) returned in its last step: one row per prover of rank 0, the proof bytes and the
commitment bytes V as float32 values 0..255.  The inputs of that step depend on the arguments only, so two builds of the
project can be compared output for output.

The reference itself (Rust) cannot be built in this image; `--impl reference` times the oracle port.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

# the concurrent provers use one CUDA stream each: give every stream its own hardware work queue (default: 8 shared)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_emit = print
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = "synthetic R1CS circuit 2^20 multipliers (MSM ~2^21 points, IPP 20 rounds) at 1/2/4/8 GPUs"
NLEAVES = 512             # the reference's largest circuit: 512-leaf MiMC Merkle tree, 511 nodes x 1944 = 993 384 multipliers
N_MULT = (NLEAVES - 1) * 1944
GENS_CAP = 1 << 20
REF_SAMPLE_LEAVES = 32    # reference arm: every step proves the 32-leaf tree of the same family (31 nodes, N = 2^16): bounded sample
DTYPE = "u32 limbs (GF(2^255-19), Z_l)"


def config_dict():
    """identical in both arms (the driver compares them)"""
    return {"workload": WORKLOAD, "n_multipliers": N_MULT, "padded_n": GENS_CAP, "commitments": NLEAVES,
            "circuit": "MerkleTree256 over %d committed leaves, library API: the reference's test_merkle_tree_gadget_512 "
                       "(merkle_tree_gadget.rs:473-545, BulletproofGens::new(1048576, 1))" % NLEAVES,
            "byte_exact": True}


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local, dist


def barrier_max(dist, local, value):
    """barrier + max over ranks of a python float"""
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device="cuda:%d" % local)
    dist.barrier()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def oracle_prove(inst, cap, ext, threads):
    """-> (seconds, proof, V) of the CPU oracle prover (oracle/bpo.c) on `threads` OpenMP threads"""
    import oracle_lib as ol
    ol.lib().bpo_set_threads(threads)
    rp, tv, tc = inst["csr"]  # (instances of one family share the coefficient array; reading "csr" installs this instance's constant)
    tcb = tc.tobytes() if hasattr(tc, "tobytes") else tc
    t0 = time.perf_counter()
    proof, V = ol.r1cs_prove(inst["label"], cap, inst["aL"], inst["aR"], inst["aO"], inst["vals"], inst["blinds"], rp, tv, tcb, ext)
    return time.perf_counter() - t0, proof, V


def dump_outputs(path, outputs):
    """--dump-outputs: `outputs` = the (proof, V) byte strings of one step, one per prover, written as float32 arrays of byte
    values (exact); the rows beyond the first that fit in 64 MB are left out"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    row_bytes = 4 * (len(outputs[0][0]) + len(outputs[0][1]))
    outputs = outputs[:max(1, (64 << 20) // row_bytes)]
    for name, col in (("proofs", 0), ("commitments", 1)):
        rows = np.array([np.frombuffer(o[col], dtype=np.uint8) for o in outputs], dtype=np.float32)
        np.save(os.path.join(path, name + ".npy"), rows)


def run_reference(args):
    """Reference arm: the reference's CPU algorithm for the same path on the host cores (oracle port, OpenMP on all cores; the
    Rust crate cannot be built here).  A complete 2^20 proof takes the oracle ~20 s on 16 cores, so every step is a bounded
    sample: one complete proof of the SAME circuit family at 1/16 of the size (the 32-leaf instead of the 512-leaf tree, N = 2^16);
    proving cost is linear in the multiplier count (constant-time Straus commitments + per-element generator folds; the
    Pippenger share only gets cheaper per point with size), so proofs/s at full size = sample proofs/s / (n_full / n_sample).
    bench.py's own arm times ONE complete full-size oracle proof beside the GPU figure (cpu_baseline) as the calibration."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from bulletproofs_gadgets_b200 import gadgets
    import oracle_lib as ol
    cores = os.cpu_count() or 1
    full = os.environ.get("BPG_REF_FULL") == "1"
    inst = gadgets.merkle_tree_instances(NLEAVES if full else REF_SAMPLE_LEAVES, [None], trace_on_device=False)[0]
    cap = 1
    while cap < inst["n"]:
        cap *= 2
    scale = N_MULT / inst["n"]
    ol.gens(0, cap)  # BulletproofGens::new outside the timed steps, as for the GPU arm
    for _ in range(args.warmup):
        oracle_prove(inst, cap, bytes(32), cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, proof, V = oracle_prove(inst, cap, bytes(32), cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(proof, V)])
    v = args.steps / dt / scale
    sample = ("every step = 1 complete oracle proof of a %d-multiplier circuit of the same family (N = %d), OpenMP on all host cores; "
              "value = sample proofs/s / %.2f (cost linear in the multiplier count)" % (inst["n"], cap, scale)) if not full else \
        "full workload: complete proofs of the 993 384-multiplier circuit, OpenMP on all host cores"
    line = {"impl": "reference", "metric": "r1cs_proofs_per_sec", "value": v, "unit": "proofs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic", "config": config_dict(),
            "cpu_baseline": {"value": v, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------- MSM sweeps
def cpu_msm_mpoints(n, dist_kind, cores):
    """oracle (dalek's vartime Pippenger restated, OpenMP) Mpoints/s on the same kind of input, n capped so it stays ~seconds"""
    import numpy as np
    import oracle_lib as ol
    rng = np.random.default_rng(1 if dist_kind == "uniform" else 2)
    h = n // 2
    if dist_kind == "uniform":
        raw = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        raw[:, 31] &= 0x0F
    else:
        raw = np.zeros((n, 32), dtype=np.uint8)
        raw[:, 0] = rng.integers(0, 2, size=n, dtype=np.uint8)
    ol.lib().bpo_set_threads(cores)
    ol.gens(0, h)
    sG, sH = raw[:h].tobytes(), raw[h:2 * h].tobytes()
    t0 = time.perf_counter()
    out = ol.msm_gens(sG, sH, h, 0)
    dt = time.perf_counter() - t0
    return n / dt / 1e6, out, (sG, sH)


def msm_sweep(ctx, sizes, reps=5, dist="uniform", cpu_sizes=(), cores=1):
    """MSM Mpoints/s over the resident generators with device-resident scalars (points = n/2 G + n/2 H).
    dist = "uniform": 252-bit scalars (SURVEY 8d MSM-uniform); "bits": scalars in {0, 1} (MSM-bits, the range-proof shape).
    For the sizes in cpu_sizes the oracle's vartime MSM runs on the same scalars: its Mpoints/s is listed beside the GPU's and
    the compressed results must be equal."""
    import ctypes as C
    import numpy as np
    out = {}
    for n in sizes:
        h = n // 2
        # the same stream as cpu_msm_mpoints (fresh generator per size so both sides see identical scalars)
        r2 = np.random.default_rng(1 if dist == "uniform" else 2)
        if dist == "uniform":
            raw = r2.integers(0, 256, size=(n, 32), dtype=np.uint8)
            raw[:, 31] &= 0x0F
        else:
            raw = np.zeros((n, 32), dtype=np.uint8)
            raw[:, 0] = r2.integers(0, 2, size=n, dtype=np.uint8)
        d = ctx.dev_alloc(32 * n)
        ctx.dev_upload(d, raw.tobytes())
        dG, dH = d, C.c_void_p(d.value + 32 * h)
        got = ctx.msm_gens_dev(dG, dH, h, 0)  # warm-up (sizes exceed L2 only from 2^20 up; tables are re-gathered randomly)
        ctx.event_record(0)
        for _ in range(reps):
            ctx.msm_gens_dev(dG, dH, h, 0)
        ctx.event_record(1)
        ms = ctx.event_elapsed_ms(0, 1) / reps
        out[str(n)] = {"ms": ms, "mpoints_per_s": n / ms / 1e3}
        if n in cpu_sizes:
            cpu_mp, want, _ = cpu_msm_mpoints(n, dist, cores)
            out[str(n)].update({"cpu_mpoints_per_s": cpu_mp, "cpu_cores": cores, "equals_oracle": got == want})
        ctx.dev_free(d)
    return out


def msm_var_sweep(ctx, sizes, reps=3, cpu_sizes=(), cores=1):
    """SURVEY 8d MSM-var: variable-base MSM through the host-buffer entry point bpg_msm (n compressed points + n scalars
    uploaded, decompressed, bucket method): the path of the verifier's own points.  Host-timed (the call is synchronous)."""
    import numpy as np
    import oracle_lib as ol
    out = {}
    rng = np.random.default_rng(3)
    maxn = max(sizes)
    G, H = ctx.gens_export(0, min(maxn // 2, ctx.gens_capacity()))
    pts = G + H
    while len(pts) < 32 * maxn:
        pts = pts + pts
    raw = rng.integers(0, 256, size=(maxn, 32), dtype=np.uint8)
    raw[:, 31] &= 0x0F
    sc = raw.tobytes()
    # the caller's buffers are page-locked (bpg_host_alloc), as a host application feeding large MSMs would keep them
    h_sc, hh_sc = ctx.host_alloc(sc)
    h_pt, hh_pt = ctx.host_alloc(pts[:32 * maxn])
    for n in sizes:
        got = ctx.msm(h_sc, h_pt, n)
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.msm(h_sc, h_pt, n)
        ms = (time.perf_counter() - t0) * 1e3 / reps
        out[str(n)] = {"ms": ms, "mpoints_per_s": n / ms / 1e3, "h2d_bytes": 64 * n, "host_buffers": "page-locked"}
        if n in cpu_sizes:
            sn, pn = sc[:32 * n], pts[:32 * n]
            ol.lib().bpo_set_threads(cores)
            t0 = time.perf_counter()
            want = ol.msm(sn, pn)
            dt = time.perf_counter() - t0
            out[str(n)].update({"cpu_mpoints_per_s": n / dt / 1e6, "cpu_cores": cores, "equals_oracle": got == want})
    ctx.host_free(hh_sc)
    ctx.host_free(hh_pt)
    return out


def fold_sweep(ctx, sizes, peak_mac):
    """the literal IPP generator fold as a standalone op (bpg_fold_points: out_i = u^-1 P_i + u Q_i, SURVEY 8a a7 / K5).  Kernel
    time from the library's events around k_fold_kernel; work per output: 252 doublings + <= 142 additions of 8 field
    multiplications each (shared-scalar Straus) = 2.27e5 MAC32."""
    import numpy as np
    import oracle_lib as ol
    out = {}
    maxn = max(sizes)
    G, H = ctx.gens_export(0, maxn)
    rng = np.random.default_rng(9)
    sl = (int.from_bytes(rng.bytes(32), "little") >> 4).to_bytes(32, "little")
    sr = (int.from_bytes(rng.bytes(32), "little") >> 4).to_bytes(32, "little")
    mac_per_output = (252 + 142) * 8 * 72.0
    for n in sizes:
        ctx.fold_points(sl, sr, G[:32 * n], H[:32 * n])
        t0 = time.perf_counter()
        got = ctx.fold_points(sl, sr, G[:32 * n], H[:32 * n])
        dt = time.perf_counter() - t0
        kms = ctx.event_elapsed_ms(12, 13)
        out[str(n)] = {"kernel_ms": kms, "outputs_per_sec_kernel": n / (kms * 1e-3), "outputs_per_sec_e2e": n / dt,
                       "int_frac": n * mac_per_output / (kms * 1e-3) / peak_mac}
        if n <= 4096:
            out[str(n)]["equals_oracle"] = got == ol.fold_points(sl, sr, G[:32 * n], H[:32 * n])
    return out


def msm_sharded_sweep(ctx, dist, local, rank, world, sizes, reps=5, parity_n=1 << 16):
    """ONE MSM of n points split by point range over the ranks (DESIGN.md section 6, parallel.msm_gens_sharded): every rank
    sums its slice of the resident generators, the 128-byte partial points are all-gathered over NCCL and added on every rank.
    Timed on the host around barrier + synchronize (the collective runs on torch's stream), max over ranks.
    `oracle_parity`: at parity_n points rank 0 also runs the CPU oracle on the full scalar vectors; every rank's sharded
    result must equal it (multi-GPU parity that the 1-GPU test box cannot show)."""
    import ctypes as C
    import numpy as np
    from bulletproofs_gadgets_b200 import parallel
    out = {}
    maxn = max(sizes)
    ctx.gens_ensure(maxn // 2)
    rng = np.random.default_rng(7)
    dev = "cuda:%d" % local
    parallel.enable_comm(ctx, dev)  # the library's own NCCL communicator: the all-gather is enqueued on the context's stream
    for n in [parity_n] + list(sizes):
        h = n // 2
        lo, hi = parallel.shard_range(h, rank, world)
        raw = rng.integers(0, 256, size=(2 * h, 32), dtype=np.uint8)  # same stream on every rank: sG | sH
        raw[:, 31] &= 0x0F
        mine = np.concatenate([raw[lo:hi], raw[h + lo:h + hi]])
        d = ctx.dev_alloc(32 * len(mine))
        ctx.dev_upload(d, mine.tobytes())
        dG, dH = d, C.c_void_p(d.value + 32 * (hi - lo))
        first = parallel.msm_gens_sharded(ctx, dG, dH, h, dev)  # warm-up, and a cross-rank agreement check
        agree = parallel.allgather_bytes(first, dev)
        if any(a != first for a in agree):
            raise SystemExit("sharded MSM: ranks disagree on the result")
        if n == parity_n and "oracle_parity" not in out:
            want = first
            if rank == 0:
                import oracle_lib as ol
                ol.lib().bpo_set_threads(os.cpu_count() or 1)
                want = ol.msm_gens(raw[:h].tobytes(), raw[h:].tobytes(), h, 0)
            want = parallel.allgather_bytes(want, dev)[0]
            if want != first:
                raise SystemExit("sharded MSM: result differs from the CPU oracle")
            out["oracle_parity"] = {"points": n, "all_ranks_equal_oracle": True}
            ctx.dev_free(d)
            continue
        barrier_max(dist, local, 0.0)
        t0 = time.perf_counter()
        for _ in range(reps):
            parallel.msm_gens_sharded(ctx, dG, dH, h, dev)
        ms = barrier_max(dist, local, (time.perf_counter() - t0) * 1e3 / reps)
        out[str(n)] = {"ms": ms, "mpoints_per_s": n / ms / 1e3, "points_per_rank": 2 * (hi - lo)}
        ctx.dev_free(d)
    parallel.disable_comm(ctx)
    out["exchange"] = "ncclAllGather of the 128-byte partial points enqueued by libbpg on the context's stream (bpg_comm_init)"
    return out


def one_large_proof(bpg, gadgets, ctx, inst, dist, local, rank, world):
    """ONE proof of the headline circuit on `world` GPUs -- strong scaling.  With world > 1 every MSM of the proof is cut by point
    range over the ranks (bpg_ctx_set_shard) and the partial points are all-gathered; all ranks return the same bytes (checked).
    Latency is quoted with device-side blinding (the 2n sequential transcript-RNG draws of the byte-exact mode, ~0.7 s of one
    host core, are the same on every rank and hide nothing here); `oracle_parity` proves byte-exactness of the sharded prover
    against the CPU oracle on a mid-size circuit of the same family (rank 0 runs the oracle, every rank must match)."""
    from bulletproofs_gadgets_b200 import parallel
    dev = "cuda:%d" % local
    circ = gadgets.Circuit(ctx, inst["n"], inst["m"], inst["csr"])
    if world > 1:
        parallel.enable_comm(ctx, dev)
    FAST = bpg._lib.FLAG_FAST_BLINDING
    ext = b"\x44" * 32
    res = {"n_multipliers": inst["n"], "padded_n": GENS_CAP, "gpus": world}
    if world > 1:
        mid = gadgets.merkle_tree_instances(16, [11], ctx=ctx)[0]  # 29 160 multipliers, N = 2^15: late fold + sharded exchange paths
        cm = gadgets.Circuit(ctx, mid["n"], mid["m"], mid["csr"])
        got = cm.prove(mid, b"\x45" * 32)
        want = got
        if rank == 0:
            _, p, V = oracle_prove(mid, 1 << 15, b"\x45" * 32, os.cpu_count() or 1)
            want = (p, V)
        wb = parallel.allgather_bytes(want[0] + want[1], dev)[0]
        if wb != got[0] + got[1]:
            raise SystemExit("sharded prover: proof bytes differ from the CPU oracle")
        cm.close()
        res["oracle_parity"] = {"n_multipliers": mid["n"], "all_ranks_equal_oracle": True}
    # the witness is made resident first (as for `value`): the strong-scaling figure is the device path, not a replicated H2D copy
    import ctypes as C
    n = inst["n"]
    d_w = ctx.dev_alloc(3 * 32 * n)
    ctx.dev_upload(d_w, inst["aL"] + inst["aR"] + inst["aO"])
    host_inst = inst
    inst = dict(inst)
    inst["aL"], inst["aR"], inst["aO"] = (C.cast(C.c_void_p(d_w.value + 32 * n * k), C.c_char_p) for k in range(3))
    FAST |= bpg._lib.FLAG_WITNESS_ON_DEVICE
    proof, V = circ.prove(inst, ext, FAST)  # warm-up (buffers, late-fold tables)
    if world > 1:
        same = parallel.allgather_bytes(proof, dev)
        if any(p != proof for p in same):
            raise SystemExit("sharded prover: ranks returned different proof bytes")
    if not circ.verify(inst["label"], V, proof):
        raise SystemExit("sharded prover: the verifier rejected the proof")
    barrier_max(dist, local, 0.0)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        circ.prove(inst, ext, FAST)
    ms = barrier_max(dist, local, (time.perf_counter() - t0) * 1e3 / reps)
    if world > 1:
        parallel.disable_comm(ctx)
    ctx.dev_free(d_w)
    inst = host_inst
    circ.close()
    res.update({"prove_ms_fast_blinding": ms, "proofs_per_sec": 1e3 / ms,
                "mode": "MSMs split by point range over the ranks; ncclAllGather of the partial points enqueued by libbpg on its own stream" if world > 1 else "one GPU"})
    return res


# ------------------------------------------------------------------------------------------------- BASELINE configs[4]
def _cfg5_assemble(job):
    """worker process (no CUDA): assemble one config-5 circuit through the front-end, return CSR + witness"""
    kind, k, valid = job
    import random
    from bulletproofs_gadgets_b200 import frontend as fe
    rnd = random.Random(60000 + k)
    label = b"cfg5-%d" % k
    if kind == "lt":
        a, b = sorted(rnd.sample(range(1 << 56), 2))
        if not valid:
            a, b = b, a
        run = fe.ProverRun(label, "LESS_THAN W0 W1\n", "", "W0 = 0x%014x\nW1 = 0x%014x\n" % (a, b), test_seed=k)
    else:
        vals = rnd.sample(range(1 << 40), 5)
        member = vals[1 + k % 4] if valid else vals[0]
        inst = "".join("I%d = 0x%010x\n" % (i, vals[1 + i]) for i in (0, 1, 2))
        wt = "W0 = 0x%010x\nW1 = 0x%010x\n" % (member, vals[4])
        run = fe.ProverRun(label, "SET_MEMBER W0 I0 W1 I1 I2\n", inst, wt, test_seed=k)
    p = run.prover
    enc = lambda xs: b"".join(int(x).to_bytes(32, "little") for x in xs)
    rp, tv, tc = p.csr()
    # the assignment is evaluated on the proving context's device (bpg_witness_eval): hand over the recorded combinations
    wit = (enc(p._in_L), enc(p._in_R), list(p._w_ptr), list(p._w_var), bytes(p._w_coeff))
    return (k, label, p.num_vars, len(p.v), rp, tv, tc, wit, enc(p.v), enc(p.v_blinding), valid)


def batch_verify_config5(bpg, ctx, dist, local, rank, world, total, cores):
    """BASELINE configs[4]: batch verification of `total` SET_MEMBER / LESS_THAN proofs (the shapes of the reference's
    tests/resources/set_membership.*, less_than.*: set size 4 with 40-bit values, 56-bit comparisons), 1 % of the statements
    false, sharded over the ranks (proof k -> rank k mod world, no collective; verdicts gathered at the end).
    The circuits are assembled by the front-end driver (frontend.py, the restated gadget library), proved on this rank's GPU,
    verified in batches of 64 by bpg_r1cs_verify_batch, and every verdict is compared with the CPU oracle verifier's."""
    import ctypes as C
    import multiprocessing as mp
    from concurrent.futures import ThreadPoolExecutor
    import oracle_lib as ol
    from bulletproofs_gadgets_b200 import parallel
    jobs = [("sm" if k % 2 == 0 else "lt", k, (k % 100) != 37) for k in range(total)]
    mine = [j for j in jobs if j[1] % world == rank]
    t0 = time.perf_counter()
    nproc = max(1, min(16, cores // max(world, 1)))
    with mp.get_context("spawn").Pool(nproc) as pool:
        built = pool.map(_cfg5_assemble, mine, chunksize=32)
    t_asm = time.perf_counter() - t0
    ctx.gens_ensure(512)
    nctx = 8
    ctxs = [ctx] + [bpg.Context(local) for _ in range(nctx - 1)]
    for c in ctxs:
        c.gens_ensure(512)
    items = [None] * len(built)

    def prove_slice(ci):
        c = ctxs[ci]
        for idx in range(ci, len(built), nctx):
            k, label, n, m, rp, tv, tc, (inL, inR, wp, wv, wc), v, vb, valid = built[idx]
            aL, aR, aO = C.create_string_buffer(inL, 32 * n), C.create_string_buffer(inR, 32 * n), C.create_string_buffer(32 * n)
            c.check(c.lib.bpg_witness_eval(c.h, n, m, (C.c_uint32 * len(wp))(*wp), (C.c_uint32 * max(1, len(wv)))(*wv), wc, v, aL, aR, aO))
            h = C.c_void_p()
            c.check(c.lib.bpg_circuit_create(c.h, n, m, len(rp) - 1, (C.c_uint32 * len(rp))(*rp), (C.c_uint32 * max(1, len(tv)))(*tv), tc, C.byref(h)))
            cap = 1 + 32 * (14 + 64 + 2)
            proof, V = C.create_string_buffer(cap), C.create_string_buffer(32 * max(1, m))
            ext = hashlib.sha256(b"cfg5 ext %d" % k).digest()
            rc = c.lib.bpg_r1cs_prove(c.h, h, label, len(label), aL, aR, aO, v, vb, ext, 0, V, proof, cap)
            if rc < 0:
                c.check(rc)
            items[idx] = (h, label, V.raw[:32 * m], proof.raw[:rc], os.urandom(32))

    t0 = time.perf_counter()
    with ThreadPoolExecutor(nctx) as tp:
        list(tp.map(prove_slice, range(nctx)))
    t_prove = time.perf_counter() - t0
    # circuits were created on their prover's context; verification only needs the device, any context of it will do
    B = 64

    def verify_slice(ci):
        c = ctxs[ci]
        out = {}
        for b0 in range(ci * B, len(items), nctx * B):
            chunk = items[b0:b0 + B]
            for j, acc in enumerate(c.verify_batch(chunk)):
                out[b0 + j] = acc
        return out

    for c in ctxs:
        c.sync()
    barrier_max(dist, local, 0.0)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(nctx) as tp:
        parts = list(tp.map(verify_slice, range(nctx)))
    for c in ctxs:
        c.sync()
    t_verify = barrier_max(dist, local, time.perf_counter() - t0)
    verdicts = {}
    for p in parts:
        verdicts.update(p)
    # oracle verdicts for this rank's shard (CPU), then everything is gathered
    ol.lib().bpo_set_threads(1)

    def oracle_one(idx):
        k, label, n, m, rp, tv, tc = built[idx][:7]
        _, _, V, proof, _ = items[idx]
        cap = 8
        while cap < n:
            cap *= 2
        return ol.r1cs_verify(label, cap, n, V, rp, tv, tc, proof, bytes(32))

    ol.gens(0, 512)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max(1, cores // max(world, 1))) as tp:
        want = list(tp.map(oracle_one, range(len(built))))
    t_oracle = time.perf_counter() - t0
    local_pairs = [(built[i][0], bool(verdicts[i])) for i in range(len(built))]
    all_gpu = parallel.gather_verdicts(local_pairs, total, "cuda:%d" % local if world > 1 else None)
    all_cpu = parallel.gather_verdicts([(built[i][0], bool(want[i])) for i in range(len(built))], total, "cuda:%d" % local if world > 1 else None)
    expected = [j[2] for j in jobs]
    for it in items:
        ctx.lib.bpg_circuit_destroy(it[0])
    for c in ctxs[1:]:
        c.close()
    return {"proofs": total, "invalid": expected.count(False), "gpus": world, "verify_s": t_verify, "verifications_per_sec": total / t_verify,
            "verdicts_match_oracle": all_gpu == all_cpu, "verdicts_match_expected": all_gpu == expected,
            "batch": B, "contexts_per_gpu": nctx, "shapes": "SET_MEMBER (set of 4, 40-bit values, 8 multipliers) / LESS_THAN (56-bit values, 379 multipliers)",
            "setup": {"assemble_s": t_asm, "gpu_prove_s": t_prove, "proofs_per_sec_proving": len(built) / t_prove, "oracle_verify_s": t_oracle,
                      "oracle_verifications_per_sec": len(built) / t_oracle, "oracle_threads": max(1, cores // max(world, 1))}}


# ------------------------------------------------------------------------------------------------------------ provers
class ProverLane:
    """one host thread's private context: own bpg_ctx (stream, workspace), circuit copy, own witness (host + HBM-resident)"""

    def __init__(self, bpg, gadgets, device, inst, cap, keep_bytes=True):
        import ctypes as C
        self.ctx = bpg.Context(device)
        self.ctx.gens_ensure(cap)
        self.inst = inst
        self.circ = gadgets.Circuit(self.ctx, inst["n"], inst["m"], inst["csr"])
        n = inst["n"]
        self.d_w = self.ctx.dev_alloc(3 * 32 * n)
        for k, key in enumerate(("aL", "aR", "aO")):
            self.ctx.dev_upload(C.c_void_p(self.d_w.value + 32 * n * k), inst[key])
        self.dev_inst = dict(inst)
        self.dev_inst["aL"], self.dev_inst["aR"], self.dev_inst["aO"] = (C.cast(C.c_void_p(self.d_w.value + 32 * n * k), C.c_char_p) for k in range(3))

        # the end-to-end leg hands the library HOST buffers: the witness sits in page-locked host memory (bpg_host_alloc), as
        # the bench contract's "inputs from pinned host memory" and as a Rust caller would keep its assignment vectors
        self.host_inst = dict(inst)
        self.h_w = []
        for k in ("aL", "aR", "aO"):
            ptr, handle = self.ctx.host_alloc(inst[k])
            self.host_inst[k] = ptr
            self.h_w.append(handle)
            if not keep_bytes:
                inst[k] = None  # the pageable copy is not needed again (48 lanes x 100 MB)

    def prove(self, ext, flags, resident):
        return self.circ.prove(self.dev_inst if resident else self.host_inst, ext, flags)

    def close(self):
        self.circ.close()
        for h in self.h_w:
            self.ctx.host_free(h)
        self.ctx.dev_free(self.d_w)
        self.ctx.close()


class LaneSet:
    """P free-running provers on one GPU; timed(flags, resident, steps) runs P * steps proofs, one per prover and step"""

    def __init__(self, bpg, gadgets, device, insts, cap, rank):
        from concurrent.futures import ThreadPoolExecutor
        self.lanes = [ProverLane(bpg, gadgets, device, inst, cap, keep_bytes=(k == 0)) for k, inst in enumerate(insts)]
        self.P = len(self.lanes)
        self.pool = ThreadPoolExecutor(max_workers=self.P)
        self.rank = rank
        self.host_cpu_ms = 0.0
        self.region = 0
        self.prefetch = True
        self.last = [None] * self.P  # (proof, V) of every lane's proof in the last step of the latest region

    def _ext(self, ticket):
        # every proof of the run gets its own 32 bytes standing for the reference's thread_rng draw
        return hashlib.sha256(b"bench ext %d %d %d" % (self.rank, self.region, ticket)).digest()

    def _lane_run(self, k, flags, resident, steps):
        """Lane k proves tickets k, k + P, ... (ticket s * P + k in step s), so every proof's witness and ext_rng32 are the same
        from run to run.  Before proving a ticket it hands the opening of its NEXT one to the library (bpg_r1cs_prove_prefetch),
        so the sequential transcript-RNG stream of that proof is drawn by a background host thread while this one is on the device."""
        ln = self.lanes[k]
        time.sleep(0.001 * k)  # staggered start (inside the timed region)
        tickets = range(k, self.P * steps, self.P)
        for i, cur in enumerate(tickets):
            if i + 1 < len(tickets) and self.prefetch:
                ln.circ.prefetch(ln.inst, self._ext(tickets[i + 1]), flags)
            self.last[k] = ln.prove(self._ext(cur), flags, resident)

    def timed(self, flags, resident, steps):
        """-> (ms, launches).  The region is bracketed by a sync of every context on both sides; device time by CUDA events on
        lane 0's stream, wall clock beside it, the larger of the two is reported."""
        self.region += 1
        self.last = [None] * self.P
        for ln in self.lanes:
            ln.ctx.sync()
        l0 = sum(ln.ctx.launch_count() for ln in self.lanes)
        ctx = self.lanes[0].ctx
        ctx.event_record(2)
        c0 = os.times()
        t0 = time.perf_counter()
        list(self.pool.map(lambda k: self._lane_run(k, flags, resident, steps), range(self.P)))
        for ln in self.lanes:
            ln.ctx.sync()
        ctx.event_record(3)
        ms_dev = ctx.event_elapsed_ms(2, 3)
        wall = (time.perf_counter() - t0) * 1e3
        c1 = os.times()
        self.host_cpu_ms = 1e3 * ((c1.user - c0.user) + (c1.system - c0.system)) / max(1, self.P * steps)
        return max(ms_dev, wall), sum(ln.ctx.launch_count() for ln in self.lanes) - l0

    def close(self):
        self.pool.shutdown()
        for ln in self.lanes:
            ln.close()


def run_ours(args):
    world, rank, local, dist = dist_setup()
    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import gadgets
    cores = os.cpu_count() or 1
    per_gpu = cores / max(world, 1)
    # Concurrent provers per GPU: a 2^20 proof is ~55 ms of device work and ~0.1 s of (lane-shared) host RNG, so a handful of
    # proofs in flight hide the host side; each prover holds ~1.3 GB of HBM workspace.
    # (measured on a 16-core host, byte-exact: 8 / 12 / 24 / 32 / 48 provers -> 11 / 15.0 / 19.6 / 20.1 / 21.4 proofs/s: a lane
    # waits for its next RNG stream -- 0.75 s however many lanes share the SIMD registers -- unless its turn on the GPU takes
    # longer than that; at 48 the byte-exact rate reaches the fast-blinding rate, i.e. the GPU is the limit)
    P = args.provers if args.provers > 0 else 48
    blocking = P * world > cores
    ctx0 = bpg.Context(local)
    ctx0.lib.bpg_set_blocking_sync(1 if blocking else 0)
    ctx0.gens_ensure(GENS_CAP)
    t0 = time.perf_counter()
    # lane 0 of rank 0 proves the reference's own test instance (every leaf = W1, root pinned by merkle_tree_gadget.rs:476);
    # every other lane / rank has its own random leaves
    insts = gadgets.merkle_tree_instances(NLEAVES, [None if (rank == 0 and k == 0) else 7 + 1000 * rank + k for k in range(P)], ctx=ctx0)
    setup_s = {"instances_s": time.perf_counter() - t0}
    t0 = time.perf_counter()
    lanes = LaneSet(bpg, gadgets, local, insts, GENS_CAP, rank)
    setup_s["lanes_s"] = time.perf_counter() - t0
    try:
        used = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=memory.used", "--format=csv,noheader,nounits"], capture_output=True,
                              text=True, timeout=10).stdout.strip()
        setup_s["hbm_used_mib"] = float(used)
    except Exception:
        pass
    ctx, circ, inst, n = lanes.lanes[0].ctx, lanes.lanes[0].circ, insts[0], insts[0]["n"]
    RES = bpg._lib.FLAG_WITNESS_ON_DEVICE
    FAST = bpg._lib.FLAG_FAST_BLINDING

    ext0 = bytes(32)
    proof0, V0 = circ.prove(inst, ext0)  # also the proof the oracle must reproduce (cpu_baseline leg)
    if not circ.verify(inst["label"], V0, proof0):
        raise SystemExit("self-check failed: the verifier rejected the benchmark proof")
    if (proof0, V0) != lanes.lanes[0].prove(ext0, RES, True):
        raise SystemExit("self-check failed: resident-witness proof differs from the host-buffer proof")

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # started before the warm-up: the first nvidia-smi invocations (cold NVML start) are slow
    lanes.timed(RES, True, args.warmup)  # W untimed steps in exactly the shape of the timed region
    sampler.samples.clear()
    ctx.prof_enable(True)
    barrier_max(dist, local, 0.0)
    ms_value, launches = lanes.timed(RES, True, args.steps)
    last_step = lanes.last
    ms_value = barrier_max(dist, local, ms_value)
    cpu_ms_value = lanes.host_cpu_ms
    nl_c, kms_c, pairs_c = ctx.prof_read()   # lane 0's launches inside the timed region: they share the GPU with the other lanes
    ctx.prof_enable(False)
    barrier_max(dist, local, 0.0)
    ms_e2e, _ = lanes.timed(0, False, args.steps)
    ms_e2e = barrier_max(dist, local, ms_e2e)
    ms_fast = None
    if not args.no_extras:
        barrier_max(dist, local, 0.0)
        ms_fast, _ = lanes.timed(RES | FAST, True, max(1, args.steps // 2))
        ms_fast = barrier_max(dist, local, ms_fast) / max(1, args.steps // 2) * args.steps
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=10)
    ctx0.lib.bpg_set_blocking_sync(0)
    # the dominant kernel timed alone (one prover, nothing else on the GPU): this is the figure the roofline fraction is quoted on
    barrier_max(dist, local, 0.0)
    ctx.prof_enable(True)
    ctx.event_record(4)
    lanes.lanes[0].prove(ext0, RES | FAST, True)  # device-side blinding: no host RNG gap inside the events
    ctx.event_record(5)
    solo_ms = ctx.event_elapsed_ms(4, 5)
    per_launch = ctx.prof_read_launches()
    ctx.prof_enable(False)
    big_cut = 0.25 * max([p for _, p in per_launch] or [0])
    big = [(m, p) for m, p in per_launch if p >= big_cut]
    small = [(m, p) for m, p in per_launch if p < big_cut]
    nl, kms, pairs = len(big), sum(m for m, _ in big), sum(p for _, p in big)
    small_launches = {"launches": len(small), "avg_launch_ms": (sum(m for m, _ in small) / len(small)) if small else None,
                      "pairs_per_launch": (sum(p for _, p in small) / len(small)) if small else None,
                      "share_of_kernel_time": (sum(m for m, _ in small) / max(sum(m for m, _ in per_launch), 1e-12)) if per_launch else None}
    nproofs = world * P * args.steps

    extras = {}
    if rank == 0 and not args.no_extras:
        t0 = time.perf_counter()
        lanes.lanes[0].prove(ext0, RES, True)
        extras["single_proof_latency_ms"] = 1e3 * (time.perf_counter() - t0)
        extras["single_proof_latency_ms_fast_blinding"] = solo_ms
        t0 = time.perf_counter()
        for _ in range(3):
            circ.verify(inst["label"], V0, proof0)
        extras["verify_ms"] = 1e3 * (time.perf_counter() - t0) / 3
        extras["single_warp_latency_cycles"] = ctx.bench_latency(200)
        # MiMC (a10 / a11): independent Merkle nodes (2-block sponges), digests only and with the in-circuit witness trace.
        # Kernel time from CUDA events recorded by the library around k_mimc_sponge; 972 mod-l multiplications per block =
        # 1.32e5 MAC32 (SURVEY 8d), trace mode writes 93 312 B per block.
        mac_per_block, trace_bytes = 972 * 136.0, 972 * 96.0
        ms_i0, mac0 = ctx.bench_imad(400)
        peak_mac = mac0 / ms_i0 * 1e3
        hbm_pk = 6543.1
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_pk = json.load(f).get("hbm_gbs", hbm_pk)
        except Exception:
            pass
        mim = {}
        for nh, tr in ((1 << 17, False), (1 << 13, True)):
            leaves = [[os.urandom(32), os.urandom(32)] for _ in range(nh)]
            ctx.mimc_sponge_batch(leaves[:256], trace=tr)
            t0 = time.perf_counter()
            ctx.mimc_sponge_batch(leaves, trace=tr)
            dt = time.perf_counter() - t0
            mk_ms = ctx.event_elapsed_ms(14, 15)
            blocks = 2 * nh
            e = {"merkle_nodes": nh, "kernel_ms": mk_ms, "blocks_per_sec_kernel": blocks / (mk_ms * 1e-3), "nodes_per_sec_e2e": nh / dt,
                 "mac32_per_sec": blocks * mac_per_block / (mk_ms * 1e-3), "int_frac": blocks * mac_per_block / (mk_ms * 1e-3) / peak_mac}
            if tr:
                e["hbm_write_gbs"] = blocks * trace_bytes / (mk_ms * 1e-3) / 1e9
                e["hbm_frac"] = e["hbm_write_gbs"] / hbm_pk
            mim["trace" if tr else "digest"] = e
        mim["note"] = "one thread per sponge (the rounds of one sponge are sequential); int_frac against the measured dependent fe_mul chain rate"
        extras["mimc"] = mim
        extras["fold_points"] = fold_sweep(ctx, [1 << 12] if args.quick else [1 << 12, 1 << 16, 1 << 18], peak_mac)
        sizes = [1 << k for k in range(16, 17 + 1)] if args.quick else [1 << k for k in range(16, 22 + 1)]
        if not args.quick:
            ctx.gens_ensure(1 << 21)
        cpu_sizes = (1 << 16,) if args.quick or args.no_cpu else (1 << 16, 1 << 18, 1 << 20, 1 << 22)
        if args.no_cpu:
            cpu_sizes = ()
        extras["msm"] = msm_sweep(ctx, sizes, cpu_sizes=cpu_sizes, cores=cores)
        extras["msm_bits"] = msm_sweep(ctx, sizes, dist="bits", cpu_sizes=cpu_sizes[:2], cores=cores)
        vs = [1 << 10, 1 << 12] if args.quick else [1 << 10, 1 << 12, 1 << 14, 1 << 16, 1 << 18, 1 << 20, 1 << 22]
        extras["msm_var"] = msm_var_sweep(ctx, vs, cpu_sizes=() if args.no_cpu else ((1 << 12,) if args.quick else (1 << 16, 1 << 20)), cores=cores)

    if world > 1 and not args.no_extras:
        extras["msm_sharded"] = msm_sharded_sweep(ctx, dist, local, rank, world, [1 << 20] if args.quick else [1 << 20, 1 << 22])
    if not args.no_extras and not args.quick:
        # every rank must hold the SAME instance here (the lanes' witnesses differ per rank): the reference's test instance
        shared = inst if rank == 0 else gadgets.merkle_tree_instances(NLEAVES, [None], ctx=ctx0)[0]
        extras["one_proof_2p20"] = one_large_proof(bpg, gadgets, ctx, shared, dist, local, rank, world)
        del shared

    # the full-size oracle proof beside the GPU's (rank 0, N = 1 only): ~20 s on 16 cores + BulletproofGens::new
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        import oracle_lib as ol
        ol.lib().bpo_set_threads(cores)
        t0 = time.perf_counter()
        ol.gens(0, GENS_CAP)
        t_gens = time.perf_counter() - t0
        t_cpu, proof_cpu, V_cpu = oracle_prove(inst, GENS_CAP, ext0, cores)
        cpu = {"value": 1.0 / t_cpu, "unit": "proofs/s", "cores": cores, "kind": "port",
               "sample": "1 complete proof of the same 993 384-multiplier circuit (the reference's test instance) on all host cores (oracle/bpo.c, OpenMP), %.1f s; "
                         "BulletproofGens::new(2^20) beside it: %.1f s" % (t_cpu, t_gens),
               "proof_bytes_equal_gpu": (proof_cpu, V_cpu) == (proof0, V0)}
        if not args.quick:
            # what the reference binary does today: one thread -- on a 1/16-size circuit of the same family, scaled
            small = gadgets.merkle_tree_instances(REF_SAMPLE_LEAVES, [None], trace_on_device=False)[0]
            t_one, _, _ = oracle_prove(small, 1 << 16, ext0, 1)
            cpu["single_thread_value"] = 1.0 / (t_one * N_MULT / small["n"])
            cpu["single_thread_sample"] = "1 thread, %d-multiplier circuit, %.1f s, scaled by the multiplier count" % (small["n"], t_one)

    lanes.close()  # free the 2^20 workspaces before the small-circuit extras

    if not args.no_extras and not args.quick:
        extras["batch_verify_8192"] = batch_verify_config5(bpg, ctx0, dist, local, rank, world, args.cfg5, cores)
    if rank == 0 and not args.no_extras and not args.quick:
        extras["config1_merkle_depth32"] = config1_throughput(bpg, gadgets, local, ctx0, cores, args)

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_ach = (pairs * 100.0) / (kms * 1e-3) / 1e9 if kms > 0 else None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_accumulate_traffic.json")) as f:
                tj = json.load(f)
            traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) / tj["pairs_in_that_launch"] * (pairs / nl if nl else 0)
        except Exception:
            pass
        # integer view: one mixed addition = 7 field multiplications = 504 32x32->64 multiply-accumulates;
        # peak = the MAC32 rate a dependent fe_mul chain sustains at full occupancy on this GPU (bpg_bench_imad, measured here)
        ms_i, mac = ctx0.bench_imad(400)
        imad_peak = mac / ms_i * 1e3
        imad_ach = pairs * 504.0 / (kms * 1e-3) if kms > 0 else None
        line = {"metric": "r1cs_proofs_per_sec", "value": nproofs / (ms_value * 1e-3), "unit": "proofs/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": config_dict(),
                "run": {"proofs_per_step_per_gpu": P, "constraints": int(len(inst["csr"][0]) - 1),
                        "concurrency": "%d independent provers per GPU (own host thread, bpg_ctx and witness each); a step is one proof per prover; "
                                       "every proof has its own ext_rng32" % P,
                        "l2": "window tables (3.2 GB at 2^20 capacity, one set per GPU shared by all provers) exceed the 126 MB L2",
                        "setup_s": setup_s},
                "e2e": {"value": nproofs / (ms_e2e * 1e-3), "unit": "proofs/s", "h2d_bytes_per_step": P * (3 * 32 * n + 2 * 32 * inst["m"] + 128 * n),
                        "d2h_bytes_per_step": P * (len(proof0) + 32 * inst["m"])},
                "gpu_launches": int(launches),
                "proofs_per_sec_fast_blinding": (nproofs / (ms_fast * 1e-3)) if ms_fast else None,
                "host_cores": cores, "host_cpu_ms_per_proof": cpu_ms_value,
                "roofline": {"bound": "integer-multiply pipe (IMAD.WIDE); the contract's hbm view is listed as hbm_*", "kernel": "k_msm_accumulate",
                             "achieved": imad_ach / 1e12 if imad_ach else None, "peak": imad_peak / 1e12, "unit": "TMAC32/s",
                             "frac": (imad_ach / imad_peak) if imad_ach else None, "int_frac": (imad_ach / imad_peak) if imad_ach else None,
                             "peak_note": "measured here: dependent field-multiply chain at full occupancy (bpg_bench_imad); 504 MAC32 per mixed addition",
                             "hbm_achieved": hbm_ach, "hbm_peak": hbm_peak, "hbm_unit": "GB/s", "hbm_frac": (hbm_ach / hbm_peak) if hbm_ach else None,
                             "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                             "traffic": traffic, "launches": int(nl),
                             "algorithmic_bytes_per_launch": (pairs / nl * 100.0) if nl else None,
                             "avg_launch_ms": kms / nl if nl else None, "pairs_per_launch": pairs / nl if nl else None,
                             "note": "CUDA events on the library's stream around every full-size launch (>= 25 % of the largest pair count) of one proof run alone after the timed region",
                             "small_launches": small_launches,
                             "share_of_step": (sum(m for m, _ in per_launch) / solo_ms) if solo_ms > 0 else None,
                             "share_note": "all k_msm_accumulate launches / device time of the same solo proof (compare profiles/r02_launch_summary_2p20.txt)",
                             "in_timed_region": {"launches": int(nl_c), "avg_launch_ms": kms_c / nl_c if nl_c else None,
                                                 "note": "lane 0's launches while %d other provers share the GPU: the kernel runs on a lowest-priority stream, so this "
                                                         "interval includes the time its blocks wait for slots behind every other prover's kernels" % (P - 1)}},
                "cpu_baseline": cpu, "clocks": sampler.summary()}
        line.update(extras)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
        _emit(json.dumps(line))
    ctx0.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def config1_throughput(bpg, gadgets, local, ctx0, cores, args):
    """BASELINE configs[1] (round 1's headline): Merkle membership, depth 32, n = 63 180, N = 2^16, byte-exact, many provers"""
    P = 64
    ctx0.lib.bpg_set_blocking_sync(1 if P > cores else 0)
    inst = gadgets.merkle_path_instance(32, seed=4, ctx=ctx0)
    lanes = LaneSet(bpg, gadgets, local, [dict(inst) for _ in range(P)], 1 << 16, 0)
    RES = bpg._lib.FLAG_WITNESS_ON_DEVICE
    lanes.timed(RES, True, 4)
    ms, launches = lanes.timed(RES, True, 6)
    res = {"workload": "merkle_tree membership with mimc_hash, depth 32, single proof", "n_multipliers": inst["n"], "provers": P,
           "proofs_per_sec": P * 6 / (ms * 1e-3), "launches_per_proof": launches / (P * 6), "host_cpu_ms_per_proof": lanes.host_cpu_ms}
    if not args.no_cpu:
        t_cpu, proof_cpu, V_cpu = oracle_prove(dict(inst), 1 << 16, bytes(32), cores)
        res["cpu_proofs_per_sec"] = 1.0 / t_cpu
        res["cpu_cores"] = cores
        res["proof_bytes_equal_oracle"] = (proof_cpu, V_cpu) == lanes.lanes[0].circ.prove(inst, bytes(32))
    lanes.close()
    ctx0.lib.bpg_set_blocking_sync(0)
    return res


def main():
    # stdout carries exactly ONE JSON line: everything else that libraries print there (e.g. NCCL's version banner) goes to stderr
    saved = os.dup(1)
    os.dup2(2, 1)
    global _emit
    def _emit(text):
        os.write(saved, (text + "\n").encode())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--provers", type=int, default=0, help="concurrent provers (host threads / contexts) per GPU; 0 = auto")
    ap.add_argument("--cfg5", type=int, default=8192, help="proofs in the batch-verification extra (BASELINE configs[4])")
    ap.add_argument("--quick", action="store_true", help="small MSM sweep only, no config extras")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed region's last-step outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
