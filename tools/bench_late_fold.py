"""Load sweep of the late-fold point (kernels_msm.cuh, prover.inl): for each BPG_LATE_FOLD_LG value, n' = 2^value folded
generators per vector, one subprocess each (the library reads the variable once per process):
  - bench.py's flagship workload (993 384 multipliers, N = 2^20, 48 provers with prefetch, byte-exact): proofs/s and the solo
    proof's k_msm_accumulate launch list (bpg_prof_* events: full-size launches and their pairs);
  - one solo fast-blinding proof of the same circuit under torch.profiler: device time per kernel, the late-fold kernels and
    k_msm_accumulate broken out.
Writes profiles/r07_late_fold.json (or --out).  Usage:  python tools/bench_late_fold.py --lg 13 14 15 16 --steps 20 --warmup 5"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOLD_KERNELS = ("k_mat_block", "k_mat_reduce", "k_mat_chain", "k_mat_affine", "k_msm_finish", "k_msm_heavy")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                       timeout=30).stdout.strip()
    return q


def solo():
    """child: one warm solo proof, then one profiled proof; prints a JSON line of per-kernel device time"""
    sys.path.insert(0, ROOT)
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bulletproofs_gadgets_b200 as bpg
    from bulletproofs_gadgets_b200 import gadgets
    torch.cuda.init()
    ctx = bpg.Context(0)
    ctx.gens_ensure(1 << 20)
    inst = gadgets.merkle_tree_instances(512, [None], ctx=ctx)[0]
    circ = gadgets.Circuit(ctx, inst["n"], inst["m"], inst["csr"])
    FAST = bpg._lib.FLAG_FAST_BLINDING
    ext = b"\x11" * 32
    circ.prove(inst, ext, FAST)  # warm-up: buffers, late-fold tables
    ctx.prof_enable(True)
    circ.prove(inst, ext, FAST)
    launches = ctx.prof_read_launches()
    ctx.prof_enable(False)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        circ.prove(inst, ext, FAST)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name.split("(")[0].replace("void ", "").split("<")[0].strip()
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        d = per.setdefault(name, [0, 0.0])
        d[0] += 1
        d[1] += t / 1e3
    big_cut = 0.25 * max([p for _, p in launches] or [0])
    full = [(m, p) for m, p in launches if p >= big_cut]
    acc_ms = per.get("k_msm_accumulate", [0, 0.0])[1]
    fold = {k: per[k][1] for k in FOLD_KERNELS if k in per}
    print(json.dumps({"device_ms_total": sum(v[1] for v in per.values()), "kernels_ms": {k: round(v[1], 4) for k, v in sorted(per.items(), key=lambda x: -x[1][1])},
                      "launches": {k: v[0] for k, v in per.items()}, "k_msm_accumulate_ms": acc_ms, "fold_kernels_ms": fold,
                      "accumulate_launches_full_size": len(full), "accumulate_pairs_full_size": [int(p) for _, p in full],
                      "accumulate_pairs_total": int(sum(p for _, p in launches))}))
    circ.close()
    ctx.close()


def run(lg, args):
    env = dict(os.environ)
    if lg:
        env["BPG_LATE_FOLD_LG"] = str(lg)
    rec = {"late_lg": lg or "default"}
    t0 = time.time()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup),
                          "--no-extras", "--no-cpu"], env=env, capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode or not lines:
        rec["bench_error"] = out.stderr[-2000:]
    else:
        b = json.loads(lines[-1])
        rf = b.get("roofline", {})
        rec["proofs_per_sec"] = b["value"]
        rec["e2e"] = b["e2e"]["value"]
        rec["solo_full_size_accumulate_launches"] = rf.get("launches")
        rec["solo_pairs_per_full_size_launch"] = rf.get("pairs_per_launch")
        rec["hbm_used_mib_before_first_proof"] = b["run"]["setup_s"].get("hbm_used_mib")
    rec["bench_wall_s"] = time.time() - t0
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--solo"], env=env, capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    rec["solo"] = json.loads(lines[-1]) if lines and not out.returncode else {"error": out.stderr[-2000:]}
    print(json.dumps({k: v for k, v in rec.items() if k != "solo"}), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lg", type=int, nargs="+", default=[13, 14, 15, 16], help="BPG_LATE_FOLD_LG values (0 = the library's default)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_late_fold.json"))
    ap.add_argument("--solo", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.solo:
        return solo()
    res = {"card": card(), "workload": "bench.py --gpus 1 --steps %d --warmup %d --no-extras --no-cpu (N = 2^20, 48 provers, byte-exact)" % (args.steps, args.warmup),
           "sweep": [run(lg, args) for lg in args.lg]}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
