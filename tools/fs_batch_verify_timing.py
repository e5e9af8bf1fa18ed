"""Cost of checking statement-bound proofs: one vp_verify_fs_bound, and vp_verify_fs_bound_batch against one check per call.

  python tools/fs_batch_verify_timing.py [--reps N] [--warm W] [--out FILE]

Workloads: C1 (one SHA256_64 per statement) and SHA256_64 x 16 per statement, B in {1, 8, 32, 148, 512}. Medians of warm
calls (host clock around calls that end in a stream synchronisation) of:
  single     one vp_verify_fs_bound, split into the host replay of its challenges (vp_fs_challenges on the same statement
             and transcript, the replay it runs) and the rest (statement digests, the device sums, the round checks);
  batch      one vp_verify_fs_bound_batch over B statements (distinct inputs and contexts), split into the device part
             (vp_last_prove_ms: upload, roots, challenge replay, sums) and the host part (the rest of the call: argument
             checks, read-back, the round checks of every statement);
  singles    B vp_verify_fs_bound calls, one after another, on the same proofs (vp_set_inputs before each).
Every proof comes from vp_prove_fs_bound_batch; every verdict must be an accept. The card's name and power limit are read
in the same run; JSON only with --out."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fs_batch_timing import inputs_for, sha256_64, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--cases", default="C1:1,8,32,148,512;SHA256_64x16:1,8,32,148,512")
    ap.add_argument("--out", help="also write the results to this JSON file")
    a = ap.parse_args()
    import __graft_entry__ as E
    B = E.binding()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = dict(gpu=smi[0] if smi else "unknown", reps=a.reps, warm=a.warm, cases={})
    print(f"gpu: {res['gpu']}", flush=True)
    for spec in a.cases.split(";"):
        name, sizes = spec.split(":")
        K = 1 if name == "C1" else int(name.split("x")[1])
        tmpl = sha256_64(B)
        circ = tmpl if K == 1 else tmpl.replicate(K)
        p = B.Prover(circ)
        case = dict(instances_per_statement=K, rows=[])
        for n in (int(x) for x in sizes.split(",")):
            x = inputs_for(circ, n, n)
            rng = random.Random(n)
            ctxs = [bytes(rng.randrange(256) for _ in range(32)) for _ in range(n)]
            tr, _, st, out = p.prove_fs_bound_batch(x, ctxs, return_outputs=True)
            for _ in range(a.warm):
                acc = p.verify_fs_bound_batch(x, ctxs, out, tr)[0]
            if not acc.all():
                sys.exit(f"{name} B={n}: the batch rejected statements {np.flatnonzero(~acc)}")
            batch_ms, device_ms = [], []
            for _ in range(a.reps):
                batch_ms += timed(lambda: p.verify_fs_bound_batch(x, ctxs, out, tr), 1)
                device_ms.append(p.last_prove_ms)
            launches = p.last_prove_launches

            def singles():
                for b in range(n):
                    p.set_inputs(x[b])
                    if not p.verify_fs_bound(ctxs[b], out[b], tr[b])[0]:
                        sys.exit(f"{name} B={n}: statement {b} rejected by vp_verify_fs_bound")
            singles()
            single_ms = timed(singles, max(1, a.reps if n <= 32 else 2))
            med = dict(batch=float(np.median(batch_ms)), singles=float(np.median(single_ms)))
            dev = float(np.median(device_ms))
            row = dict(B=n, median_ms=med, per_proof_ms=dict(batch=med["batch"] / n, singles=med["singles"] / n),
                       speedup=med["singles"] / med["batch"], batch_split_ms=dict(device=dev, host=med["batch"] - dev),
                       launches_batch=launches, raw_ms=dict(batch=batch_ms, device=device_ms, singles=single_ms))
            if n == 1:   # one vp_verify_fs_bound, and its host replay
                p.set_inputs(x[0])
                for _ in range(a.warm):
                    p.verify_fs_bound(ctxs[0], out[0], tr[0])
                one = timed(lambda: p.verify_fs_bound(ctxs[0], out[0], tr[0]), a.reps)
                replay = timed(lambda: circ.fs_challenges(st[0].tobytes(), tr[0]), a.reps)
                one_m, rep_m = float(np.median(one)), float(np.median(replay))
                case["single_verify"] = dict(total_ms=one_m, host_replay_ms=rep_m, rest_ms=one_m - rep_m,
                                             raw_ms=dict(total=one, host_replay=replay))
                print(f"{name}: one vp_verify_fs_bound {one_m:7.2f} ms = host challenge replay {rep_m:6.2f} ms + rest "
                      f"{one_m - rep_m:6.2f} ms", flush=True)
            case["rows"].append(row)
            print(f"{name} B={n:4d}: batch {med['batch']:9.2f} ms ({med['batch'] / n:7.3f} ms/proof, {launches} launches; device "
                  f"{dev:7.2f} ms, host {med['batch'] - dev:7.2f} ms)  {n} single calls {med['singles']:9.2f} ms "
                  f"({med['singles'] / n:7.3f} ms/proof)  speedup {med['singles'] / med['batch']:6.2f}x", flush=True)
        p.close()
        res["cases"][name] = case
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
