"""Cost of aggregate statement-bound proofs (vp_prove_fs_aggregate / vp_verify_fs_aggregate) against a batch of B proofs of
the same statements.

  python tools/fs_aggregate_timing.py [--reps N] [--warm W] [--out FILE]

Workloads: C1 (one SHA256_64 per statement) with B in {8, 32, 148, 512, 1024}, and SHA256_64 x 16 per statement with B in
{8, 32}. Statement b is instances [b K, (b + 1) K) of replicate(SHA256_64, B K) (its own inputs, as replication draws them)
with its own context. Medians of warm calls (host clock around calls that end in a stream synchronisation) of:
  agg_prove     one vp_prove_fs_aggregate over the B statements;
  agg_verify    one vp_verify_fs_aggregate of that proof, with the outputs the prover computed;
  agg_digest    one vp_aggregate_digest on the evaluated context (roots, statements, aggregate and their read-back);
  batch_prove   one vp_prove_fs_bound_batch over the same B statements (inputs and contexts) on a K-instance context;
  batch_verify  one vp_verify_fs_bound_batch of those proofs;
  bound         one vp_prove_fs_bound on the B K-instance context with a zero context: one proof over all instances
                with one statement (fs_batch_timing's "aggregate" column), so agg_prove - bound is the cost of the B
                per-statement digests.
Proof bytes: 16 per transcript element (one transcript for the aggregate, B for the batch). Exits non-zero if an aggregate
proof differs from vp_prove_fs(aggregate) or is rejected, or if a batch proof is rejected. The card's name and power limit
are read in the same run; JSON only with --out."""
import argparse
import hashlib
import json
import os
import random
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fs_batch_timing import sha256_64, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--cases", default="C1:8,32,148,512,1024;SHA256_64x16:8,32")
    ap.add_argument("--out", help="also write the results to this JSON file")
    a = ap.parse_args()
    import __graft_entry__ as E
    B = E.binding()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = dict(gpu=smi[0] if smi else "unknown", reps=a.reps, warm=a.warm, cases={})
    print(f"gpu: {res['gpu']}", flush=True)
    tmpl = sha256_64(B)
    for spec in a.cases.split(";"):
        name, sizes = spec.split(":")
        K = 1 if name == "C1" else int(name.split("x")[1])
        stmt_circ = tmpl if K == 1 else tmpl.replicate(K)
        q = B.Prover(stmt_circ)
        rows = []
        for n in (int(x) for x in sizes.split(",")):
            circ = tmpl.replicate(K * n)
            rng = random.Random(n)
            ctxs = [bytes(rng.randrange(256) for _ in range(32)) for _ in range(n)]
            p = B.Prover(circ)
            tr, ch, st, agg = p.prove_fs_aggregate(n, ctxs)   # the call that is checked; also the first warm-up
            for _ in range(a.warm):
                p.prove_fs_aggregate(n, ctxs)
            prove_ms = timed(lambda: p.prove_fs_aggregate(n, ctxs), a.reps)
            launches, device_ms = p.last_prove_launches, p.last_prove_ms
            tr_ref, ch_ref = p.prove_fs(agg)
            if not ((tr == tr_ref).all() and (ch == ch_ref).all()):
                sys.exit(f"{name} B={n}: the aggregate proof differs from vp_prove_fs(aggregate)")
            outputs = p.values(circ.n_layers - 1)
            verdict = p.verify_fs_aggregate(n, ctxs, outputs, tr)
            for _ in range(a.warm):
                p.verify_fs_aggregate(n, ctxs, outputs, tr)
            if verdict != (True, 0, 0):
                sys.exit(f"{name} B={n}: the aggregate proof was rejected: {verdict}")
            verify_ms = timed(lambda: p.verify_fs_aggregate(n, ctxs, outputs, tr), a.reps)
            for _ in range(a.warm):
                p.aggregate_digest(n, ctxs)
            digest_ms = timed(lambda: p.aggregate_digest(n, ctxs), a.reps)
            for _ in range(a.warm):
                p.prove_fs_bound(bytes(32))
            bound_ms = timed(lambda: p.prove_fs_bound(bytes(32)), a.reps)
            x = np.asarray(circ.inputs(), dtype=np.uint64).reshape(n, -1)
            p.close()

            btr, _, _, bout = q.prove_fs_bound_batch(x, ctxs, return_outputs=True)
            for _ in range(a.warm):
                q.prove_fs_bound_batch(x, ctxs)
            bprove_ms = timed(lambda: q.prove_fs_bound_batch(x, ctxs), a.reps)
            acc = q.verify_fs_bound_batch(x, ctxs, bout, btr)[0]
            for _ in range(a.warm):
                q.verify_fs_bound_batch(x, ctxs, bout, btr)
            if not acc.all():
                sys.exit(f"{name} B={n}: the batch rejected statements {np.flatnonzero(~acc)}")
            bverify_ms = timed(lambda: q.verify_fs_bound_batch(x, ctxs, bout, btr), a.reps)

            med = {k: float(np.median(v)) for k, v in (("agg_prove", prove_ms), ("agg_verify", verify_ms), ("agg_digest", digest_ms),
                                                        ("batch_prove", bprove_ms), ("batch_verify", bverify_ms),
                                                        ("bound", bound_ms))}
            proof_bytes = dict(aggregate=16 * circ.transcript_len, batch=16 * btr.size)
            rows.append(dict(B=n, instances=K * n, median_ms=med, proof_bytes=proof_bytes, launches_agg_prove=launches,
                             device_ms_last_agg_prove=device_ms, digest_overhead_ms=med["agg_prove"] - med["bound"],
                             transcript_sha256=hashlib.sha256(tr.tobytes()).hexdigest(), aggregate=agg.hex(),
                             raw_ms=dict(agg_prove=prove_ms, agg_verify=verify_ms, agg_digest=digest_ms, batch_prove=bprove_ms,
                                         batch_verify=bverify_ms, bound=bound_ms)))
            print(f"{name} B={n:5d}: aggregate prove {med['agg_prove']:8.2f} ms ({launches} launches), verify {med['agg_verify']:8.2f} ms, "
                  f"{proof_bytes['aggregate']:8d} B | batch prove {med['batch_prove']:8.2f} ms, verify {med['batch_verify']:8.2f} ms, "
                  f"{proof_bytes['batch']:10d} B | bound proof of {K * n} instances {med['bound']:8.2f} ms "
                  f"(aggregate - bound {med['agg_prove'] - med['bound']:6.2f} ms; vp_aggregate_digest {med['agg_digest']:6.2f} ms)",
                  flush=True)
        q.close()
        res["cases"][name] = dict(instances_per_statement=K, rows=rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
