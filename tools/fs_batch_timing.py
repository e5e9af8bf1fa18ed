"""Throughput of batched statement-bound proofs (vp_prove_fs_bound_batch) against one proof per call.

  python tools/fs_batch_timing.py [--reps N] [--warm W] [--out FILE]

Workloads: C1 (one SHA256_64 per statement) with B in {1, 8, 32, 148, 512}, and SHA256_64 x 16 per statement with B in
{1, 8, 32}. For each B, medians of warm calls (host clock around calls that end in a stream synchronisation) of:
  batch      one vp_prove_fs_bound_batch call over B statements (distinct inputs and contexts);
  singles    B vp_prove_fs_bound calls, one after another, on the same inputs and contexts (vp_set_inputs before each);
  aggregate  one vp_prove_fs_bound on replicate(template, B): one proof over all B statements' instances, for context.
Checks that every batch proof equals its single proof (SHA-256 of all transcripts). Also block 0's per-round stamps of
statement 0 for the batch (vp_fs_round_stamps). The card's name and power limit are read in the same run; JSON only with
--out."""
import argparse
import hashlib
import json
import lzma
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fs_timing import split  # noqa: E402


def sha256_64(B):
    with lzma.open(os.path.join(ROOT, "tests", "golden", "SHA256_64.pws.xz"), "rb") as f:
        return B.Circuit.from_pws_text(f.read())


def inputs_for(circ, n, seed):
    """n distinct input vectors: the circuit's own inputs with a few bits flipped (0/1 inputs stay 0/1)"""
    base = np.asarray(circ.inputs(), dtype=np.uint64)
    rng = np.random.default_rng(seed)
    out = np.repeat(base[None, :], n, axis=0)
    for b in range(n):
        for i in rng.choice(len(base), size=min(8, len(base)), replace=False):
            x = int(out[b, i])
            out[b, i] = 1 - x if x in (0, 1) else int(rng.integers(0, (1 << 61) - 1))
    return out


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()   # every call below ends in a stream synchronisation
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--cases", default="C1:1,8,32,148,512;SHA256_64x16:1,8,32")
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
        rows = []
        p = B.Prover(circ)
        for n in (int(x) for x in sizes.split(",")):
            x = inputs_for(circ, n, n)
            rng = random.Random(n)
            ctxs = [bytes(rng.randrange(256) for _ in range(32)) for _ in range(n)]
            for _ in range(a.warm):
                tr, _, _ = p.prove_fs_bound_batch(x, ctxs)
            batch_ms = timed(lambda: p.prove_fs_bound_batch(x, ctxs), a.reps)
            launches, device_ms = p.last_prove_launches, p.last_prove_ms
            sp = split(p.fs_round_stamps(), circ)

            singles_tr = []

            def singles():
                singles_tr.clear()
                for b in range(n):
                    p.set_inputs(x[b])
                    singles_tr.append(p.prove_fs_bound(ctxs[b])[0])
            singles()
            single_ms = timed(singles, max(1, a.reps if n <= 32 else 2))
            same = hashlib.sha256(tr.tobytes()).hexdigest() == hashlib.sha256(np.stack(singles_tr).tobytes()).hexdigest()
            if not same:
                sys.exit(f"{name} B={n}: batch transcripts differ from the single proofs")
            single_launches = p.last_prove_launches

            agg = tmpl.replicate(K * n) if K * n > 1 else tmpl
            q = B.Prover(agg)
            for _ in range(a.warm):
                q.prove_fs_bound(bytes(32))
            agg_ms = timed(lambda: q.prove_fs_bound(bytes(32)), a.reps)
            q.close()
            med = dict(batch=float(np.median(batch_ms)), singles=float(np.median(single_ms)), aggregate=float(np.median(agg_ms)))
            rows.append(dict(B=n, median_ms=med, per_proof_ms=dict(batch=med["batch"] / n, singles=med["singles"] / n),
                             speedup=med["singles"] / med["batch"], launches_batch=launches, launches_single=single_launches,
                             device_ms_last_batch=device_ms, round_split_statement0=sp,
                             transcripts_sha256=hashlib.sha256(tr.tobytes()).hexdigest(),
                             raw_ms=dict(batch=batch_ms, singles=single_ms, aggregate=agg_ms)))
            print(f"{name} B={n:4d}: batch {med['batch']:9.2f} ms ({med['batch'] / n:7.3f} ms/proof, {launches} launches)  "
                  f"{n} single calls {med['singles']:9.2f} ms ({med['singles'] / n:7.3f} ms/proof)  speedup {med['singles'] / med['batch']:6.2f}x  "
                  f"aggregate proof of {K * n} instances {med['aggregate']:8.2f} ms | statement 0: fold {sp['fold_ms']:.2f} ms, "
                  f"barrier+reduce {sp['barrier_reduce_ms']:.2f} ms, draw {sp['draw_ms']:.2f} ms, release {sp['release_ms']:.2f} ms",
                  flush=True)
        p.close()
        res["cases"][name] = dict(instances_per_statement=K, rows=rows)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
