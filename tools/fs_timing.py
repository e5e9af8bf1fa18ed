"""Timing of the statement-bound Fiat-Shamir proof against vp_prove and against the host-loop vp_prove_fs of another build.

  python tools/fs_timing.py --parent-lib DIR/libvirgo_b200.so [--reps N] [--blocks B] [--out FILE]
  (DIR also holds that build's binding.py, e.g. `git worktree add DIR/src <commit> && make -C DIR/src/virgo-plus_b200`, then
  copy libvirgo_b200.so and binding.py from there to DIR.)

For C1 (one SHA256_64 proof) and C3 (SHA256_64 x 1024), medians of warm calls (host clock around calls that end in a
stream synchronisation) of:
  vp_prove (device-resident inputs and challenges), vp_prove_fs_bound, vp_statement_digest alone, and vp_prove_fs(statement)
  of the library at --parent-lib (loaded through VP_LIB in a separate process; blocks of the two alternate).
Both libraries get the same statement as the seed; the SHA-256 of both transcripts is recorded and the script fails if they
differ. Also the per-round split of the bound proof from block 0's %globaltimer stamps (vp_fs_round_stamps): own fold
work, barrier + reduce, draw, release barrier. The card's name and power limit are read in the same run."""
import argparse
import hashlib
import json
import lzma
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def circuit(B, case):
    with lzma.open(os.path.join(ROOT, "tests", "golden", "SHA256_64.pws.xz"), "rb") as f:
        c = B.Circuit.from_pws_text(f.read())
    return c if case == "C1" else c.replicate(1024)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def worker(case, statement_hex, reps, warm, parent_lib):
    """runs in a process with VP_LIB set: vp_prove_fs(statement) of that library, through the binding.py kept beside it
    (the other build's own ctypes declarations)"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("vp_binding_other", os.path.join(os.path.dirname(os.path.abspath(parent_lib)), "binding.py"))
    B = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(B)
    circ = circuit(B, case)
    p = B.Prover(circ)
    st = bytes.fromhex(statement_hex)
    for _ in range(warm):
        tr, _ = p.prove_fs(st)
    ms = timed(lambda: p.prove_fs(st), reps)
    tr, _ = p.prove_fs(st)
    p.close()
    print(json.dumps(dict(ms=ms, transcript_sha256=hashlib.sha256(tr.tobytes()).hexdigest(), lib=B.LIB_PATH)))


def split(stamps, circ):
    """per-round phases (ns) from the stamps; the release barrier only inside a phase"""
    s = stamps.astype(np.int64)
    fold, reduce_, draw = s[:, 1] - s[:, 0], s[:, 2] - s[:, 1], s[:, 3] - s[:, 2]
    n = circ.n_layers
    rel, r = [], 0
    for i in range(n - 1, 0, -1):
        for cnt in (circ.bit_length(i - 1), max(circ.max_dad_bit_length(i), 0), circ.bit_length(i - 1)):
            for j in range(1, cnt):
                rel.append(s[r + j, 0] - s[r + j - 1, 3])
            r += cnt
    assert r == len(s)
    rel = np.array(rel or [0])
    tot = lambda a: float(a.sum()) / 1e6
    return dict(rounds=int(len(s)), fold_ms=tot(fold), barrier_reduce_ms=tot(reduce_), draw_ms=tot(draw), release_ms=tot(rel),
                draw_us_median=float(np.median(draw)) / 1e3, fold_us_median=float(np.median(fold)) / 1e3,
                barrier_reduce_us_median=float(np.median(reduce_)) / 1e3, release_us_median=float(np.median(rel)) / 1e3,
                first_to_last_ms=float(s[-1, 3] - s[0, 0]) / 1e6)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--warm", type=int, default=3)
    ap.add_argument("--cases", default="C1,C3")
    ap.add_argument("--out", help="also write the results (medians, raw samples, round split) to this JSON file")
    ap.add_argument("--worker", nargs=2, metavar=("CASE", "STATEMENT"))
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker[0], a.worker[1], a.reps, a.warm, a.parent_lib)
    if not os.path.exists(a.parent_lib):
        sys.exit(f"{a.parent_lib}: no such library")
    import __graft_entry__ as E
    B = E.binding()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    ctx = bytes(range(100, 132))
    res = dict(gpu=smi[0] if smi else "unknown", context_hex=ctx.hex(), reps_per_block=a.reps, blocks=a.blocks, cases={})
    for case in a.cases.split(","):
        circ = circuit(B, case)
        p = B.Prover(circ)
        p.set_challenges(circ.draw_challenges())
        tr, ch, st = p.prove_fs_bound(ctx)
        for _ in range(a.warm):
            p.prove()
            p.prove_fs_bound(ctx)
            p.statement_digest(ctx)
        new_sha = hashlib.sha256(tr.tobytes()).hexdigest()
        t = dict(vp_prove=[], prove_fs_bound=[], statement_digest=[], parent_prove_fs=[])
        parent_sha = None
        for b in range(a.blocks):
            p.set_challenges(circ.draw_challenges())
            t["vp_prove"] += timed(lambda: p.prove(), a.reps)
            t["prove_fs_bound"] += timed(lambda: p.prove_fs_bound(ctx), a.reps)
            t["statement_digest"] += timed(lambda: p.statement_digest(ctx), a.reps)
            env = dict(os.environ, VP_LIB=os.path.abspath(a.parent_lib))
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--parent-lib", a.parent_lib, "--reps", str(a.reps), "--warm",
                                  str(a.warm if b == 0 else 1), "--worker", case, st.hex()], env=env, capture_output=True, text=True)
            if out.returncode != 0:
                sys.exit(f"parent worker failed:\n{out.stderr[-3000:]}")
            w = json.loads(out.stdout.strip().splitlines()[-1])
            t["parent_prove_fs"] += w["ms"]
            parent_sha = w["transcript_sha256"]
            if parent_sha != new_sha:
                sys.exit(f"{case}: transcript of the parent's vp_prove_fs(statement) {parent_sha} != vp_prove_fs_bound {new_sha}")
        p.prove_fs_bound(ctx)
        sp = split(p.fs_round_stamps(), circ)
        med = {k: float(np.median(v)) for k, v in t.items()}
        res["cases"][case] = dict(instances=int(circ.instances), layers=circ.n_layers, median_ms=med, samples=len(t["vp_prove"]),
                                  device_ms_last_bound=p.last_prove_ms, launches_bound=p.last_prove_launches, round_split=sp,
                                  statement_hex=st.hex(), transcript_sha256=new_sha, parent_transcript_sha256=parent_sha, raw_ms=t)
        p.close()
        print(f"{case}: median ms  vp_prove {med['vp_prove']:.3f}  prove_fs_bound {med['prove_fs_bound']:.3f}  "
              f"(statement digest {med['statement_digest']:.3f})  parent vp_prove_fs {med['parent_prove_fs']:.3f}  | rounds {sp['rounds']}: "
              f"fold {sp['fold_ms']:.3f} ms, barrier+reduce {sp['barrier_reduce_ms']:.3f} ms, draw {sp['draw_ms']:.3f} ms "
              f"({sp['draw_us_median']:.2f} us median), release {sp['release_ms']:.3f} ms; transcripts equal ({new_sha[:16]})", flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(f"gpu: {res['gpu']}")


if __name__ == "__main__":
    main()
