"""Statement-bound batches from device memory (vp_*_fs_bound_batch_dev, torch CUDA tensors) against the same batches from
host memory (vp_prove_fs_bound_batch, vp_verify_fs_bound_batch), on the same statements, alternating in one run.

  python tools/fs_device_batch_timing.py [--reps N] [--warm W] [--cases SPEC] [--out FILE]

Workloads: C1 (one SHA256_64 per statement) and SHA256_64 x 16 per statement, B in {8, 32, 148, 512}. Per call kind,
medians of `reps` warm calls of:
  host     one host-memory call (host clock; the call ends in a stream synchronisation), and its device window
           (vp_last_prove_ms); for verify, host - device is the host part: everything the call does outside its device
           window -- the binding's array conversions, the library's argument checks and canonical scans, the read-back
           and the round checks of every statement (Engine::verify_check) -- so an upper bound on verify_check alone,
           which the device call replaces;
  device   one device-memory call plus a synchronisation of the current stream (host clock), the time the call takes to
           return (enqueue only), and its device time (vp_last_prove_ms: the whole call, screening and, for verify, the
           claim chain k_verify_check included);
  kernels  for verify, the device time of k_verify_check (the claim chain of all B statements, which replaces the host
           checks) and of k_batch_screen, from torch.profiler in one extra device call after the timed ones.
The inputs and contexts are already on the device for the device calls and on the host for the host calls (that is
what each serves). Every device result must equal the host call's (transcripts, challenges, statements, outputs; every
verdict an accept). The card's name and power limit are read in the same run; JSON only with --out."""
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

from fs_batch_timing import inputs_for, sha256_64  # noqa: E402


def fe_tensor(torch, a):
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.view(np.int64).reshape(a.shape + (2,)).copy()).cuda()


def fe_array(t):
    a = np.ascontiguousarray(t.cpu().numpy())
    return a.view(np.dtype([("re", "<u8"), ("im", "<u8")])).reshape(a.shape[:-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--cases", default="C1:8,32,148,512;SHA256_64x16:8,32,148,512")
    ap.add_argument("--out", help="also write the results to this JSON file")
    a = ap.parse_args()
    import torch

    import __graft_entry__ as E
    B = E.binding()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = dict(gpu=smi[0] if smi else "unknown", reps=a.reps, warm=a.warm, cases={})
    print(f"gpu: {res['gpu']}", flush=True)
    stream = torch.cuda.current_stream()
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
            xd = torch.from_numpy(np.ascontiguousarray(x).view(np.int64).copy()).cuda()
            cd = torch.from_numpy(np.frombuffer(b"".join(ctxs), np.uint8).reshape(n, 32).copy()).cuda()
            want = p.prove_fs_bound_batch(x, ctxs, return_outputs=True)
            outd, trd = fe_tensor(torch, want[3]), fe_tensor(torch, want[0])
            # the results must agree before anything is timed
            tr, ch, st, out, status = p.prove_fs_bound_batch_cuda(xd, cd, challenges=True, outputs=True)
            acc, code, _, _ = p.verify_fs_bound_batch_cuda(xd, cd, outd, trd)
            stream.synchronize()
            if status.cpu().any() or not (fe_array(tr) == want[0]).all() or not (fe_array(ch) == want[1]).all() \
                    or not (st.cpu().numpy() == want[2]).all() or not (fe_array(out) == want[3]).all():
                sys.exit(f"{name} B={n}: the device batch differs from the host batch")
            if not acc.cpu().all() or code.cpu().any() or not p.verify_fs_bound_batch(x, ctxs, want[3], want[0])[0].all():
                sys.exit(f"{name} B={n}: a proof was rejected")
            calls = dict(
                prove_host=lambda: p.prove_fs_bound_batch(x, ctxs),
                prove_device=lambda: p.prove_fs_bound_batch_cuda(xd, cd),
                verify_host=lambda: p.verify_fs_bound_batch(x, ctxs, want[3], want[0]),
                verify_device=lambda: p.verify_fs_bound_batch_cuda(xd, cd, outd, trd),
            )
            raw = {k: dict(total=[], enqueue=[], device=[]) for k in calls}
            for it in range(a.warm + a.reps):
                for k, fn in calls.items():   # alternating: host and device calls of both kinds in every repetition
                    stream.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    t1 = time.perf_counter()
                    stream.synchronize()
                    t2 = time.perf_counter()
                    dev = p.last_prove_ms
                    launches = p.last_prove_launches
                    if it >= a.warm:
                        raw[k]["total"].append((t2 - t0) * 1e3)
                        raw[k]["enqueue"].append((t1 - t0) * 1e3)
                        raw[k]["device"].append(dev)
                        raw[k]["launches"] = launches
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                calls["verify_device"]()
                stream.synchronize()
            kern = {}
            for ev in prof.key_averages():
                for kname in ("k_verify_check", "k_batch_screen"):
                    if kname in ev.key:
                        us = getattr(ev, "device_time_total", None)
                        kern[kname] = kern.get(kname, 0.0) + (us if us is not None else ev.cuda_time_total) / 1e3
            med = {k: {m: float(np.median(v[m])) for m in ("total", "enqueue", "device")} | dict(launches=v["launches"])
                   for k, v in raw.items()}
            row = dict(B=n, median_ms=med, verify_kernel_ms=kern, raw_ms=raw)
            case["rows"].append(row)
            for kind in ("prove", "verify"):
                h, d = med[f"{kind}_host"], med[f"{kind}_device"]
                extra = ""
                if kind == "verify":
                    extra = (f"; host part of the host call {h['total'] - h['device']:7.2f} ms vs k_verify_check "
                             f"{kern.get('k_verify_check', float('nan')):6.3f} ms (k_batch_screen "
                             f"{kern.get('k_batch_screen', float('nan')):6.3f} ms)")
                print(f"{name} B={n:4d} {kind:6s}: host memory {h['total']:8.2f} ms (device {h['device']:8.2f} ms, "
                      f"{h['launches']} launches) | device memory {d['total']:8.2f} ms (returns after {d['enqueue']:6.2f} ms, "
                      f"device {d['device']:8.2f} ms, {d['launches']} launches){extra}", flush=True)
        p.close()
        res["cases"][name] = case
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
