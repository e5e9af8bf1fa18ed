#!/usr/bin/env python3
"""bench.py -- GKR prover throughput (gates/s) and sumcheck ms/proof on B200, beside the CPU reference.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, through the C ABI)
      [--dump-outputs DIR]                                 + the transcript of the last timed proof as DIR/transcript.npy
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU prover on the host cores

One step = one complete GKR proof (evaluate + every phase-1 / phase-2 / Liu sumcheck of every layer +
input-layer MLE) of the workload circuit on synthetic inputs:
  N = 1 : BASELINE.json configs[2], SHA256_64 x 1024 data-parallel instances (94.9 M gates).
  N > 1 : weak scaling, 1024 instances per GPU (see DESIGN.md "Multi-GPU").
`value` = gates/s with inputs and challenges resident in HBM; `e2e` = the same through
vp_prove_local (= vp_prove(host_io=1) for the witness slice a rank holds): inputs + challenges copied from pinned
host memory and the transcript copied back inside the timed region. Prints ONE JSON line on rank 0.

Every line carries its own correctness evidence (`parity`): the SHA-256 of the timed transcript, whether all ranks
hold the same one, the device verifier's verdict (vp_verify; collective on a sharded context), the comparison with
the hash the UNMODIFIED reference prover produced for this circuit where tests/golden/full_size.json has one
(1024 and 2048 instances), and at N > 1 the comparison with the same circuit proved on ONE GPU in the same run.
Extras: N = 1: C2, C1, C4 on one GPU, the drop-in class, loader timings, CPU sample; N > 1: C4 strong scaling
(one 65 x 2^20 proof sharded over N GPUs); N = 8: C5 (2^14 instances).
"""
import hashlib
import argparse
import ctypes
import json
import lzma
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

SHA_PWS = os.path.join(ROOT, "tests", "golden", "SHA256_64.pws.xz")
METRIC = "gkr_prover_gates_per_s"
UNIT = "gates/s"


def _jd(o):
    if isinstance(o, (np.floating,)):
        return float(o)
    if isinstance(o, (np.integer,)):
        return int(o)
    raise TypeError(str(type(o)))


def load_sha(B):
    with lzma.open(SHA_PWS, "rb") as f:
        return B.Circuit.from_pws_text(f.read())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=3)
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx.append(float(s[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)   # before any pinned allocation: first touch places the pages
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B = entry.binding()

    inst = args.instances
    t_load = time.time()
    tmpl = load_sha(B)
    loader_ms = (time.time() - t_load) * 1e3
    env = Env(torch, dist, B, rank, local_rank, world)
    barrier, max_over_ranks = env.barrier, env.max_over_ranks
    # weak scaling: `inst` instances per GPU; ONE proof of the (inst * world)-instance circuit, every sumcheck table
    # dealt out to the ranks in contiguous block ranges (DESIGN.md "Multi-GPU")
    circ = tmpl.replicate(inst * world)
    gates = circ.total_gates // world
    t_create = time.time()
    prover = env.make_prover(circ)
    create_ms = (time.time() - t_create) * 1e3
    stream = torch.cuda.Stream(device=local_rank)
    prover.set_stream(stream.cuda_stream)

    ch = circ.draw_challenges()
    all_inputs = circ.inputs()
    np_in, np_ch, np_tr = env.pinned_io(prover, circ, all_inputs, ch)

    # ---------------- resident: inputs + challenges already in HBM
    prover.set_inputs(all_inputs)
    prover.set_challenges(np_ch)
    for _ in range(args.warmup):
        prover.prove()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            prover.prove()
        e1.record(stream)
    barrier()
    ms_resident = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = prover.last_prove_launches
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, prover.transcript())
    # the same K steps again with a CUDA-event pair around every kernel launch (per-class device time for the
    # roofline object; the event pairs cost a few % so `value` comes from the un-instrumented pass above)
    prover.set_profiling(True)
    lanes = prover.set_lanes(1)   # one lane: a launch's event-pair duration is its own (no other phase's kernels on the SMs)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            prover.prove()
        e1.record(stream)
    barrier()
    ms_profiled = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    prof = prover.profile()
    prover.set_profiling(False)
    lanes = prover.set_lanes(6)   # the default: 6 on one GPU, 3 on a sharded context

    # ---------------- e2e: host buffers in, transcript out, every step
    for _ in range(max(1, args.warmup // 2)):
        prover.prove_local(np_in, np_ch, np_tr)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            prover.prove_local(np_in, np_ch, np_tr)
        e1.record(stream)
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    clocks = sampler.summary()
    tr_e2e = np_tr.copy()

    total_gates = gates * world
    line = {
        "metric": METRIC, "value": total_gates / (ms_resident * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_resident, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (F_p^2, p=2^61-1)", "data": "synthetic",
        "config": {
            "workload": f"SHA256_64 x {inst * world} data-parallel instances ({inst} per GPU; BASELINE.json configs[2] at N=1, "
                        f"configs[4] family at N>1), {gates} gates per GPU, one full GKR proof per step",
            "instances_per_gpu": inst, "gates_per_gpu": gates, "rounds": None,
            "l2": "tables + values are several GB per proof, far larger than the 126 MB L2 (no flush needed)",
            "lanes": lanes, "host_numa_node": numa,
            "parallelism": "1 GPU" if world == 1 else f"one proof sharded over {world} GPUs: every sumcheck table cut into contiguous block "
                           f"ranges by index (= contiguous instance slices), local rounds without communication, one exchange per "
                           f"sumcheck phase, each rank evaluates and uploads only its own instance slice",
        },
        # bytes counted from the buffers the ranks really copy: a rank uploads the witness of its own instance range only
        "e2e": {"value": total_gates / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(env.sum_over_ranks(np_in.nbytes + np_ch.nbytes)),
                "d2h_bytes_per_step": int(np_tr.nbytes) * world,
                "api": "vp_prove_local: pinned host witness slice + challenges in, transcript out, per rank"},
        "loader": {"pws_parse_layer_subset_ms": loader_ms, "vp_create_ms": create_ms,
                   "what": "SHA256_64.pws text -> layered circuit + subsets (host, one core; the reference's parse + "
                           "DAG_to_layered + subsetInit, main.cpp:15-231, circuit.cpp:43-80); vp_create = host CSR build + upload "
                           "for the replicated circuit"},
        "gpu_launches": int(launches) * args.steps,
        "clocks": clocks,
    }
    # roofline of the dominant kernel (K6d, k_phase_dfs: all rounds of one sumcheck phase) from live CUDA-event timing of
    # every launch. achieved = SURVEY 8(d) algorithmic bytes (144 B per live table entry per sumcheck) / device time.
    peak, peak_src = measured_peaks()
    rf = prof["round_fold"]
    if rf["launches"]:
        ach = rf["bytes"] / (rf["ms"] * 1e-3) / 1e9
        step_share = rf["ms"] / sum(v["ms"] for v in prof.values())   # share of the summed kernel time (the two lanes overlap)
        ctr = dfs_counters(inst, world)
        line["roofline"] = {"bound": "hbm", "kernel": "k_phase_dfs (all rounds of one sumcheck phase in one cooperative launch: fused fold + round polynomials, two rounds per pass)",
                            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": ctr.get("traffic_bytes_per_launch"),
                            "peak_source": peak_src, "launches_per_step": rf["launches"] // args.steps,
                            "avg_launch_us": rf["ms"] * 1e3 / rf["launches"], "share_of_step": step_share,
                            "ms_per_step_instrumented": ms_profiled,
                            "bytes_model": "144 B per live table entry per sumcheck (SURVEY 8d: 3 tables x 16 B, read N_k + write N_k/2 "
                                           "per round); the kernel itself moves ~80 B per entry (two rounds per pass) and is bound by "
                                           "integer-pipe latency, see DESIGN.md and profiles/",
                            "alg_bytes_per_launch": rf["bytes"] / rf["launches"],
                            "note": "launch durations come from the instrumented pass, which runs the phases on ONE stream "
                                    "(vp_set_lanes(1)); `value` is the un-instrumented pass with the six lanes overlapped, so the "
                                    "per-class times add up to more than the step. `traffic` = DRAM bytes read + written per launch "
                                    "(ncu, profiles/r2_dfs_counters.json), averaged over the 42 launches of one proof like `achieved`. "
                                    "`frac` is the SURVEY 8(d) algorithmic-byte figure the contract asks for; the kernel is NOT HBM bound: "
                                    "`dram_frac` = its real DRAM traffic over the measured HBM peak, `int_pipe.frac` = issued warp "
                                    "instructions per clock per SM over the limit of its own instruction mix (4 issue slots, ALU pipe and "
                                    "FMA-heavy pipe 2 / clk / SM each), `bound` names the larger of the two"}
        add_binding_roofline(line["roofline"], ctr, rf["ms"] * 1e-3 / rf["launches"], peak, clocks)
        add_step_int_frac(line["roofline"], inst, world, ms_resident, clocks)
    line["kernel_classes"] = {k: {"ms_per_step": v["ms"] / args.steps, "GBps": (v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] else None),
                                  "launches_per_step": v["launches"] // args.steps} for k, v in prof.items() if v["launches"]}
    line["kernel_classes"]["note"] = ("per-class device time of the instrumented ONE-LANE pass; it overstates init_liu by one field "
                                      "product per table entry (the pre-scaled beta_u table only exists on the second lane set of "
                                      "the multi-lane runs that `value` times)")

    # From here on nothing may cost the headline: rank 0 prints the line even if an optional leg throws, hangs in a
    # collective because another rank failed, or torchrun tears the job down (see LineGuard).
    guard = LineGuard(line, armed=(rank == 0), deadline_s=args.extras_deadline)
    try:
        # ---------------- correctness evidence for what was just timed (every N)
        line["parity"] = env.parity(prover, circ, tr_e2e, all_inputs, ch, "sha256_64_x%d" % (inst * world),
                                    single_gpu_check=(world > 1 and not args.no_extras))
        line["verifier"] = line["parity"]["verifier"]
        prover.close()
        del prover
        if not args.no_extras:
            if world == 1:
                guard.leg("pc_commit", run_pc_commit, B, tmpl)
                guard.leg("fft_gkr", run_fft_gkr, B)
                guard.leg("sumcheck_c2", run_c2, B, peak)
                guard.leg("single_proof_c1", run_c1, B, tmpl)
                guard.leg("dropin", run_dropin, B, tmpl, circ, inst)
                guard.leg("c4_single_gpu", run_c4, env, B, args)
                guard.leg("cpu_baseline", cpu_baseline_sample, args)
            else:
                # collective legs: an exception on one rank would leave the others waiting, so it ends the run (the
                # guard still prints what rank 0 has)
                line["strong_c4"] = run_c4(env, B, args)
                if world == 8:
                    line["c5"] = run_c5(env, B, tmpl, args)
        if world > 1:
            dist.destroy_process_group()
    except BaseException as e:
        line["extras_error"] = f"{type(e).__name__}: {e}"[:400]
        raise
    finally:
        guard.finish()


class LineGuard:
    """Makes sure the ONE JSON line is printed exactly once by rank 0, whatever happens after the timed regions.

    The timed numbers are complete before the correctness legs and the side measurements start. Those legs can fail
    in ways a try/except around them cannot catch: a rank blocked inside a C call (an NCCL collective whose peer
    died) never returns to the interpreter, and torchrun answers a dead rank with SIGTERM to the others. So a
    daemon thread waits on a pipe that (a) the signal wake-up fd writes to when SIGTERM / SIGINT arrive and (b)
    times out after `deadline_s`; in both cases it prints the line with an `extras_error` note and ends the process.
    finish() is the normal path: it prints the line from the main thread."""

    def __init__(self, line, armed, deadline_s):
        import threading
        self.line, self.armed, self.deadline_s = line, armed, deadline_s
        self.lock = threading.Lock()
        self.done = False
        if not armed:
            return
        import signal
        self.rfd, self.wfd = os.pipe()
        os.set_blocking(self.wfd, False)
        try:
            for sig in (signal.SIGTERM, signal.SIGINT):
                signal.signal(sig, lambda *_: None)      # a Python-level handler, so the C-level one feeds the wake-up fd
            signal.set_wakeup_fd(self.wfd, warn_on_full_buffer=False)
        except ValueError:                                # not the main thread: time-out only
            pass
        threading.Thread(target=self._watch, daemon=True).start()

    def leg(self, name, fn, *a):
        """an optional single-process leg: its failure is recorded in its own slot"""
        try:
            self.line[name] = fn(*a)
        except Exception as e:
            self.line[name] = {"error": f"{type(e).__name__}: {e}"[:400]}

    def _emit_once(self, note=None):
        with self.lock:
            if self.done:
                return
            self.done = True
            if note:
                self.line.setdefault("extras_error", note)
            emit(self.line)

    def _watch(self):
        import select
        r, _, _ = select.select([self.rfd], [], [], self.deadline_s)
        if self.done:
            return
        self._emit_once("terminated by a signal after the timed regions (another rank failed?)" if r else
                        f"the legs after the timed regions did not finish within {self.deadline_s} s")
        os._exit(0 if not r else 1)

    def finish(self):
        if self.armed:
            self._emit_once()


def bind_to_gpu_numa_node(torch, local_rank):
    """Run this rank's host thread on the CPU socket its GPU hangs off (sysfs numa_node of the GPU's PCI function), so that
    the pinned witness buffers are first-touched there and host->device copies do not cross the socket interconnect. With one
    process per GPU started by torchrun nothing else places the ranks. Returns the node, or None if it cannot be determined."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


class Env:
    """process-group plumbing shared by the workload legs (torch.distributed carries ids, barriers and timing only)"""

    def __init__(self, torch, dist, B, rank, local_rank, world):
        self.torch, self.dist, self.B, self.rank, self.local_rank, self.world = torch, dist, B, rank, local_rank, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def make_prover(self, circ):
        B, torch = self.B, self.torch
        if self.world == 1:
            return B.Prover(circ, device=self.local_rank)
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if self.rank == 0:
            idt.copy_(torch.from_numpy(B.nccl_unique_id()))
        self.dist.broadcast(idt, 0)
        return B.Prover(circ, device=self.local_rank, rank=self.rank, world=self.world, nccl_id=idt.cpu().numpy())

    def pinned_io(self, prover, circ, all_inputs, ch):
        """pinned host buffers of one rank: ITS witness slice (vp_input_range), the challenges, the transcript"""
        torch, B = self.torch, self.B
        lo, hi = prover.input_range()
        s0 = circ.num_inputs // circ.instances
        pin_in = torch.empty(max(1, (hi - lo) * s0), dtype=torch.int64).pin_memory()
        pin_ch = torch.empty(len(ch) * 2, dtype=torch.int64).pin_memory()
        pin_tr = torch.empty(circ.transcript_len * 2, dtype=torch.int64).pin_memory()
        np_in = pin_in.numpy().view(np.uint64)[:(hi - lo) * s0]
        np_in[:] = all_inputs[lo * s0:hi * s0]
        np_ch = pin_ch.numpy().view(np.uint64).view(B.F_DTYPE)
        np_ch[:] = ch
        np_tr = pin_tr.numpy().view(np.uint64).view(B.F_DTYPE)
        self._keep = getattr(self, "_keep", []) + [pin_in, pin_ch, pin_tr]
        return np_in, np_ch, np_tr

    def parity(self, prover, circ, tr, all_inputs, ch, golden_name, single_gpu_check):
        """what proves that the timed transcript is the reference's: hash, rank agreement, device verifier (collective),
        reference golden hash when there is one, and at N > 1 the same circuit proved on one GPU by rank 0"""
        out = {"transcript_sha256": sha256_of(tr), "transcript_len": int(len(tr))}
        if self.world > 1:
            hashes = [None] * self.world
            self.dist.all_gather_object(hashes, out["transcript_sha256"])
            out["all_ranks_same_transcript"] = len(set(hashes)) == 1
        t0 = time.time()
        ok, code, layer = prover.verify(tr)
        out["verifier"] = {"accept": bool(ok), "fail_code": int(code), "fail_layer": int(layer), "wall_ms": (time.time() - t0) * 1e3,
                           "what": "vp_verify (verifier.cpp's checks; O(#gates) sums on the device" +
                                   (", sharded over the ranks: collective call" if self.world > 1 else "") + ") on the timed transcript"}
        g = golden_full(golden_name)
        if g:
            out["reference_prover_sha256"] = g["transcript_sha256"]
            out["equals_reference_prover"] = g["transcript_sha256"] == out["transcript_sha256"]
        if single_gpu_check:
            eq = None
            if self.rank == 0:
                os.environ["VP_ONE_LANE"] = "1"          # one lane: a third of the table memory of the default context
                try:
                    p1 = self.B.Prover(circ, device=self.local_rank)
                    tr1 = p1.prove(inputs=all_inputs, challenges=ch)
                    eq = sha256_of(tr1) == out["transcript_sha256"]
                    p1.close()
                finally:
                    del os.environ["VP_ONE_LANE"]
            self.barrier()
            out["equals_single_gpu_proof"] = eq
        return out


def sha256_of(tr):
    return hashlib.sha256(np.ascontiguousarray(tr).tobytes()).hexdigest()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, tr):
    """--dump-outputs: the transcript of the last timed proof (what a caller reads back with vp_get_transcript) as out_dir/transcript.npy,
    float32 of shape (len, 16): the 16 little-endian bytes of each F_p^2 element (re, then im). The elements are integers
    below 2^61 that no float type holds exactly; a byte is exact in float32, and a changed element changes some byte by
    at least 1, which a comparison with an absolute tolerance below 1 (and no relative one) always catches. Inputs and challenges are fixed (the .pws inputs, challenge seed 3396), so
    two builds run with the same arguments can be compared file for file."""
    rows = np.ascontiguousarray(tr).view(np.uint8).reshape(len(tr), 16).astype(np.float32)
    assert rows.nbytes <= DUMP_LIMIT_BYTES, rows.nbytes   # 64 B per element, 3 elements per round: ~350k sumcheck rounds to reach it
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "transcript.npy"), rows)


def golden_full(name):
    try:
        with open(os.path.join(ROOT, "tests", "golden", "full_size.json")) as f:
            return json.load(f).get(name)
    except Exception:
        return None


def timed_proofs(env, prover, steps, warmup):
    """device-timed resident proofs, max over ranks -> ms per proof"""
    torch = env.torch
    for _ in range(warmup):
        prover.prove()
    env.barrier()
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        prover.prove()
    e1.record(st)
    env.barrier()
    return env.max_over_ranks(e0.elapsed_time(e1)) / steps


def run_c4(env, B, args):
    """BASELINE.json configs[3]: synthetic unlayered circuit, 65 layers x 2^20 random add/mul gates with operands from
    any earlier layer (2^26 gates); ONE proof, sharded over the N GPUs of the run (strong scaling)."""
    t0 = time.time()
    circ = B.Circuit.random(65, 20, 7)
    gen_ms = (time.time() - t0) * 1e3
    t0 = time.time()
    p = env.make_prover(circ)
    create_ms = (time.time() - t0) * 1e3
    p.set_stream(env.torch.cuda.current_stream().cuda_stream)
    ch, inp = circ.draw_challenges(), circ.inputs()
    p.set_inputs(inp)
    p.set_challenges(ch)
    ms = timed_proofs(env, p, max(3, args.steps // 2), 3)
    np_in, np_ch, np_tr = env.pinned_io(p, circ, inp, ch)
    p.prove_local(np_in, np_ch, np_tr)
    out = {"workload": "random add/mul circuit, 65 layers x 2^20 gates (67.1 M gates), one proof sharded over %d GPU(s)" % env.world,
           "ms_per_proof": ms, "gates_per_s": circ.total_gates / (ms * 1e-3), "n_gpus": env.world, "scaling": "strong",
           "circuit_gen_ms": gen_ms, "vp_create_ms": create_ms,
           "parity": env.parity(p, circ, np_tr.copy(), inp, ch, "random_65x20", single_gpu_check=False)}
    p.close()
    return out


def run_c5(env, B, tmpl, args):
    """BASELINE.json configs[4]: SHA256 batch of 2^14 instances (1.52 G gates) on 8 GPUs"""
    circ = tmpl.replicate(2048 * env.world)
    t0 = time.time()
    p = env.make_prover(circ)
    create_ms = (time.time() - t0) * 1e3
    p.set_stream(env.torch.cuda.current_stream().cuda_stream)
    ch, inp = circ.draw_challenges(), circ.inputs()
    p.set_inputs(inp)
    p.set_challenges(ch)
    ms = timed_proofs(env, p, max(3, args.steps // 2), 3)
    np_in, np_ch, np_tr = env.pinned_io(p, circ, inp, ch)
    p.prove_local(np_in, np_ch, np_tr)
    out = {"workload": "SHA256_64 x %d instances (%d gates), one proof sharded over %d GPUs" % (circ.instances, circ.total_gates, env.world),
           "ms_per_proof": ms, "gates_per_s": circ.total_gates / (ms * 1e-3), "n_gpus": env.world, "vp_create_ms": create_ms,
           "parity": env.parity(p, circ, np_tr.copy(), inp, ch, "sha256_64_x%d" % circ.instances, single_gpu_check=True)}
    p.close()
    return out


_P61 = (1 << 61) - 1


def _mulmod61(a, b):
    """a * b mod 2^61 - 1 on uint64 numpy arrays of canonical values (31-bit limbs: every partial sum stays below 2^64)"""
    m31, m30 = np.uint64((1 << 31) - 1), np.uint64((1 << 30) - 1)
    a0, a1, b0, b1 = a & m31, a >> np.uint64(31), b & m31, b >> np.uint64(31)
    mid = a1 * b0 + a0 * b1
    t = np.uint64(2) * (a1 * b1) + (mid >> np.uint64(30)) + ((mid & m30) << np.uint64(31)) + a0 * b0
    pp = np.uint64(_P61)
    t = (t & pp) + (t >> np.uint64(61))
    t = (t & pp) + (t >> np.uint64(61))
    return np.where(t >= pp, t - pp, t)


def eq_table(B, r):
    """initBetaTable(output, n, r, F_ONE) (the public array verifyPoly commits, verifier.cpp:367-383) with numpy:
    out[k] = prod_i (bit_i(k) ? r_i : 1 - r_i) over F_p[i]/(i^2 + 1)"""
    pp = np.uint64(_P61)
    sub = lambda x, y: np.where(x >= y, x - y, x + pp - y)
    add = lambda x, y: np.where(x + y >= pp, x + y - pp, x + y)
    re, im = np.ones(1, np.uint64), np.zeros(1, np.uint64)
    for x in r:
        xr, xi = np.uint64(x["re"]), np.uint64(x["im"])
        tr = sub(_mulmod61(re, xr), _mulmod61(im, xi))
        ti = add(_mulmod61(re, xi), _mulmod61(im, xr))
        re, im = np.concatenate([sub(re, tr), tr]), np.concatenate([sub(im, ti), ti])
    out = np.zeros(len(re), B.F_DTYPE)
    out["re"], out["im"] = re, im
    return out


def _rand_fe(B, seed, n):
    rng = np.random.default_rng(seed)
    a = np.zeros(n, B.F_DTYPE)
    a["re"] = rng.integers(0, _P61, n, dtype=np.uint64)
    a["im"] = rng.integers(0, _P61, n, dtype=np.uint64)
    return a


def run_pc_commit(B, tmpl):
    """SURVEY 8(f) N1: prover::commit_private (the polynomial commitment's commit phase) on the device, for the input layer
    of SHA256_64 and of SHA256_64 x 16, beside what the reference's own commit_private_array took on one host core
    (tests/golden/pc_commit.json, recorded with oracle/_ref/ref_pc_commit) and with the Merkle roots compared"""
    def load(name):
        try:
            with open(os.path.join(ROOT, "tests", "golden", name)) as f:
                return json.load(f)
        except Exception:
            return {}
    golden, golden_fri = load("pc_commit.json"), load("pc_fri.json")
    out = {}
    for name, circ in (("sha256_64", tmpl), ("sha256_64_x16", tmpl.replicate(16)), ("sha256_64_x1024", tmpl.replicate(1024))):
        p = B.Prover(circ)
        root = p.commit_private()
        ms = []
        for _ in range(5):
            p.commit_private()
            ms.append(p.last_commit_ms)
        g = golden.get(name, {})
        out[name] = {"inputs": int(circ.num_inputs), "log_len": int(circ.bit_length(0)), "device_ms": statistics.median(ms),
                     "root": root.hex(), "root_equals_reference": (root.hex() == g.get("root")) if g else None,
                     "reference_cpu_seconds": g.get("reference_commit_seconds")}
        # commit_public_array + the FRI commit phase on the inputs of tests/golden/make_golden_pc_fri.py: the eq table of
        # the point default_rng(2024) draws, fold challenges from default_rng(2224)
        b = int(circ.bit_length(0))
        q, r = eq_table(B, _rand_fe(B, 2024, b)), _rand_fe(B, 2224, b - 6)
        ms_pub, ms_fri = [], []
        for _ in range(3):
            root_h, _ = p.commit_public(q)
            ms_pub.append(p.last_commit_ms)
            roots = p.fri_commit_steps(r)
            ms_fri.append(p.last_commit_ms)
        gf = golden_fri.get(name, {})
        out[name].update({"commit_public_device_ms": statistics.median(ms_pub), "fri_commit_phase_device_ms": statistics.median(ms_fri),
                          "fri_steps": len(r), "root_h_equals_reference": (root_h.hex() == gf.get("root_h")) if gf else None,
                          "fri_roots_equal_reference": ([x.hex() for x in roots] == gf.get("roots")) if gf else None,
                          "reference_fri_commit_phase_seconds": gf.get("reference_fri_commit_seconds")})
        p.close()
    out["what"] = ("commit_private: 64 inverse NTTs + 2048 coset NTTs over F_p^2, 65 SHA3-256 per Merkle leaf, array-heap Merkle tree "
                   "(vp_commit_private); commit_public: the same encoding of the public array, per-slice 2n-point products -> quotient h "
                   "-> its extension, virtual oracle, second tree (vp_commit_public); FRI commit phase: log_len - 6 folds of the 64 "
                   "codewords with leaf chains and a tree per level (vp_fri_commit_steps)")
    return out


def run_fft_gkr(B):
    """SURVEY 8(f) N4: the commitment's inner GKR (fft_circuit_gkr::fft_gkr, once per opening) on the device, on the randomness
    stream of tests/golden/fft_gkr.json (glibc random() after srand(seed)): its running claims, proof size and verdict are
    compared with what the UNMODIFIED reference functions produced on the same stream; reference seconds from that file."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "fft_gkr.json")) as f:
            golden = json.load(f)
    except Exception:
        golden = {}
    out = {}
    for name in ("lg7_seed3396", "lg13_seed2024", "lg17_seed7"):
        g = golden.get(name)
        if not g:
            continue
        lg = g["lg"]
        rnd = B.draw_field(B.fft_gkr_rnd_count(lg), g["seed"])
        first = B.fft_gkr(lg, rnd, want_layers=False)
        runs = [B.fft_gkr(lg, rnd, want_layers=False) for _ in range(5)]
        r = runs[-1]
        fe_hex = lambda x: "%016x%016x" % (int(x["re"]), int(x["im"]))
        claims = [fe_hex(r["claims"][i]) for i in (0, 1, 2, 3, 3 + lg, 4 + lg, 5 + lg)]
        out[name] = {"lg_size": lg, "commitment_entries": 1 << (lg + 6), "device_ms": statistics.median(x["device_ms"] for x in runs),
                     "wall_ms": statistics.median(x["prover_seconds"] for x in runs) * 1e3, "first_call_wall_ms": first["prover_seconds"] * 1e3,
                     "verifier_ms": r["verifier_seconds"] * 1e3, "ok": r["ok"], "proof_size": r["proof_size"],
                     "claims_and_proof_size_equal_reference": claims == g["claims"] and r["proof_size"] == g["proof_size"],
                     "reference_cpu_seconds": g["reference_prover_seconds"]}
    B.fft_gkr_release()
    out["what"] = ("eq table, lg inverse-FFT butterfly layers, 64 x 2^lg products and their sums evaluated on the device; 2 + 2 lg sumchecks "
                   "(one pass-kernel launch each) without a host round trip; the verifier's closed forms on the host (vp_fft_gkr). "
                   "first_call_wall_ms includes creating the two cached sumcheck objects")
    return out


def run_dropin(B, tmpl, circ, inst):
    """What the reference program sees. (1) oracle/_ref/virgo_plus_run_b200 = the reference's UNMODIFIED main.cpp + verifier.cpp +
    polynomial commitment linked against the drop-in `prover` class (host/prover.cpp -> this library): its own `Prove Time`
    line on SHA256_64.pws (the class's proveTime(): host wall time inside prover methods, like prover.cpp:549-551).
    (2) the same method-by-method API (one launch per round; the polynomial comes back through mapped pinned memory the host spins on)
    on the benchmark circuit."""
    import re
    import tempfile
    out = {}
    exe = os.path.join(ROOT, "oracle", "_ref", "virgo_plus_run_b200")
    if os.path.exists(exe):
        with tempfile.TemporaryDirectory() as td:
            pws = os.path.join(td, "SHA256_64.pws")
            with lzma.open(SHA_PWS, "rb") as f, open(pws, "wb") as g:
                g.write(f.read())
            best = None
            for _ in range(3):
                t0 = time.time()
                r = subprocess.run([exe, pws], capture_output=True, text=True, timeout=300)
                wall = time.time() - t0
                m = re.search(r"Prove Time ([0-9.]+)", r.stdout)
                pc = re.search(r"Polynomial commitment: prove time ([0-9.]+)", r.stdout)
                if m and "Verification pass" in r.stderr:
                    cur = {"prove_time_s": float(m.group(1)), "pc_prove_time_s": float(pc.group(1)) if pc else None, "process_wall_s": wall}
                    if best is None or cur["prove_time_s"] < best["prove_time_s"]:
                        best = cur
            out["dropin_c1"] = dict(best or {"error": "virgo_plus_run_b200 did not print Verification pass"},
                                    what="SHA256_64.pws through the reference's UNMODIFIED main + verifier + polynomial-commitment query phase; the GKR prover, both "
                                         "commitments, the FRI folds and the commitment's inner GKR = this library; prove_time_s / pc_prove_time_s are the "
                                         "program's own `Prove Time` / `Polynomial commitment: prove time` (reference CPU: 0.142 / 0.258 s); best of 3 "
                                         "processes (each pays CUDA context creation outside those timers)")
    p = B.Prover(circ)
    B.prove_interactive(p, circ)
    t0 = time.time()
    base = p.proveTime()
    B.prove_interactive(p, circ)
    out["interactive_c3"] = {"prove_time_s": p.proveTime() - base, "wall_s": time.time() - t0,
                             "what": "SHA256_64 x %d through vp_round / vp_finalize* (the calls the drop-in class forwards to), driven from "
                                     "Python; prove_time_s = time inside the entry points (proveTime())" % inst}
    p.close()
    return out


def dfs_counters(inst, world):
    """ncu counters of k_phase_dfs for this workload (tools/dfs_counters.py -> profiles/r2_dfs_counters.json), or {}"""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dfs_counters.json")) as f:
            d = json.load(f)
        return d if d.get("instances") == inst and world == 1 else {}
    except Exception:
        return {}


def add_step_int_frac(rf, inst, world, ms_step, clocks):
    """How busy the integer pipes are over the WHOLE step (six lanes overlapped): warp instructions of one proof (ncu launch
    list of the same command, profiles/r2_step_counters.json) over what the pipes could issue in the measured step time."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_step_counters.json")) as f:
            c = json.load(f)
        if c.get("instances") != inst or world != 1 or not clocks.get("sm_mhz"):
            return
        ipc = c["warp_insts_per_proof"] / (ms_step * 1e-3 * clocks["sm_mhz"] * 1e6 * c.get("n_sm", 148))
        rf["step_int_pipe"] = {"warp_insts_per_step": c["warp_insts_per_proof"], "achieved_warp_inst_per_clk_per_sm": ipc,
                               "peak_for_this_mix": c["mix_limited_ipc_per_sm"], "frac": ipc / c["mix_limited_ipc_per_sm"],
                               "what": "all kernels of one proof over the un-instrumented step time"}
    except Exception:
        pass


def add_binding_roofline(rf, ctr, avg_launch_s, hbm_peak_gbs, clocks):
    """north_star: report HBM GB/s and integer-pipe utilisation, name the binding one. Counters per launch come from the
    committed ncu capture of the same command; durations are the live CUDA-event ones of this run."""
    if not ctr:
        return
    if ctr.get("traffic_bytes_per_launch"):
        rf["dram_frac"] = ctr["traffic_bytes_per_launch"] / avg_launch_s / 1e9 / hbm_peak_gbs
    if ctr.get("warp_insts_per_launch") and clocks.get("sm_mhz"):
        n_sm = ctr.get("n_sm", 148)
        ipc = ctr["warp_insts_per_launch"] / (avg_launch_s * clocks["sm_mhz"] * 1e6 * n_sm)     # warp instructions / clk / SM
        peak_ipc = ctr.get("mix_limited_ipc_per_sm")                                            # from the instruction mix + microbenchmarked pipe rates
        rf["int_pipe"] = {"achieved_warp_inst_per_clk_per_sm": ipc, "peak_for_this_mix": peak_ipc,
                          "frac": ipc / peak_ipc if peak_ipc else None, "alu_pipe_pct_ncu": ctr.get("alu_pipe_pct"),
                          "fma_pipe_pct_ncu": ctr.get("fma_pipe_pct"), "source": ctr.get("source")}
        if peak_ipc and rf.get("dram_frac") is not None:
            rf["bound"] = "int_pipe" if ipc / peak_ipc >= rf["dram_frac"] else "hbm"
            rf["binding_frac"] = max(ipc / peak_ipc, rf["dram_frac"])


def run_c2(B, peak):
    """BASELINE.json configs[1]: stand-alone multilinear sumcheck, random F_p^2 tables of 2^24 entries."""
    log_n = 24
    s = B.Sumcheck(log_n)
    s.fill_random(1)
    rng = np.random.default_rng(0)
    r = np.zeros(log_n, B.F_DTYPE)
    r["re"] = rng.integers(0, B.P, log_n, dtype=np.uint64)
    r["im"] = rng.integers(0, B.P, log_n, dtype=np.uint64)
    for _ in range(3):
        s.run(r)
    ms = [s.run(r)[1] for _ in range(10)]
    rm = s.round_ms()
    for _ in range(3):
        s.run(r, fused=True)
    msf = [s.run(r, fused=True)[1] for _ in range(10)]
    N = 1 << log_n
    alg = 144 * N - 144
    out = {"workload": "3 tables x 2^24 random F_p^2 entries, 24 rounds",
           "ms_per_proof": statistics.median(msf), "ms_per_proof_best": min(msf),
           "mode": "one cooperative launch, two rounds per pass (challenges known up front, as in vp_prove)",
           "algorithmic_GB": alg / 1e9, "achieved_GBps": alg / (statistics.median(msf) * 1e-3) / 1e9,
           "frac_of_peak": alg / (statistics.median(msf) * 1e-3) / 1e9 / peak,
           "one_round_per_launch": {"ms_per_proof": statistics.median(ms), "what": "the interactive path: 24 launches, each round waits for its challenge",
                                    "round2_GBps": 72 * N / (rm[1] * 1e-3) / 1e9, "round2_frac_of_peak": 72 * N / (rm[1] * 1e-3) / 1e9 / peak}}
    s.close()
    return out


def run_c1(B, tmpl):
    """BASELINE.json configs[0] on the GPU: one SHA256_64 proof (latency-bound: 439 dependent rounds)."""
    p = B.Prover(tmpl)
    p.set_challenges(tmpl.draw_challenges())
    for _ in range(3):
        p.prove()
    ms = []
    for _ in range(10):
        p.prove()
        ms.append(p.last_prove_ms)
    out = {"workload": "SHA256_64, 1 instance, 92723 gates", "ms_per_proof": statistics.median(ms),
           "gates_per_s": 92723 / (statistics.median(ms) * 1e-3), "launches": p.last_prove_launches}
    p.close()
    return out


# ---------------------------------------------------------------------------------------- CPU reference
def _ref_worker(k_inst, reps, out_q):
    """one process: the unmodified reference prover (oracle/_ref/libref_gkr.so) -- or the C oracle port when
    the compiled reference is unavailable -- on SHA256_64 x k_inst; reports seconds per proof."""
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 2)  # the reference prints per-layer progress lines on stderr
    B, O = entry.binding(), entry.oracle()
    flat = load_sha(B).replicate(k_inst).expand().flat()
    kind = "reference" if O.ref_available() else "port"
    secs = []
    for _ in range(reps):
        if kind == "reference":
            _, ps, es = O.ref_prove(flat)
            secs.append(ps + es)
        else:
            _, _, s = O.OracleCircuit(flat).prove()
            secs.append(s)
    out_q.put((kind, secs))


def cpu_run(k_inst, procs, reps):
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    ps = [ctx.Process(target=_ref_worker, args=(k_inst, reps, q)) for _ in range(procs)]
    t0 = time.time()
    for p in ps:
        p.start()
    res = [q.get() for _ in ps]
    for p in ps:
        p.join()
    wall = time.time() - t0
    return res, wall


def cpu_baseline_sample(args):
    """bounded sample for the `cpu_baseline` object of our line: 1 core, SHA256_64 x 16 instances, 1 proof"""
    k = 16
    res, _ = cpu_run(k, 1, 1)
    kind, secs = res[0]
    g = 92723 * k
    out = {"value": g / secs[0], "unit": UNIT, "cores": 1, "kind": kind,
           "sample": f"SHA256_64 x {k} instances ({g} gates), one proof, prover methods + evaluate timed (the reference's `Prove Time`)",
           "seconds": secs[0]}
    # SURVEY 8(d): the reference's own benchmark case, C1 = SHA256_64 x 1, median of 5 proofs on one core
    res1, _ = cpu_run(1, 1, 5)
    out["c1_seconds_median_of_5"] = statistics.median(res1[0][1])
    out["c1_gates_per_s"] = 92723 / out["c1_seconds_median_of_5"]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = max(1, min(os.cpu_count() or 1, 64))
    k = 8
    g = 92723 * k
    # per step: every host core proves an independent SHA256_64 x k batch (the reference is single-threaded)
    total = args.warmup + args.steps
    res, _ = cpu_run(k, procs, total)
    kind = res[0][0]
    per_step = [max(r[1][s] for r in res) for s in range(total)][args.warmup:]
    sec = sum(per_step) / len(per_step)
    value = procs * g / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 limbs (F_p^2, p=2^61-1)", "data": "synthetic",
        "config": {"workload": f"SHA256_64 x {k} instances per process ({g} gates), {procs} independent processes "
                               f"(bounded sample of the SHA256_64 x 1024 workload; the reference prover is single-threaded)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind,
                         "sample": f"{procs} processes x SHA256_64 x {k} instances per step, max time over processes"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=1024, help="SHA256_64 instances per GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the C1/C2 side measurements and the CPU sample")
    ap.add_argument("--extras-deadline", type=float, default=900.0,
                    help="seconds the legs after the timed regions may take before rank 0 prints the line without them")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the transcript of the last timed proof to DIR/transcript.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; the reference arm has no dump")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    # The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on stdout at
    # communicator creation): keep the real stdout aside, point fd 1 at stderr for the run, print the line at the end.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    global _OUT
    _OUT = real_stdout
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    real_stdout.flush()


_OUT = None


def emit(line):
    out = _OUT or sys.stdout
    out.write(json.dumps(line, default=_jd) + "\n")
    out.flush()


if __name__ == "__main__":
    main()
