#!/usr/bin/env python3
"""Regenerates the golden fixtures in this directory by running the UNMODIFIED reference
(oracle/_ref/ref_dump, built from /root/reference by `make -C oracle ref`) on:

  sha256_64          data/SHA256_64.pws as shipped (config C1)
  sha256_64_x2, _x3  the same circuit replicated K times, inputs-first instance-major (SURVEY 9.3)
  small_*            hand-written / seeded-random .pws circuits covering every gate type the parser
                     emits, operand swaps (Sub->AntiSub, Naab->AntiNaab), the Not fall-through quirk,
                     empty and single-element dad subsets, layers of size 1
  random_pws_<seed>  seeded random .pws circuits (random_pws), stored without the .pws

For each case it stores  <name>.pws.xz (except sha256_64, already here), <name>.transcript.txt.xz
(lines "TAG real img", the prover->verifier messages and received challenges in emission order) and
<name>.circuit.sha256 (digest of the reference's layeredCircuit after subsetInit in the canonical
flat layout of ref_dump.cpp::dump_circuit); small cases also keep the full <name>.circuit.bin.xz.

Only runnable where /root/reference exists (this container). The GPU box uses the committed files.
"""
import hashlib
import lzma
import os
import random
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_DUMP = os.path.join(ROOT, "oracle", "_ref", "ref_dump")


def replicate_pws(text, K):
    """K instances, all inputs of all instances first (instance-major), then all gates instance-major."""
    lines = [l for l in text.decode().split("\n") if l.strip()]
    inputs, gates, outs = [], [], []
    for l in lines:
        tok = l.split()
        if tok[1].startswith("O"):
            outs.append(tok)
        elif tok[3].startswith("I"):
            inputs.append(tok)
        else:
            gates.append(tok)
    in_rank = {int(t[1][1:]): i for i, t in enumerate(inputs)}
    g_rank = {int(t[1][1:]): i for i, t in enumerate(gates)}
    n_in, n_g = len(inputs), len(gates)

    def vid(old, k):
        return k * n_in + in_rank[old] if old in in_rank else K * n_in + k * n_g + g_rank[old]

    out = []
    for k in range(K):
        for t in inputs:
            out.append(f"P V{vid(int(t[1][1:]), k)} = I{k * n_in + in_rank[int(t[1][1:])]} E")
    for k in range(K):
        for t in gates:
            a, op, b = int(t[3][1:]), t[4], int(t[5][1:])
            out.append(f"P V{vid(int(t[1][1:]), k)} = V{vid(a, k)} {op} V{vid(b, k)} E")
    for k in range(K):
        for t in outs:
            out.append(f"P O{k * (n_in + n_g) + int(t[1][1:])} = V{vid(int(t[3][1:]), k)} E")
    return ("\n".join(out) + "\n").encode()


N_PAD_INPUTS = 200  # the reference's polynomial commitment needs bl(0) >= 8 (fails/crashes below)


def build_pws(n_in, gates):
    """gates: list of (op, a, b); operands are 'iK' (input K) or 'gK' (K-th gate of this list)."""
    def vid(x):
        return int(x[1:]) if x[0] == "i" else n_in + int(x[1:])
    lines = [f"P V{i} = I{i} E" for i in range(n_in)]
    for k, (op, a, b) in enumerate(gates):
        lines.append(f"P V{n_in + k} = V{vid(a)} {op} V{vid(b)} E")
    lines.append(f"P O{n_in + len(gates)} = V{n_in + len(gates) - 1} E")
    return ("\n".join(lines) + "\n").encode()


# every gate type the parser emits, both operand orders (Sub->AntiSub, Naab->AntiNaab swaps),
# operands from several layers back; every layer keeps >= 2 gates (a 1-gate layer has bitLength 0
# and makes the REFERENCE write r_u[-1] in sumcheckFinalize1, prover.cpp:496 -- heap corruption)
SMALL_ALLOPS = [
    ("+", "i0", "i1"), ("*", "i2", "i3"), ("NOT", "i1", "i1"), ("XOR", "i4", "i5"), ("minus", "i3", "i2"),
    ("NAAB", "i5", "i0"),                                   # g0..g5  layer 1
    ("minus", "g0", "i0"), ("minus", "i0", "g0"), ("NAAB", "g1", "i1"), ("NAAB", "i1", "g1"),
    ("XOR", "g3", "i2"), ("*", "g2", "g2"), ("+", "g4", "g5"),   # g6..g12 layer 2
    ("*", "g6", "g7"), ("+", "g8", "i3"), ("XOR", "g9", "g10"), ("minus", "g11", "g12"),  # g13..g16 layer 3
    ("*", "g13", "g14"), ("+", "g15", "g16"), ("NAAB", "g16", "g0"),  # g17..g19 layer 4
    ("*", "g17", "g18"), ("+", "g19", "i0"),  # g20, g21 layer 5
    ("+", "g20", "g21"), ("minus", "g21", "g20"),  # layer 6
]

# two interleaved chains: small layers (2 gates, bitLength 1), subsets of size 1 and 2
SMALL_CHAIN = [
    ("*", "i0", "i1"), ("+", "i2", "i3"),
    ("+", "g0", "g0"), ("*", "g1", "g0"),
    ("*", "g2", "g0"), ("XOR", "g3", "i0"),
    ("XOR", "g4", "i0"), ("+", "g5", "g4"),
    ("+", "g6", "g7"), ("*", "g7", "g6"),
]

# NOT applied to a non-input whose raw id is a valid index of the previous layer: the reference
# stores the RAW DAG id as u (main.cpp:104-110 fall-through) and evaluates the wrong wire.
# Layer 1 has 2*n_in gates so that the raw ids n_in+0 / n_in+3 are valid (but wrong) layer-1 indices.
def small_notquirk():
    n_in = N_PAD_INPUTS + 5
    g = [("+", f"i{k % n_in}", f"i{(k + 1) % n_in}") for k in range(2 * n_in)]    # layer 1: 2*n_in gates
    g += [("NOT", "g0", "g0"), ("NOT", "g3", "g3"), ("*", "g1", "g2")]              # layer 2, u = raw ids
    n1 = len(g)
    g += [("*", f"g{n1 - 3}", f"g{n1 - 2}"), ("+", f"g{n1 - 1}", "g5")]          # layer 3
    return build_pws(n_in, g)


def random_pws(seed, n_in, n_gates):
    """seeded random DAG; the last two gates of every window feed forward so no layer ends up with 1 gate"""
    rng = random.Random(seed)
    lines = [f"P V{i} = I{i} E" for i in range(n_in)]
    ops = ["+", "*", "XOR", "minus", "NAAB"]
    for g in range(n_in, n_in + n_gates):
        if rng.random() < 0.08:
            a = rng.randrange(n_in)  # NOT of an input keeps raw id == in-layer id
            lines.append(f"P V{g} = V{a} NOT V{a} E")
        else:
            lo = 0 if rng.random() < 0.3 else max(0, g - 12)
            a, b = rng.randrange(lo, g), rng.randrange(0, g)
            lines.append(f"P V{g} = V{a} {rng.choice(ops)} V{b} E")
    lines.append(f"P O{n_in + n_gates} = V{n_in + n_gates - 1} E")
    return ("\n".join(lines) + "\n").encode()


def run_case(name, pws_bytes, keep_pws=True, keep_circuit=False):
    with tempfile.TemporaryDirectory() as td:
        pws = os.path.join(td, name + ".pws")
        with open(pws, "wb") as f:
            f.write(pws_bytes)
        prefix = os.path.join(td, name)
        out = subprocess.run([REF_DUMP, pws, prefix], capture_output=True, text=True, check=True).stdout
        assert "VERIFY 1" in out, f"{name}: the reference verifier rejected its own proof\n{out}"
        tr = open(prefix + ".transcript.txt", "rb").read()
        cb = open(prefix + ".circuit.bin", "rb").read()
    if keep_pws:
        with lzma.open(os.path.join(HERE, name + ".pws.xz"), "wb", preset=9) as f:
            f.write(pws_bytes)
    with lzma.open(os.path.join(HERE, name + ".transcript.txt.xz"), "wb", preset=9) as f:
        f.write(tr)
    with open(os.path.join(HERE, name + ".circuit.sha256"), "w") as f:
        f.write(hashlib.sha256(cb).hexdigest() + "\n")
    if keep_circuit:
        with lzma.open(os.path.join(HERE, name + ".circuit.bin.xz"), "wb", preset=9) as f:
            f.write(cb)
    stats = [l for l in out.split("\n") if l.startswith(("proof size", "Input size", "mult counter"))]
    with open(os.path.join(HERE, name + ".stats.txt"), "w") as f:
        f.write("\n".join(stats) + "\n")
    print(f"{name}: {len(tr.splitlines())} transcript lines, circuit {len(cb)} B; {'; '.join(stats)}")


def main():
    if not os.path.exists(REF_DUMP):
        sys.exit("oracle/_ref/ref_dump missing: run `make -C oracle ref` (needs /root/reference)")
    with lzma.open(os.path.join(HERE, "SHA256_64.pws.xz"), "rb") as f:
        sha = f.read()
    run_case("sha256_64", sha, keep_pws=False)
    run_case("sha256_64_x2", replicate_pws(sha, 2), keep_pws=False)
    run_case("sha256_64_x3", replicate_pws(sha, 3), keep_pws=False)
    run_case("small_allops", build_pws(N_PAD_INPUTS, SMALL_ALLOPS), keep_circuit=True)
    run_case("small_chain", build_pws(N_PAD_INPUTS, SMALL_CHAIN), keep_circuit=True)
    run_case("small_notquirk", small_notquirk(), keep_circuit=True)
    run_case("small_random_a", random_pws(1, 200, 150), keep_circuit=True)
    run_case("small_random_b", random_pws(2, 333, 600), keep_circuit=True)
    run_case("small_random_c", random_pws(3, 260, 60), keep_circuit=True)
    # test_loader_and_oracle_match_live_reference_on_random_pws regenerates these .pws files from the seed
    for seed, n_in, n_gates in [(11, 200, 450), (12, 257, 900), (13, 511, 200), (14, 300, 90)]:
        run_case(f"random_pws_{seed}", random_pws(seed, n_in, n_gates), keep_pws=False, keep_circuit=True)


if __name__ == "__main__":
    main()
