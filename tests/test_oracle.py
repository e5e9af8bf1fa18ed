"""CPU tests (no GPU): the oracle and the host loader against golden fixtures recorded from the
UNMODIFIED reference (tests/golden/make_golden.py), plus the C-ABI surface of the product library."""
import hashlib
import importlib.util
import os
import re
import subprocess

import numpy as np
import pytest

import sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["small_allops", "small_chain", "small_notquirk", "small_random_a", "small_random_b", "small_random_c"]


def _make_golden():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(H.GOLDEN, "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _case_circuit(B, name, sha_pws_text):
    if name == "sha256_64":
        return B.Circuit.from_pws_text(sha_pws_text)
    if name.startswith("sha256_64_x"):
        return B.Circuit.from_pws_text(_make_golden().replicate_pws(sha_pws_text, int(name[-1])))
    return B.Circuit.from_pws_text(H.golden_bytes(name + ".pws.xz"))


# ------------------------------------------------------------------ loader == reference loader
@pytest.mark.parametrize("name", ["sha256_64", "sha256_64_x2", "sha256_64_x3"] + SMALL)
def test_loader_matches_reference_circuit(B, sha_pws_text, name):
    circ = _case_circuit(B, name, sha_pws_text)
    assert H.circuit_digest(circ) == H.golden_text(name + ".circuit.sha256").strip()
    if name in SMALL:
        assert H.circuit_dump(circ) == H.golden_bytes(name + ".circuit.bin.xz")


@pytest.mark.parametrize("K", [2, 3])
def test_template_replication_equals_reference_layering(B, sha_circuit, K):
    """template x K, materialised by the index rules, == the reference's layering of the K-fold .pws"""
    ex = sha_circuit.replicate(K).expand()
    assert H.circuit_digest(ex) == H.golden_text(f"sha256_64_x{K}.circuit.sha256").strip()


# ------------------------------------------------------------------ oracle == reference prover
@pytest.mark.parametrize("name", ["sha256_64", "sha256_64_x2", "sha256_64_x3"] + SMALL)
def test_oracle_transcript_matches_reference(B, O, sha_pws_text, name):
    circ = _case_circuit(B, name, sha_pws_text)
    oc = O.OracleCircuit(circ.flat())
    tr, ch, _ = oc.prove()
    want = H.golden_bytes(name + ".transcript.txt.xz").decode()
    got = H.transcript_text(circ, tr, ch)
    assert got == want
    ok, code, layer = oc.verify(tr)
    assert ok, (code, layer)
    # the host challenge stream (private random_r state) equals the oracle's (global srandom state)
    ch2 = circ.draw_challenges()
    assert (ch2["re"] == ch["re"]).all() and (ch2["im"] == ch["im"]).all()


def test_sha256_64_known_answers(B, O, sha_circuit):
    """SURVEY.md 9.5: values recorded independently by the surveyor from the unmodified reference."""
    want = H.golden_bytes("sha256_64.transcript.txt.xz").decode()
    first_1918 = "".join(l + "\n" for l in want.split("\n")[:1918])
    assert hashlib.sha256(first_1918.encode()).hexdigest() == \
        "6754c5ba1182b4f9914e2ea79ae7367c164e1d3fcc3db0b5d227bb5acaa2d622"
    ch = sha_circuit.draw_challenges()
    assert len(ch) == 813
    assert (int(ch[0]["re"]), int(ch[0]["im"])) == (69318801402563806, 1662776802730791352)
    assert (int(ch[1]["re"]), int(ch[1]["im"])) == (1980605035210677997, 152700460719136691)
    assert sha_circuit.inputs()[:3].tolist() == [1804289383, 846930886, 1681692777]
    assert [sha_circuit.layer_size(i) for i in range(15)] == \
        [7226, 37116, 24713, 14216, 8148, 4106, 2053, 1164, 487, 176, 176, 176, 64, 64, 64]
    assert [sha_circuit.max_dad_bit_length(i) for i in range(1, 15)] == [13, 14, 12, 13, 12, 12, 10, 9, 8, 7, 7, 6, 6, 6]
    assert sha_circuit.total_gates == 92723


def test_oracle_rejects_tampering(B, O):
    circ = B.Circuit.from_pws_text(H.golden_bytes("small_allops.pws.xz"))
    oc = O.OracleCircuit(circ.flat())
    tr, _, _ = oc.prove()
    for idx in [0, 1, 5, len(tr) // 2, len(tr) - 2, len(tr) - 1]:
        bad = tr.copy()
        bad[idx]["im"] = (int(bad[idx]["im"]) + 1) % B.P
        assert not oc.verify(bad)[0], idx


# ------------------------------------------------------------------ field
def test_field_against_python_ints(B, O):
    P = B.P
    rng = np.random.default_rng(1)
    edge = [0, 1, 2, P - 1, P - 2, (1 << 60), (1 << 60) + 1, (1 << 32) - 1, 1 << 32]
    vals = [(a, b) for a in edge for b in edge[:4]] + \
        [tuple(int(x) for x in rng.integers(0, P, 2, dtype=np.uint64)) for _ in range(300)]
    for x in vals[:60]:
        for y in vals[::7]:
            assert O.f_add(x, y) == ((x[0] + y[0]) % P, (x[1] + y[1]) % P)
            assert O.f_sub(x, y) == ((x[0] - y[0]) % P, (x[1] - y[1]) % P)
            assert O.f_mul(x, y) == ((x[0] * y[0] - x[1] * y[1]) % P, (x[0] * y[1] + x[1] * y[0]) % P)


def test_beta_table_is_eq(B, O):
    P = B.P
    rng = np.random.default_rng(2)
    for nb in [0, 1, 2, 5]:
        r = np.zeros(nb, B.F_DTYPE)
        r["re"] = rng.integers(0, P, nb, dtype=np.uint64)
        r["im"] = rng.integers(0, P, nb, dtype=np.uint64)
        init = (int(rng.integers(0, P)), int(rng.integers(0, P)))
        tab = O.beta_table(r, init)
        for i in range(1 << nb):
            acc = init
            for k in range(nb):
                rk = (int(r[k]["re"]), int(r[k]["im"]))
                acc = O.f_mul(acc, rk if (i >> k) & 1 else O.f_sub((1, 0), rk))
            assert (int(tab[i]["re"]), int(tab[i]["im"])) == acc


# ------------------------------------------------------------------ loader edge cases
def test_loader_rejects_bad_input(B):
    with pytest.raises(B.VpError):
        B.Circuit.from_pws_text(b"")                                  # nothing parsed
    with pytest.raises(B.VpError):
        B.Circuit.from_pws_text(b"P V0 = I0 E\nP V2 = V0 + V0 E\n")   # hole: V1 never defined
    with pytest.raises(B.VpError):
        B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = V0 + V5 E\n")   # undefined operand
    with pytest.raises(B.VpError):
        # NOT of a non-input whose raw id is out of range of the previous layer (reference: OOB read)
        B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 + V1 E\nP V3 = V2 NOT V2 E\n")
    with pytest.raises(B.VpError):
        B.Circuit.load_pws("/nonexistent/file.pws")


def test_loader_ignores_unknown_lines(B):
    """Release build of the reference skips lines no regex matches (assert(false) compiled out)."""
    a = B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 * V1 E\nP V3 = V2 + V0 E\nP O4 = V3 E\n")
    b = B.Circuit.from_pws_text(b"# comment\nP V0 = I0 E\nP V1 = I1 E\n\nP V2 = V0 * V1 E\r\nP V2 = V0 * V1 E\n"
                                b"P V3 = V2 + V0 E\nP V9 = V2 / V0 E\nP O4 = V3 E\n")
    assert H.circuit_dump(a) == H.circuit_dump(b)


def test_random_circuit_is_valid_and_deterministic(B, O):
    a, b = B.Circuit.random(5, 4, 9), B.Circuit.random(5, 4, 9)
    assert H.circuit_dump(a) == H.circuit_dump(b)
    assert H.circuit_dump(a) != H.circuit_dump(B.Circuit.random(5, 4, 10))
    oc = O.OracleCircuit(a.flat())
    tr, _, _ = oc.prove()
    assert oc.verify(tr)[0]


def test_oracle_handles_one_gate_layers(B, O):
    """bitLength-0 layers: the reference corrupts its heap here (r_u[-1], prover.cpp:496); the oracle
    and the product define the natural behaviour (zero rounds, claim = the single value)."""
    circ = B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 * V1 E\nP V3 = V2 + V2 E\nP V4 = V3 * V2 E\n")
    oc = O.OracleCircuit(circ.flat())
    tr, _, _ = oc.prove()
    assert oc.verify(tr)[0]


# ------------------------------------------------------------------ C ABI surface
def test_library_exports_every_declared_symbol(B):
    hdr = open(os.path.join(ROOT, "include", "virgo_b200.h")).read()
    declared = set(re.findall(r"\b(vp_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) > 50
    out = subprocess.check_output(["nm", "-D", "--defined-only", B.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    missing = sorted(declared - exported)
    assert not missing, f"declared in include/virgo_b200.h but not exported: {missing}"
    lib = B.lib()
    for name in declared:
        getattr(lib, name)
    assert b"sm_100a" in lib.vp_version()


def test_no_cpu_fallback(B, sha_circuit):
    """Without a GPU every prover entry point must fail loudly (never compute on the CPU)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(B.VpError) as e:
        B.Prover(sha_circuit)
    assert e.value.code == -3 and "no CPU fallback" in str(e.value)
    with pytest.raises(B.VpError):
        B.Sumcheck(4)


def test_product_does_not_reference_the_oracle():
    pkg = os.path.join(ROOT, "virgo-plus_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp", "Makefile")):
                txt = open(os.path.join(dp, fn), errors="ignore").read()
                assert "gkr_oracle" not in txt and "oracle/" not in txt, fn


# ------------------------------------------------------------------ oracle == compiled reference (in-memory circuits)
@pytest.mark.parametrize("n_layers,log_size,seed", [(3, 3, 1), (6, 6, 2), (4, 9, 3)])
def test_oracle_matches_compiled_reference_on_random_circuits(B, O, n_layers, log_size, seed):
    """Random add/mul circuits have no .pws form; compare against libref_gkr.so (the unmodified
    reference prover driven in verifier order). Runs wherever oracle/_ref was built."""
    if not O.ref_available():
        pytest.skip("oracle/_ref/libref_gkr.so not built (needs /root/reference)")
    circ = B.Circuit.random(n_layers, log_size, seed)
    flat = circ.flat()
    want, _, _ = O.ref_prove(flat)
    got, _, _ = O.OracleCircuit(flat).prove()
    assert (got["re"] == want["re"]).all() and (got["im"] == want["im"]).all()


# ------------------------------------------------------------------ transcript containers (host side of the product)
def test_transcript_text_and_gkrproof_container(B, O, sha_circuit):
    """the product's own text dump reproduces the reference's golden dump byte for byte, and the GKRProof byte
    stream (src/GKRProof.hpp:23-58 layout) round-trips"""
    import struct
    tr, ch, _ = O.OracleCircuit(sha_circuit.flat()).prove()
    assert sha_circuit.transcript_text(tr, ch) == H.golden_bytes("sha256_64.transcript.txt.xz").decode()
    blob = sha_circuit.to_gkrproof(tr)
    n = sha_circuit.n_layers
    assert struct.unpack_from("<Q", blob, 0)[0] == n                       # final_claims_u: one slot per layer id
    # layer 14's claim_u sits in slot 14 of final_claims_u
    re, im = struct.unpack_from("<QQ", blob, 8 + 16 * (n - 1))
    assert (re, im) == (int(tr[1 + 3 * sha_circuit.bit_length(n - 2)]["re"]), int(tr[1 + 3 * sha_circuit.bit_length(n - 2)]["im"]))
    # 439 round polynomials x 48 B + claims: GKR part = reference proof size 22 976 B + the zero slots / length words
    back = sha_circuit.from_gkrproof(blob)
    assert (back["re"] == tr["re"]).all() and (back["im"] == tr["im"]).all()
    with pytest.raises(B.VpError):
        sha_circuit.from_gkrproof(blob[:-8])
    with pytest.raises(B.VpError):
        sha_circuit.from_gkrproof(blob + b"\\0" * 8)


# ------------------------------------------------------------------ hostile loader input (ADVICE.md round 1)
def test_loader_rejects_hostile_ids_without_allocating(B):
    """a .pws line with a huge variable id must be rejected, not answered with a tgt + 1 sized allocation / abort"""
    for text in (b"P V0 = I0 E\nP V99999999999 = V0 + V0 E\n",
                 b"P V0 = I0 E\nP V184467440737095516150 = V0 + V0 E\n",     # does not fit 64 bits
                 b"P V0 = I0 E\nP V5 = V0 + V0 E\n"):                          # hole: ids must be dense
        with pytest.raises(B.VpError):
            B.Circuit.from_pws_text(text)
    c = B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 + V1 E\n")
    assert c.n_layers == 2 and c.total_gates == 1
    with pytest.raises(B.VpError):
        c.replicate(1 << 40)                      # layer size * instances overflows the 2^31 limit
    with pytest.raises(B.VpError):
        B.Circuit.from_arrays([2, 1], [6, 6, 1], [-1, -1, 0], [1, 2, 0], [0, 0, 1 << 33])   # v does not fit 32 bits
    # a caller-supplied dad subset with an out-of-range entry that no gate references
    with pytest.raises(B.VpError):
        B.Circuit.from_arrays([2, 1], [6, 6, 1], [-1, -1, 0], [1, 2, 0], [0, 0, 1], lv=[0, 0, 0],
                              dad_size=[0, 0, 2, 0], dad_id=[1, 7])


# ------------------------------------------------------------------ polynomial commitment, commit phase (N1): oracle pinned
def _pc_golden():
    import json
    with open(os.path.join(H.GOLDEN, "pc_commit.json")) as f:
        return json.load(f)


def _pc_make():
    spec = importlib.util.spec_from_file_location("make_golden_pc", os.path.join(H.GOLDEN, "make_golden_pc.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_sha3_256_known_answers(O):
    """FIPS 202 / NIST example values; the commitment hashes 64-byte blocks only (one Keccak-f permutation)"""
    assert O.sha3_256(b"").hex() == "a7ffc6f8bf1ed76651c14756a061d662f580ff4de43b49fa82d80a4b80f8434a"
    assert O.sha3_256(b"abc").hex() == "3a985da74fe225b2045c172d6bd390bd855f086e3e9d525b46bfe24511431532"
    assert O.sha3_256(b"\xa3" * 200).hex() == "79f38adec5c20307a98ef76e8324afbfd46cfd81b22e3973c65fa1bd9de31787"
    for n in (1, 55, 64, 135, 136, 137, 300):
        msg = bytes((7 * i + n) % 256 for i in range(n))
        assert O.sha3_256(msg) == hashlib.sha3_256(msg).digest()


@pytest.mark.parametrize("name", ["random_6_1", "random_7_2", "random_9_3", "random_10_4", "random_11_5", "random_12_6", "sha256_64", "sha256_64_x16"])
def test_pc_oracle_matches_reference_commit(B, O, name):
    """pc_oracle.c == the reference's commit_private_array: root, codewords, leaf hashes, tree (golden: make_golden_pc.py)"""
    g = _pc_golden()[name]
    mk = _pc_make()
    a, b = mk.case_array(B, O, name)
    assert b == g["log_len"] and len(a) == g["n"]
    got = mk.digest_of(O.pc_commit_private(a, b))
    for k in ("root", "l_eval_sha256", "leaf_sha256", "tree_sha256", "slice_size"):
        assert got[k] == g[k], k


def test_pc_oracle_matches_live_reference_when_available(B, O):
    if not os.path.exists(O.REF_PC):
        pytest.skip("oracle/_ref/ref_pc_commit not built")
    rng = np.random.default_rng(77)
    for b in (6, 9, 11):
        a = np.zeros(1 << b, O.F_DTYPE)
        a["re"] = rng.integers(0, B.P, 1 << b, dtype=np.uint64)
        a["im"] = rng.integers(0, B.P, 1 << b, dtype=np.uint64)
        r, o = O.ref_pc_commit(a, b), O.pc_commit_private(a, b)
        assert r["root"] == o["root"] and (r["l_eval"] == o["l_eval"]).all() and (r["leaf_hash"] == o["leaf_hash"]).all()


# ------------------------------------------------------------------ Fiat-Shamir mode (N4): transcriptCache restated
def test_fiat_shamir_oracle_and_host_challenges(B, O, sha_circuit):
    """the oracle's FS prover/verifier agree with each other, the product's host-side vp_fs_challenges recomputes the same
    challenges from the transcript alone, and the first draws match transcriptCache::random by hand"""
    seed = bytes(range(32))
    # transcriptCache::random (transcriptCache.hpp:40-46) by hand for the first two draws
    d1 = hashlib.sha3_256(seed).digest()
    d2 = hashlib.sha3_256(d1).digest()
    P = B.P
    for circ in (B.Circuit.random(4, 4, 9), sha_circuit):
        oc = O.OracleCircuit(circ.flat())
        tr, ch = oc.prove_fs(seed)
        assert (int(ch[0]["re"]), int(ch[0]["im"])) == (int.from_bytes(d1[:8], "little") % P, int.from_bytes(d1[8:16], "little") % P)
        if circ.bit_length(circ.n_layers - 1) >= 2:
            assert (int(ch[1]["re"]), int(ch[1]["im"])) == (int.from_bytes(d2[:8], "little") % P, int.from_bytes(d2[8:16], "little") % P)
        assert oc.verify_fs(seed, tr) == (True, 0, 0)
        ch2 = oc.fs_challenges(seed, tr)
        assert (ch2 == ch).all()
        ch3 = circ.fs_challenges(seed, tr)                     # product, host only
        assert (ch3["re"] == ch["re"]).all() and (ch3["im"] == ch["im"]).all()
        bad = tr.copy()
        k = len(bad) // 2
        bad[k]["re"] = (int(bad[k]["re"]) + 1) % P
        assert not oc.verify_fs(seed, bad)[0]                  # every later challenge changes with the message
        assert not oc.verify_fs(bytes(32), tr)[0]              # another seed: other challenges
        # the FS transcript differs from the interactive one (other challenges), same length
        tr_i, _, _ = oc.prove()
        assert len(tr_i) == len(tr) and (tr_i["re"] != tr["re"]).any()


@pytest.mark.parametrize("name", ["random_6_1", "random_9_3", "random_10_4", "random_12_6", "sha256_64"])
def test_pc_oracle_matches_reference_commit_public(B, O, name):
    """pc_oracle.c's commit_public == the reference's commit_public_array: root of the second commitment, all_sum, h_eval_arr,
    virtual oracle (golden: make_golden_pc_public.py)"""
    import json
    spec = importlib.util.spec_from_file_location("make_golden_pc_public", os.path.join(H.GOLDEN, "make_golden_pc_public.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    with open(os.path.join(H.GOLDEN, "pc_commit_public.json")) as f:
        g = json.load(f)[name]
    a, q, b = mk.case_arrays(B, O, name)
    got = mk.digest_of(O.pc_commit_public(a, q, b))
    for k in ("root_h", "all_sum_sha256", "h_eval_sha256", "vow_sha256", "slice_size"):
        assert got[k] == g[k], k


def _fri_tools():
    import json
    spec = importlib.util.spec_from_file_location("make_golden_pc_fri", os.path.join(H.GOLDEN, "make_golden_pc_fri.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    with open(os.path.join(H.GOLDEN, "pc_fri.json")) as f:
        return mk, json.load(f)


@pytest.mark.parametrize("name", ["random_9_3", "random_10_4", "random_12_6", "sha256_64"])
def test_pc_oracle_matches_reference_fri_commit_phase(B, O, name):
    """pc_oracle.c's FRI commit phase == the reference's fri::commit_phase_step run on its own virtual oracle: the root of
    every level, all level codewords and trees (golden: make_golden_pc_fri.py)"""
    mk, golden = _fri_tools()
    g = golden[name]
    a, q, b, r = mk.case_inputs(B, O, name)
    pub = O.pc_commit_public(a, q, b)
    assert pub["root_h"].hex() == g["root_h"]
    got = O.pc_fri_commit_phase(pub["vow"], b - 1, r)
    d = mk.digest_of(got["roots"], got["codes"], got["trees"])
    assert len(d["roots"]) == b - 6
    for k in ("roots", "codes_sha256", "trees_sha256", "final_sha256"):
        assert d[k] == g[k], k


def test_pc_oracle_fri_fold_is_the_even_odd_split(O):
    """size-independent property of one step, checked with plain Python integers: the codeword of a polynomial f folds to
    the codeword of f_even + r f_odd on the squared domain (what makes the phase a low-degree test)"""
    P = (1 << 61) - 1
    rng = np.random.default_rng(77)
    log_N, n = 8, 8                                           # 256 points, degree < 8
    N = 1 << log_N
    mul = lambda x, y: ((x[0] * y[0] - x[1] * y[1]) % P, (x[0] * y[1] + x[1] * y[0]) % P)
    add = lambda x, y: ((x[0] + y[0]) % P, (x[1] + y[1]) % P)
    w = (2147483648, 1033321771269002680)                     # order 2^62 (fieldElement.cpp:240-241)
    for _ in range(62 - log_N):
        w = mul(w, w)
    pw = [(1, 0)]
    for _ in range(N - 1):
        pw.append(mul(pw[-1], w))
    assert mul(pw[-1], w) == (1, 0) and pw[N // 2] == (P - 1, 0)
    coef = [[(int(rng.integers(0, P)), int(rng.integers(0, P))) for _ in range(n)] for _ in range(64)]
    r = (int(rng.integers(0, P)), int(rng.integers(0, P)))

    def ev(c, x):
        acc = (0, 0)
        for a in reversed(c):
            acc = add(mul(acc, x), a)
        return acc
    vow = np.zeros(64 * N, O.F_DTYPE)
    for j in range(64):
        for k in range(N):
            vow[((k % (N // 2)) << 7) | (j << 1) | (1 if k >= N // 2 else 0)] = ev(coef[j], pw[k])
    rr = np.zeros(1, O.F_DTYPE)
    rr[0] = r
    got = O.pc_fri_commit_phase(vow, log_N, rr)["codes"][0]
    M = N // 2
    for j in (0, 17, 63):
        folded = [add(coef[j][2 * t], mul(r, coef[j][2 * t + 1])) for t in range(n // 2)]
        for k in (0, 1, 5, M // 2, M - 1):
            want = ev(folded, pw[(2 * k) % N])
            at = ((k % (M // 2)) << 7) | (j << 1) | (1 if k >= M // 2 else 0)
            assert (int(got[at]["re"]), int(got[at]["im"])) == want, (j, k)


# ------------------------------------------------------------------ the commitment's inner GKR (fft_circuit_GKR, SURVEY 8(f) N4)
FFT_GKR_CASES = ["lg1_seed3", "lg2_seed5", "lg5_seed77", "lg7_seed3396", "lg10_seed11"]


def _fft_gkr_case(O, name):
    import json
    with open(os.path.join(H.GOLDEN, "fft_gkr.json")) as f:
        g = json.load(f)[name]
    rnd = O.draw_challenges(O.fft_gkr_rnd_count(g["lg"]), seed=g["seed"])
    assert hashlib.sha256(rnd.tobytes()).hexdigest() == g["rnd_sha256"]      # the stream the reference run consumed
    return g, rnd


def fft_gkr_check_against_golden(got, g):
    """layers, the running claim after every stage the reference exposes, final alpha / beta, proof size, verdict"""
    lg = g["lg"]
    assert hashlib.sha256(np.ascontiguousarray(got["layers"]).tobytes()).hexdigest() == g["layers_sha256"]
    fe_hex = lambda x: "%016x%016x" % (int(x["re"]), int(x["im"]))
    c = got["claims"]
    assert [fe_hex(c[i]) for i in (0, 1, 2, 3, 3 + lg, 4 + lg, 5 + lg)] == g["claims"]
    assert got["proof_size"] == g["proof_size"] == g["fft_gkr_ps"] and got["ok"] and g["ok"]


@pytest.mark.parametrize("name", FFT_GKR_CASES)
def test_fft_gkr_oracle_matches_reference(O, name):
    """fftgkr_oracle.c == the UNMODIFIED reference functions driven in engage_gkr's order (golden: make_golden_fft_gkr.py)"""
    g, rnd = _fft_gkr_case(O, name)
    fft_gkr_check_against_golden(O.fft_gkr(g["lg"], rnd), g)


def test_fft_gkr_oracle_verifier_rejects_a_wrong_message(O):
    """the restated verifier is not vacuous: the claim chain pins every round polynomial (flip one coefficient -> a check fails).
    Checked with plain Python integers on the oracle's polynomials and claims of the addition layer."""
    P = (1 << 61) - 1
    g, rnd = _fft_gkr_case(O, "lg5_seed77")
    lg = g["lg"]
    out = O.fft_gkr(lg, rnd)
    mul = lambda x, y: ((x[0] * y[0] - x[1] * y[1]) % P, (x[0] * y[1] + x[1] * y[0]) % P)
    add = lambda x, y: ((x[0] + y[0]) % P, (x[1] + y[1]) % P)
    fe = lambda x: (int(x["re"]), int(x["im"]))
    ev = lambda p, x: add(mul(add(mul(fe(p[0]), x), fe(p[1])), x), fe(p[2]))
    ru = rnd[lg + 64 + 2 * (lg + 10):][:lg + 6]
    claim = fe(out["claims"][0])
    for i in range(lg + 6):
        p = out["polys"][i]
        assert add(ev(p, (0, 0)), ev(p, (1, 0))) == claim, i
        claim = ev(p, fe(ru[i]))
    bad = out["polys"][3].copy()
    bad[1]["re"] = (int(bad[1]["re"]) + 1) % P
    prev = fe(out["claims"][0])
    for i in range(3):
        prev = ev(out["polys"][i], fe(ru[i]))
    assert add(ev(bad, (0, 0)), ev(bad, (1, 0))) != prev


# ------------------------------------------------------------------ seeded random .pws circuits
@pytest.mark.parametrize("seed,n_in,n_gates", [(11, 200, 450), (12, 257, 900), (13, 511, 200), (14, 300, 90)])
def test_loader_and_oracle_match_live_reference_on_random_pws(B, O, seed, n_in, n_gates):
    """A seeded random .pws (make_golden.random_pws, regenerated here from the seed) through this repo's loader + C oracle:
    circuit dump and transcript byte-identical to what the unmodified reference's loader + prover + verifier wrote for the
    same file (golden random_pws_<seed>.*, make_golden.py). (tools/diff_reference_campaign.py ran 400 more seeds against
    the live reference: 0 mismatches.)"""
    name = f"random_pws_{seed}"
    circ = B.Circuit.from_pws_text(_make_golden().random_pws(seed, n_in, n_gates))
    assert H.circuit_dump(circ) == H.golden_bytes(name + ".circuit.bin.xz")
    tr, ch, _ = O.OracleCircuit(circ.flat()).prove()
    assert H.transcript_text(circ, tr, ch) == H.golden_bytes(name + ".transcript.txt.xz").decode()


# ------------------------------------------------------------------ Fiat-Shamir challenge source == the reference's own class
def test_fiat_shamir_challenge_source_is_the_reference_transcript_cache(B, O, sha_circuit):
    """The reference ships `transcriptCache` (lib/virgo/src/transcriptCache.hpp:14-50) but never calls it. Where the reference
    is built (oracle/_ref/ref_tcache: the UNMODIFIED class behind a script reader), replay the store / draw sequence of
    Fiat-Shamir mode (virgo-plus_b200/host/fiat_shamir.h) for an FS transcript through the reference's class: every draw must
    be the challenge the oracle used and the product's host-side vp_fs_challenges recomputes. What stays this repo's own
    design is only WHEN messages are stored and challenges drawn."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_tcache")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_tcache not built (needs /root/reference)")
    seed = bytes((7 * i + 3) & 0xff for i in range(32))
    for circ in (B.Circuit.random(5, 4, 21), B.Circuit.random(3, 1, 5), sha_circuit):
        oc = O.OracleCircuit(circ.flat())
        tr, ch = oc.prove_fs(seed)
        n = circ.n_layers
        max_bl = max(circ.bit_length(i) for i in range(n))
        script, slots = ["S " + seed.hex()], []          # slots: the challenge index every draw fills, in draw order
        fe = lambda x: script.append(f"F {int(x['re'])} {int(x['im'])}")

        def draw(ci):
            script.append("R")
            slots.append(ci)

        ti = ci = 0
        for j in range(circ.bit_length(n - 1)):
            draw(ci + j)
        ci += circ.bit_length(n - 1)
        fe(tr[ti]); ti += 1                                # Vres

        def rounds(count, base):
            nonlocal ti
            for j in range(count):
                fe(tr[ti]); fe(tr[ti + 1]); fe(tr[ti + 2]); ti += 3
                draw(base + j)

        for i in range(n - 1, 0, -1):
            pb, m = circ.bit_length(i - 1), circ.max_dad_bit_length(i)
            ci_ru, ci_assert = ci, ci + max_bl
            ci_rv = ci_assert + 1
            ci_sig = ci_rv + (m if m != -1 else 0)
            ci_rliu = ci_sig + n
            draw(ci_assert)
            rounds(pb, ci_ru)
            fe(tr[ti]); ti += 1                            # claim_u
            if m != -1:
                rounds(m, ci_rv)
                for _ in range(i):
                    fe(tr[ti]); ti += 1                    # claims_v
            for k in range(n):
                draw(ci_sig + k)
            rounds(pb, ci_rliu)
            fe(tr[ti]); ti += 1                            # claim_liu
            ci = ci_rliu + max_bl
        assert ti == len(tr) - 1 and ci == len(ch)         # the input MLE is stored last, no draw follows
        r = subprocess.run([exe], input="\n".join(script) + "\n", capture_output=True, text=True, check=True)
        draws = [tuple(int(x) for x in l.split()) for l in r.stdout.split("\n") if l.strip()]
        assert len(draws) == len(slots)
        want = np.zeros(len(ch), O.F_DTYPE)                # unused slots stay zero
        for (re_, im_), k in zip(draws, slots):
            want[k]["re"], want[k]["im"] = re_, im_
        assert (want["re"] == ch["re"]).all() and (want["im"] == ch["im"]).all()
        ch3 = circ.fs_challenges(seed, tr)                 # the product's host-side recomputation
        assert (ch3["re"] == want["re"]).all() and (ch3["im"] == want["im"]).all()


def test_gkrproof_bytes_are_read_and_rewritten_by_the_reference_container(B, O, sha_circuit, tmp_path):
    """Where the reference is built: its own (dead) GKRProof::read (src/GKRProof.hpp:101-140) parses the byte stream
    vp_transcript_to_gkrproof produces -- every member holds the transcript slice the layout says -- and its own
    GKRProof::write (:23-58) reproduces those bytes. (oracle/ref_harness/ref_gkrproof.cpp: NetIO / PolyProof are empty
    stand-ins; the product's two-element trailer sits where the reference's poly_proof would.)"""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_gkrproof")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_gkrproof not built (needs /root/reference)")
    for circ in (sha_circuit, B.Circuit.random(5, 4, 21)):
        tr, _, _ = O.OracleCircuit(circ.flat()).prove()
        blob = bytes(circ.to_gkrproof(tr))
        path = tmp_path / "proof.bin"
        path.write_bytes(blob)
        out = subprocess.run([exe, str(path)], capture_output=True, text=True, check=True).stdout.split("\n")
        assert out[-2] == f"consumed {len(blob) - 8 - 32} of {len(blob)} bytes; write() reproduces them: yes", out[-2]
        # parse the members the reference found
        it = iter(out[:-2])
        fe = lambda: tuple(int(x) for x in next(it).split())
        n = circ.n_layers

        def flat_member(name):
            head = next(it).split()
            assert head[0] == name and int(head[1]) == n, head
            return [fe() for _ in range(n)]

        def nested_member(name, per):
            head = next(it).split()
            assert head[0] == name and int(head[1]) == n, head
            rows = []
            for _ in range(n):
                cnt = int(next(it).split()[1])
                rows.append([fe() for _ in range(cnt * per)])
            return rows

        cu, cl = flat_member("final_claims_u"), flat_member("final_claims")
        cv = nested_member("final_claims_v", 1)
        pu, pv, pl = nested_member("polys_u", 3), nested_member("polys_v", 3), nested_member("polys", 3)
        # the same walk over the flat transcript as the reference's verifier makes (verifier.cpp:134-337)
        t = lambda k: (int(tr[k]["re"]), int(tr[k]["im"]))
        ti = 1
        for i in range(n - 1, 0, -1):
            pb, m = circ.bit_length(i - 1), circ.max_dad_bit_length(i)
            assert pu[i] == [t(ti + k) for k in range(3 * pb)]; ti += 3 * pb
            assert cu[i] == t(ti); ti += 1
            if m != -1:
                assert pv[i] == [t(ti + k) for k in range(3 * m)]; ti += 3 * m
                assert cv[i] == [t(ti + k) for k in range(i)]; ti += i
            else:
                assert pv[i] == [] and cv[i] == []
            assert pl[i] == [t(ti + k) for k in range(3 * pb)]; ti += 3 * pb
            assert cl[i] == t(ti); ti += 1
        assert ti == len(tr) - 1
        assert cu[0] == (0, 0) and cl[0] == (0, 0) and pu[0] == [] and pv[0] == [] and pl[0] == [] and cv[0] == []


# ------------------------------------------------------------------ verifier (N2): verdicts of the UNMODIFIED reference verifier
def verifier_verdict_cases(B, O, stride=1):
    """(circuit, oracle circuit, honest transcript, [(message index, reference verdict)]) from tests/golden/verifier_verdicts.json:
    what the stock verifier.cpp answered when message k reached it with 1 added (tools/diff_reference_verifier.py)."""
    import json
    with open(os.path.join(H.GOLDEN, "verifier_verdicts.json")) as f:
        gold = json.load(f)
    for name in SMALL:
        circ = B.Circuit.from_pws_text(H.golden_bytes(name + ".pws.xz"))
        oc = O.OracleCircuit(circ.flat())
        tr, _, _ = oc.prove()
        assert len(gold[name]) == len(tr)
        yield name, circ, oc, tr, [(k, (bool(v[0]), v[1], v[2])) for k, v in sorted((int(k), v) for k, v in gold[name].items())][::stride]


def tampered(B, tr, k):
    t = tr.copy()
    t[k]["re"] = (int(t[k]["re"]) + 1) % B.P
    return t


def test_oracle_verifier_gives_the_reference_verifiers_verdict_on_every_tampered_message(B, O):
    """2117 cases: every message of the six golden small circuits, altered one at a time. Includes the claims a prover sends for
    EMPTY dad subsets: the reference counts them in verifyLiu's claim (`~dadBitLength` is true for INT_MIN, verifier.cpp:281-284)
    and rejects a non-zero one at the first Liu round of the source layer."""
    n = 0
    for name, circ, oc, tr, cases in verifier_verdict_cases(B, O):
        assert oc.verify(tr) == (True, 0, 0)
        for k, want in cases:
            assert tuple(oc.verify(tampered(B, tr, k))) == want, (name, k)
            n += 1
        assert any(not w[0] for _, w in cases)
    assert n == 2117


def alltypes_verdict_cases(B, O, stride=1):
    """tests/golden/verifier_verdicts_alltypes.json.xz (tools/diff_reference_alltypes.py): layered circuits over ALL gate types --
    Addc / Mulc with real and complex constants, Copy, Not, assert gates: what the .pws parser never emits -- for which the
    UNMODIFIED reference (stock prover + stock verifier incl. the commitment, in-memory mode of ref_dump) accepted the honest
    run with exactly the oracle's transcript, and its verdict for every second message altered.
    -> (seed, circuit, oracle circuit, honest transcript, [(message index, reference verdict)])"""
    import json
    gold = json.loads(H.golden_bytes("verifier_verdicts_alltypes.json.xz"))
    for seed, g in sorted(gold.items(), key=lambda kv: int(kv[0])):
        a = g["arrays"]
        cst = np.zeros(len(a["c"]), B.F_DTYPE)
        cst["re"] = [x[0] for x in a["c"]]
        cst["im"] = [x[1] for x in a["c"]]
        circ = B.Circuit.from_arrays(a["sizes"], a["ty"], a["l"], a["u"], a["v"], c=cst,
                                     is_assert=a["is_assert"] if any(a["is_assert"]) else None)
        oc = O.OracleCircuit(circ.flat())
        tr, _, _ = oc.prove()
        assert len(tr) == g["transcript_len"]
        assert hashlib.sha256(np.ascontiguousarray(tr).tobytes()).hexdigest() == g["transcript_sha256"]   # what the stock verifier saw
        yield seed, circ, oc, tr, [(k, (bool(v[0]), v[1], v[2])) for k, v in sorted((int(k), v) for k, v in g["verdicts"].items())][::stride]


def test_oracle_equals_the_reference_on_all_gate_types_prover_and_verifier(B, O):
    """16 circuits x every second message: the oracle prover's transcript is what the stock verifier accepted, and the oracle
    verifier gives the stock verifier's verdict (failing check, layer) on each tampered message"""
    n = 0
    for seed, circ, oc, tr, cases in alltypes_verdict_cases(B, O):
        assert oc.verify(tr) == (True, 0, 0)
        for k, want in cases:
            assert tuple(oc.verify(tampered(B, tr, k))) == want, (seed, k)
            n += 1
    assert n > 1500


def test_loader_statement_grammar_follows_the_reference_regexes(B):
    """main.cpp:160-204: a line is a statement only if the WHOLE line matches one of the regexes (single spaces, `[0-9]+` ids with
    any number of digits); everything else is skipped -- whatever numbers it holds. Found by tools/diff_reference_pws_format.py:
    a malformed line with an overlong id used to make the loader reject the file."""
    base = b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 * V1 E\nP V3 = V2 + V0 E\nP O4 = V3 E\n"
    want = H.circuit_dump(B.Circuit.from_pws_text(base))
    skipped = [b"P V1 = V0 +  V0 E", b"P V1 = V0 + V0 E ", b" P V1 = V0 + V0 E", b"P V1 = V0 + V0 E\r", b"P V1 = V0 xor V0 E",
               b"P V1 = V0 + V0", b"V1 = V0 + V0 E", b"P V1 = V0 + I0 E", b"P V-1 = V0 + V0 E", b"P V1 = V0\t+ V0 E", b"P V1 = V0 + V0 E E",
               b"p V1 = V0 + V0 E", b"P V1.0 = V0 + V0 E", b"P V1 = V0 MINUS V0 E", b"P V = I0 E", b"P V1 = V0 +V0 E", b"\x00",
               b"P V99999999999999999999999 = I0 E x", b"P V99999999999999999999999 = V0 + V0", b"P V5 = V99999999999999999999999 NOTT V0 E"]
    for junk in skipped:
        assert H.circuit_dump(B.Circuit.from_pws_text(base + junk + b"\n")) == want, junk
        assert H.circuit_dump(B.Circuit.from_pws_text(junk + b"\n" + base)) == want, junk
    # match-preserving spellings: leading zeros; numbers the reference never uses (input index, NOT's second operand)
    assert H.circuit_dump(B.Circuit.from_pws_text(b"P V0 = I0 E\nP V01 = I1 E\nP V002 = V000 * V1 E\nP V3 = V2 + V0 E\n")) == want
    assert H.circuit_dump(B.Circuit.from_pws_text(base.replace(b"I0", b"I99999999999999999999999999"))) == want
    a = B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 * V1 E\nP V3 = V1 NOT V99999999999999999999999 E\n")
    b = B.Circuit.from_pws_text(b"P V0 = I0 E\nP V1 = I1 E\nP V2 = V0 * V1 E\nP V3 = V1 NOT V1 E\n")
    assert H.circuit_dump(a) == H.circuit_dump(b)
    # a WELL-FORMED statement with an impossible id is still an error (the reference's sscanf overflows: undefined there)
    for bad in (b"P V99999999999999999999999 = I0 E", b"P V4 = V99999999999999999999999 + V0 E", b"P V4 = V0 + V99999999999999999999999 E"):
        with pytest.raises(B.VpError):
            B.Circuit.from_pws_text(base + bad + b"\n")


@pytest.mark.parametrize("seed,K,complex_consts,with_assert", [(1, 1, False, False), (2, 1, True, True), (3, 3, True, False), (4, 5, False, True)])
def test_oracle_matches_compiled_reference_on_all_gate_types(B, O, seed, K, complex_consts, with_assert):
    """Addc / Mulc (real and complex constants), Copy, Not, assert gates, plain and replicated: the oracle prover's transcript ==
    the unmodified reference prover's (libref_gkr.so, ref_gkr_prove2; tools/diff_reference_alltypes_prover.py ran 300 circuits)."""
    if not O.ref_available():
        pytest.skip("oracle/_ref/libref_gkr.so not built (needs /root/reference)")
    import test_gpu_parity as G
    circ = G._all_types_circuit(B, 500 + seed, complex_consts=complex_consts, with_assert=with_assert)
    flat = (circ.replicate(K).expand() if K > 1 else circ).flat()
    want, _, _ = O.ref_prove(flat)
    got, _, _ = O.OracleCircuit(flat).prove()
    assert (got["re"] == want["re"]).all() and (got["im"] == want["im"]).all()
