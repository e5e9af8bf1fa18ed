"""GPU parity tests: the CUDA prover (through the C ABI) against the CPU oracle, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rand_fe(B, rng, n):
    a = np.zeros(n, B.F_DTYPE)
    a["re"] = rng.integers(0, B.P, n, dtype=np.uint64)
    a["im"] = rng.integers(0, B.P, n, dtype=np.uint64)
    return a


def _assert_same(got, want, what):
    bad = np.nonzero((got["re"] != want["re"]) | (got["im"] != want["im"]))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(want)} field elements differ, first at {bad[:5]}: " \
                          f"got {got[bad[:3]]} want {want[bad[:3]]}"


# ------------------------------------------------------------------ stand-alone sumcheck (config C2 shape)
@pytest.mark.parametrize("log_n", [1, 2, 3, 4, 5, 8, 11, 12, 14, 17])
def test_sumcheck_tables_vs_oracle(B, O, log_n):
    rng = np.random.default_rng(100 + log_n)
    n = 1 << log_n
    V, A, M = (_rand_fe(B, rng, n) for _ in range(3))
    r = _rand_fe(B, rng, log_n)
    s = B.Sumcheck(log_n)
    s.load(V, A, M)
    got, _ = s.run(r)
    want = O.sumcheck_tables(V, A, M, r)
    _assert_same(got, want, f"sumcheck 2^{log_n}")
    got2, _ = s.run(r)  # tables are restored between runs
    _assert_same(got2, want, "second run")
    got3, _ = s.run(r, fused=True)  # all rounds in one launch, two rounds per pass
    _assert_same(got3, want, "fused run")
    s.close()


def test_sumcheck_edge_values(B, O):
    """edge tables (all zero, all p-1, base field, equal pairs whose fold difference is p in weak arithmetic, zero / p-1
    alternating) x edge challenges (0, 1, p-1, i, -i, p-1 + (p-1)i, 2^31, 2^61 - 2^31) rotated through every round
    position, at 2^6, 2^15 and 2^20 entries; one round per launch and fused (k_phase_dfs: chunked passes at 2^20, one
    block alone at 2^6)"""
    for log_n in (6, 15, 20):
        _sumcheck_edge_values(B, O, log_n)


def _sumcheck_edge_values(B, O, log_n):
    P = B.P
    n = 1 << log_n
    rng = np.random.default_rng(5)
    edge = [(0, 0), (1, 0), (P - 1, 0), (0, 1), (0, P - 1), (P - 1, P - 1), (1 << 31, 0), ((1 << 61) - (1 << 31), 0)]
    challenges = [B.fe_array([edge[(j + o) % len(edge)] for j in range(log_n)]) for o in range(len(edge))]

    def const(fill):
        T = np.zeros(n, B.F_DTYPE)
        T["re"], T["im"] = fill
        return T, T, T

    def pairs():
        T = _rand_fe(B, rng, n // 2)
        return np.repeat(T, 2)

    alt = np.zeros(n, B.F_DTYPE)
    alt["re"][1::2] = alt["im"][1::2] = P - 1
    fills = [("zero", const((0, 0))), ("p-1 + (p-1)i", const((P - 1, P - 1))), ("p-1", const((P - 1, 0))), ("one", const((1, 0))),
             ("equal pairs", (pairs(), pairs(), pairs())), ("0 / p-1 + (p-1)i alternating", (alt, alt, alt))]
    s = B.Sumcheck(log_n)
    for name, (V, A, M) in fills:
        s.load(V, A, M)
        for o, r in enumerate(challenges):
            want = O.sumcheck_tables(V, A, M, r)
            got, _ = s.run(r)
            _assert_same(got, want, f"2^{log_n}, {name}, challenges rotated by {o}")
            got, _ = s.run(r, fused=True)
            _assert_same(got, want, f"2^{log_n}, {name}, challenges rotated by {o}, fused")
    s.close()


def test_sumcheck_device_random_fill(B, O):
    log_n = 10
    s = B.Sumcheck(log_n)
    s.fill_random(1)
    V, A, M = s.export()
    assert (V["re"] < B.P).all() and (M["im"] < B.P).all()
    r = O.draw_challenges(log_n)
    got, _ = s.run(r)
    _assert_same(got, O.sumcheck_tables(V, A, M, r), "device-filled tables")
    s.close()


# ------------------------------------------------------------------ full GKR proofs
def _prove_both_ways(B, O, circ, flat_circ=None):
    """batched + interactive GPU transcripts must equal the oracle's, and the oracle verifier accepts."""
    oc = O.OracleCircuit((flat_circ or circ).flat())
    want, ch_o, _ = oc.prove()
    ch = circ.draw_challenges()
    _assert_same(ch, ch_o, "challenge stream")
    p = B.Prover(circ)
    got = p.prove(inputs=circ.inputs(), challenges=ch)
    _assert_same(got, want, "batched transcript")
    ok, code, layer = oc.verify(got)
    assert ok, f"oracle verifier rejected the GPU transcript (code {code}, layer {layer})"
    p.close()
    p = B.Prover(circ)
    got_i = B.prove_interactive(p, circ)
    _assert_same(got_i, want, "interactive transcript")
    p.close()
    return want


@pytest.mark.parametrize("n_layers,log_size,seed", [(2, 0, 1), (2, 1, 2), (3, 2, 3), (4, 3, 4), (5, 5, 5), (9, 7, 6), (3, 10, 7)])
def test_random_circuits(B, O, n_layers, log_size, seed):
    circ = B.Circuit.random(n_layers, log_size, seed)
    _prove_both_ways(B, O, circ)


def test_random_circuit_c4_shape(B, O):
    """BASELINE.json configs[3] shape (random add/mul wiring, every layer 2^k gates, operands from any earlier layer)
    at a size the oracle proves in about a second: 12 layers x 2^14 gates"""
    circ = B.Circuit.random(12, 14, 2024)
    oc = O.OracleCircuit(circ.flat())
    want, _, _ = oc.prove()
    p = B.Prover(circ)
    got = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
    _assert_same(got, want, "C4-shape transcript")
    assert oc.verify(got)[0]
    p.close()


def test_evaluate_matches_oracle(B, O, sha_circuit):
    p = B.Prover(sha_circuit)
    p.evaluate()
    want = O.OracleCircuit(sha_circuit.flat()).evaluate()
    off = 0
    for i in range(sha_circuit.n_layers):
        n = sha_circuit.layer_size(i)
        _assert_same(p.values(i), want[off:off + n], f"layer {i} values")
        off += n
    p.close()


def test_sha256_64_transcript(B, O, sha_circuit):
    tr = _prove_both_ways(B, O, sha_circuit)
    # known-answer values recorded from the unmodified reference (SURVEY.md 9.5)
    assert (int(tr[0]["re"]), int(tr[0]["im"])) == (724662900143931110, 476060367020167324)
    assert (int(tr[1]["re"]), int(tr[1]["im"])) == (2211877472072237705, 669034324121346583)
    assert (int(tr[-2]["re"]), int(tr[-2]["im"])) == (2060928321185694165, 125737238808708621)


@pytest.mark.parametrize("K", [2, 3, 5])
def test_sha256_replicated_matches_expanded(B, O, sha_circuit, K):
    """K data-parallel instances through the template path == the oracle on the materialised circuit."""
    rep = sha_circuit.replicate(K)
    flat = rep.expand()
    assert flat.instances == 1 and flat.total_gates == rep.total_gates
    _prove_both_ways(B, O, rep, flat_circ=flat)


def test_replicated_random_circuit(B, O):
    circ = B.Circuit.random(4, 3, 11).replicate(7)
    _prove_both_ways(B, O, circ, flat_circ=circ.expand())


def test_negative_tampered_table_rejected(B, O, sha_circuit):
    """flip one input after the proof: the transcript no longer verifies against the circuit"""
    p = B.Prover(sha_circuit)
    ch = sha_circuit.draw_challenges()
    inp = sha_circuit.inputs()
    tr = p.prove(inputs=inp, challenges=ch)
    oc = O.OracleCircuit(sha_circuit.flat())
    assert oc.verify(tr)[0]
    bad = tr.copy()
    bad[7]["re"] = (int(bad[7]["re"]) + 1) % B.P
    assert not oc.verify(bad)[0]
    inp2 = inp.copy()
    inp2[0] ^= 1
    tr2 = p.prove(inputs=inp2, challenges=ch)
    assert not oc.verify(tr2)[0]  # oracle circuit still holds the original inputs
    p.close()


def test_inner_prod_and_proof_size(B, O, sha_circuit):
    p = B.Prover(sha_circuit)
    tr = B.prove_interactive(p, sha_circuit)
    assert abs(p.proofSize() - 22.4375) < 1e-9  # `proof size = 22.437500 kb` of the reference run
    n0 = sha_circuit.layer_size(0)
    rng = np.random.default_rng(3)
    pub = _rand_fe(B, rng, n0)
    got = p.inner_prod(pub)
    vals = p.values(0)
    acc = (0, 0)
    for i in range(n0):
        acc = O.f_add(acc, O.f_mul(vals[i], pub[i]))
    assert (int(got["re"]), int(got["im"])) == acc
    p.close()


def test_dropin_reference_verifier_accepts(tmp_path, sha_pws_text):
    """The UNMODIFIED reference main.cpp + verifier.cpp (+ its polynomial commitment), compiled against
    virgo-plus_b200/host/prover.h and linked with the B200 prover (oracle/_ref/virgo_plus_run_b200,
    built by `make -C oracle ref`), must print `Verification pass` and the reference's proof size."""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "virgo_plus_run_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/virgo_plus_run_b200 not built (needs /root/reference at build time)")
    # the binary is prebuilt where /root/reference exists and travels to the GPU box: make sure it was linked from the
    # shim sources of THIS tree (the library itself is loaded dynamically, so it is always the current one)
    import hashlib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    srcs = [os.path.join(root, "virgo-plus_b200", "host", "prover.cpp"), os.path.join(root, "virgo-plus_b200", "host", "prover.h"),
            os.path.join(root, "include", "virgo_b200.h")]
    digest = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()
    assert open(exe + ".srchash").read().strip() == digest, "virgo_plus_run_b200 is stale: run __graft_entry__.build() where /root/reference exists"
    pws = tmp_path / "SHA256_64.pws"
    pws.write_bytes(sha_pws_text)
    r = subprocess.run([exe, str(pws)], capture_output=True, text=True, timeout=300)
    assert "Verification pass" in r.stderr, r.stderr[-2000:]
    assert "proof size = 22.437500 kb" in r.stdout, r.stdout
    assert "Input size 7226" in r.stdout


# ------------------------------------------------------------------ every gate type, constants, >= 32 instances
# gate codes of inputCircuit.hpp:14-16
_MUL, _ADD, _SUB, _ANTISUB, _NAAB, _ANTINAAB, _INPUT, _MULC, _ADDC, _XOR, _NOT, _COPY = range(12)


def _all_types_circuit(B, seed, n_layers=5, max_size=24, complex_consts=False, with_assert=False):
    """random layered circuit over ALL gate types the prover knows (incl. Addc/Mulc, which the .pws parser never
    emits), operands from any earlier layer; optional zero-valued assert gates (Sub(x, x))."""
    rng = np.random.default_rng(seed)
    sizes = [int(rng.integers(3, max_size))] + [int(rng.integers(2, max_size)) for _ in range(n_layers - 1)]
    ty, l, u, v, c, asr = [], [], [], [], [], []
    for g in range(sizes[0]):
        ty.append(_INPUT); l.append(-1); u.append(int(rng.integers(0, 1 << 31))); v.append(0); c.append((0, 0)); asr.append(0)
    kinds = [_MUL, _ADD, _SUB, _ANTISUB, _NAAB, _ANTINAAB, _MULC, _ADDC, _XOR, _NOT, _COPY]
    for i in range(1, n_layers):
        for g in range(sizes[i]):
            t = kinds[int(rng.integers(0, len(kinds)))]
            uu = int(rng.integers(0, sizes[i - 1]))
            cc = (0, 0)
            a = 0
            if t in (_MULC, _ADDC):
                cc = (int(rng.integers(1, B.P)), int(rng.integers(0, B.P)) if complex_consts else 0)
            if t in (_NOT, _COPY, _MULC, _ADDC):
                ll, vv = -1, 0
            else:
                ll = int(rng.integers(0, i))
                vv = int(rng.integers(0, sizes[ll]))
            if with_assert and g == 0:   # Sub(x, x) == 0: a legal assert gate
                t, ll, vv, cc, a = _SUB, i - 1, uu, (0, 0), 1
            ty.append(t); l.append(ll); u.append(uu); v.append(vv); c.append(cc); asr.append(a)
    cst = np.zeros(len(c), B.F_DTYPE)
    cst["re"] = [x[0] for x in c]
    cst["im"] = [x[1] for x in c]
    return B.Circuit.from_arrays(sizes, ty, l, u, v, c=cst, is_assert=asr if with_assert else None)


@pytest.mark.parametrize("seed,K,complex_consts,with_assert", [(1, 1, False, False), (2, 1, True, False), (3, 1, False, True),
                                                              (4, 32, False, False), (5, 45, False, True), (6, 33, True, False),
                                                              (7, 64, False, False), (8, 100, True, True)])
def test_all_gate_types_and_instance_lanes(B, O, seed, K, complex_consts, with_assert):
    """K >= 32 with real constants takes the one-instance-per-lane init kernels; complex constants make the circuit
    values complex (no base-field shortcuts anywhere)."""
    circ = _all_types_circuit(B, seed, complex_consts=complex_consts, with_assert=with_assert)
    if K > 1:
        rep = circ.replicate(K)
        _prove_both_ways(B, O, rep, flat_circ=rep.expand())
    else:
        _prove_both_ways(B, O, circ)


@pytest.mark.parametrize("name,K", [("small_allops", 40), ("small_notquirk", 33), ("small_random_b", 70)])
def test_golden_small_circuits_replicated(B, O, name, K):
    import helpers as H
    circ = B.Circuit.from_pws_text(H.golden_bytes(name + ".pws.xz"))
    _prove_both_ways(B, O, circ)
    rep = circ.replicate(K)
    _prove_both_ways(B, O, rep, flat_circ=rep.expand())


def test_sha256_x33_instance_lanes(B, O, sha_circuit):
    """SHA256_64 x 33: real layer sizes, one full group of 32 instance lanes plus a ragged one"""
    rep = sha_circuit.replicate(33)
    want, _, _ = O.OracleCircuit(rep.expand().flat()).prove()
    p = B.Prover(rep)
    got = p.prove(inputs=rep.inputs(), challenges=rep.draw_challenges())
    _assert_same(got, want, "SHA256_64 x 33 transcript")
    p.close()


# ------------------------------------------------------------------ BASELINE.json's full sizes
# The CPU oracle proves these sizes in minutes, so parity at full size is pinned through properties instead:
#  * the two round engines of the product share no round code -- whole-proof mode (k_phase_dfs: two rounds per pass,
#    two products per pair, b derived from the claim chain, weakly canonical tables, base-field first pass, three
#    lanes) and the interactive mode (k_round: one round per launch, three products per pair, b summed directly,
#    canonical arithmetic, one stream) -- and must produce bit-identical transcripts;
#  * both are compared with the oracle (hence the reference) on the same circuits at smaller instance counts above,
#    and the K-instance transcript is a function of the template and K only.
def test_full_size_c3_whole_proof_equals_interactive(B, sha_circuit):
    """BASELINE.json configs[2]: SHA256_64 x 1024 instances (94.9 M gates)"""
    rep = sha_circuit.replicate(1024)
    p = B.Prover(rep)
    whole = p.prove(inputs=rep.inputs(), challenges=rep.draw_challenges())
    again = p.prove(inputs=rep.inputs(), challenges=rep.draw_challenges())
    _assert_same(again, whole, "second whole-proof run")
    p.close()
    p = B.Prover(rep)
    inter = B.prove_interactive(p, rep)
    p.close()
    _assert_same(whole, inter, "C3 whole-proof vs interactive transcript")
    assert np.any(whole["im"] != 0)


def test_full_size_c2_fused_equals_per_round(B, O):
    """BASELINE.json configs[1]: 3 tables x 2^24 random entries; and against the oracle at 2^20"""
    for log_n, with_oracle in ((24, False), (20, True)):
        s = B.Sumcheck(log_n)
        s.fill_random(7)
        r = O.draw_challenges(log_n)
        per_round, _ = s.run(r)
        fused, _ = s.run(r, fused=True)
        _assert_same(fused, per_round, f"2^{log_n}: fused vs one round per launch")
        if with_oracle:
            V, A, M = s.export()
            _assert_same(fused, O.sumcheck_tables(V, A, M, r), f"2^{log_n}: fused vs oracle")
        s.close()


def test_full_size_c4_whole_proof_equals_interactive(B):
    """BASELINE.json configs[3] shape at full size: 65 layers x 2^20 random add/mul gates (2^26 gates)"""
    circ = B.Circuit.random(65, 20, 1)
    p = B.Prover(circ)
    whole = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
    p.close()
    p = B.Prover(circ)
    inter = B.prove_interactive(p, circ)
    p.close()
    _assert_same(whole, inter, "C4 whole-proof vs interactive transcript")


# ------------------------------------------------------------------ device-side verifier (SURVEY 8(f) N2)
def _tamper_cases(circ, tr):
    """(name, transcript) pairs that hit every failure path of verifier.cpp:134-337"""
    import helpers as H  # noqa: F401
    n = circ.n_layers
    cases = [("honest", tr)]
    rng = np.random.default_rng(17)
    # walk the transcript layout (same as helpers.transcript_text)
    ti = 1
    top = n - 1
    pb, m = circ.bit_length(top - 1), circ.max_dad_bit_length(top)
    def flip(idx):
        bad = tr.copy()
        bad[idx]["re"] = (int(bad[idx]["re"]) + 1) % ((1 << 61) - 1)
        return bad
    cases.append(("vres", flip(0)))
    if pb:
        cases.append(("p1 round c", flip(ti + 2)))
        cases.append(("p1 round a (last)", flip(ti + 3 * (pb - 1))))
    ti += 3 * pb
    cases.append(("claim_u", flip(ti))); ti += 1
    if m != -1:
        if m:
            cases.append(("p2 round b", flip(ti + 1)))
        ti += 3 * m
        cases.append(("claim_v[0]", flip(ti))); ti += top
    if pb:
        cases.append(("liu round c", flip(ti + 2)))
    ti += 3 * pb
    cases.append(("claim_liu", flip(ti)))
    cases.append(("input mle", flip(len(tr) - 1)))
    cases.append(("random element", flip(int(rng.integers(0, len(tr))))))
    return cases


def _verify_like_oracle(B, O, circ, flat=None):
    oc = O.OracleCircuit((flat or circ).flat())
    p = B.Prover(circ)
    tr = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
    for name, t in _tamper_cases(circ, tr):
        want = oc.verify(t)
        got = p.verify(t)
        assert (bool(want[0]), want[1], want[2]) == got, f"{name}: device verifier {got}, oracle verifier {want}"
    assert p.verify(tr) == (True, 0, 0)
    p.close()


@pytest.mark.parametrize("seed,K,complex_consts,with_assert", [(1, 1, False, False), (2, 1, True, True), (4, 3, False, False),
                                                              (8, 37, True, True)])
def test_device_verifier_matches_oracle_all_gate_types(B, O, seed, K, complex_consts, with_assert):
    circ = _all_types_circuit(B, seed, complex_consts=complex_consts, with_assert=with_assert)
    if K > 1:
        rep = circ.replicate(K)
        _verify_like_oracle(B, O, rep, rep.expand())
    else:
        _verify_like_oracle(B, O, circ)


def test_device_verifier_sha256(B, O, sha_circuit):
    _verify_like_oracle(B, O, sha_circuit)
    rep = sha_circuit.replicate(5)
    _verify_like_oracle(B, O, rep, rep.expand())


def test_device_verifier_random_and_small(B, O):
    import helpers as H
    _verify_like_oracle(B, O, B.Circuit.random(6, 6, 12))
    for name in ("small_allops", "small_notquirk", "small_chain"):
        _verify_like_oracle(B, O, B.Circuit.from_pws_text(H.golden_bytes(name + ".pws.xz")))


def test_full_size_c3_device_verifier_accepts(B, sha_circuit):
    """BASELINE.json configs[2] at full size: the device verifier accepts the whole-proof transcript of SHA256_64 x 1024
    and rejects a tampered one (the verifier's sums share no code or tables with the prover)"""
    rep = sha_circuit.replicate(1024)
    p = B.Prover(rep)
    tr = p.prove(inputs=rep.inputs(), challenges=rep.draw_challenges())
    assert p.verify(tr) == (True, 0, 0)
    bad = tr.copy()
    bad[len(bad) // 2]["im"] = (int(bad[len(bad) // 2]["im"]) + 5) % B.P
    ok, code, layer = p.verify(bad)
    assert not ok and code in (1, 2, 3, 4, 5)
    p.close()


def test_lane_settings_give_identical_transcripts(B, sha_circuit):
    """vp_set_lanes: phase 1 / phase 2 / Liu on one, two, three or six streams -- same bits"""
    rep = sha_circuit.replicate(70)   # >= 64 instances: the host-io upload is cut into chunks as well
    inp, ch = rep.inputs(), rep.draw_challenges()
    p = B.Prover(rep)
    assert p.set_lanes(3) == 3
    want = p.prove(inputs=inp, challenges=ch)
    for lanes in (1, 2, 3, 6):
        assert p.set_lanes(lanes) == lanes
        _assert_same(p.prove(inputs=inp, challenges=ch), want, f"{lanes} lane(s), host buffers")
        p.set_inputs(inp)
        p.set_challenges(ch)
        p.prove()
        _assert_same(p.transcript(), want, f"{lanes} lane(s), resident")
    p.close()


# ------------------------------------------------------------------ device-only arithmetic paths, edge values
def test_device_field_primitives_edge_values(B):
    """fp_reduce_ut_weak / a96_add / mul.wide paths exist only in the device build of field.cuh: feed them 0, 1, p-1, p
    (the weak alias of 0), limb boundaries and random values through vp_selftest_field and compare with Python ints."""
    P = B.P
    edge = [0, 1, 2, P - 1, P - 2, P, (1 << 60), (1 << 60) - 1, (1 << 31) - 1, 1 << 31, (1 << 31) + 1, (1 << 32) - 1, 1 << 32,
            (1 << 30), (1 << 61) - (1 << 31), (1 << 61) - (1 << 31) - 1, 0x7FFFFFFF7FFFFFFF % P]
    rng = np.random.default_rng(99)
    vals = edge + [int(x) for x in rng.integers(0, P, 48, dtype=np.uint64)]
    n = 20000

    def arr(canonical=False):
        pool = [v for v in vals if not (canonical and v == P)]
        a = np.zeros(n, B.F_DTYPE)
        a["re"] = rng.choice(np.array(pool, dtype=np.uint64), n)
        a["im"] = rng.choice(np.array(pool, dtype=np.uint64), n)
        return a

    cm = lambda x, y: ((x[0] * y[0] - x[1] * y[1]) % P, (x[0] * y[1] + x[1] * y[0]) % P)
    t = lambda x: (int(x["re"]), int(x["im"]))
    a, b, c = arr(), arr(), arr(canonical=True)
    for op in (0, 7):   # weak fold a + c * (b - a)
        out = B.selftest_field(op, a, b, c)
        assert int(out["re"].max()) <= P and int(out["im"].max()) <= P
        for i in range(0, n, 7):
            d = ((t(b[i])[0] - t(a[i])[0]) % P, (t(b[i])[1] - t(a[i])[1]) % P)
            m = cm(d, t(c[i]))
            assert (int(out[i]["re"]) % P, int(out[i]["im"]) % P) == ((t(a[i])[0] + m[0]) % P, (t(a[i])[1] + m[1]) % P), (op, i)
    out = B.selftest_field(1, a, b, c)   # base-field data
    for i in range(0, n, 7):
        d = (int(b[i]["re"]) - int(a[i]["re"])) % P
        want = ((int(a[i]["re"]) + d * int(c[i]["re"])) % P, (d * int(c[i]["im"])) % P)
        assert (int(out[i]["re"]) % P, int(out[i]["im"]) % P) == want, i
    out = B.selftest_field(4, a, b, c)   # c + a * b
    assert int(out["re"].max()) <= P and int(out["im"].max()) <= P
    for i in range(0, n, 7):
        m = cm(t(a[i]), t(b[i]))
        assert (int(out[i]["re"]) % P, int(out[i]["im"]) % P) == ((m[0] + t(c[i])[0]) % P, (m[1] + t(c[i])[1]) % P), i
    out = B.selftest_field(5, a, b, c)   # c + a * b.re
    for i in range(0, n, 7):
        br = int(b[i]["re"])
        assert (int(out[i]["re"]) % P, int(out[i]["im"]) % P) == ((t(a[i])[0] * br + t(c[i])[0]) % P, (t(a[i])[1] * br + t(c[i])[1]) % P), i
    # any 64-bit words through the 96-bit carry-chain reduction
    big = [0, 1, P, P + 1, 2 * P, (1 << 64) - 1, (1 << 64) - 2, 1 << 63, (1 << 62) - 1, 1 << 61, 3 * P, 7 * P] + \
          [int(x) for x in rng.integers(0, 1 << 64, 40, dtype=np.uint64)]
    u = np.zeros(n, B.F_DTYPE)
    w = np.zeros(n, B.F_DTYPE)
    pick = lambda: np.array([big[k] for k in rng.integers(0, len(big), n)], dtype=np.uint64)
    u["re"], u["im"], w["re"], w["im"] = pick(), pick(), pick(), pick()
    out = B.selftest_field(3, u, w, c)
    assert int(out["re"].max()) <= P and int(out["im"].max()) <= P
    for i in range(0, n, 5):
        assert int(out[i]["re"]) % P == (int(u[i]["re"]) + (int(u[i]["im"]) << 31) + int(w[i]["re"])) % P, i
        assert int(out[i]["im"]) % P == int(w[i]["im"]) % P, i
    # lazy sums: worst-case magnitudes first
    for m_ in (1, 2, 9, 4000):
        a2, b2, c2 = arr()[:m_].copy(), arr()[:m_].copy(), arr()[:m_].copy()
        a2["re"][0] = a2["im"][0] = b2["re"][0] = b2["im"][0] = P
        out = B.selftest_field(2, a2, b2, c2)
        acc = [0, 0]
        for i in range(m_):
            mm = cm(t(a2[i]), t(b2[i]))
            acc = [(acc[0] + mm[0]) % P, (acc[1] + mm[1]) % P]
        assert t(out[0]) == tuple(acc), m_
        out = B.selftest_field(6, a2, b2, c2)
        acc = [0, 0]
        for i in range(m_):
            d = ((t(b2[i])[0] - t(a2[i])[0]) % P, (t(b2[i])[1] - t(a2[i])[1]) % P)
            acc = [(acc[0] + d[0] * int(c2[i]["re"])) % P, (acc[1] + d[1] * int(c2[i]["re"])) % P]
        assert t(out[0]) == tuple(acc), m_


# ------------------------------------------------------------------ round-2 hardening (ADVICE.md round 1)
def test_zero_constants_addc_mulc(B, O):
    """Addc / Mulc gates whose constants are ALL zero: from_arrays keeps no constant array for such a layer, the device
    still indexes one (engine uploads a zero-filled array). Values: Addc(x, 0) = x, Mulc(x, 0) = 0."""
    sizes = [4, 6, 5]
    ty = [_INPUT] * 4 + [_ADDC, _MULC, _ADDC, _ADD, _MULC, _COPY] + [_MULC, _ADDC, _MUL, _ADDC, _NOT]
    l = [-1] * 4 + [-1, -1, -1, 0, -1, -1] + [-1, -1, 0, -1, -1]
    u = [11, 22, 33, 44] + [0, 1, 2, 3, 1, 2] + [0, 1, 2, 3, 4]
    v = [0] * 4 + [0, 0, 0, 2, 0, 0] + [0, 0, 3, 0, 0]
    cst = np.zeros(len(ty), B.F_DTYPE)
    for with_c in (False, True):
        circ = B.Circuit.from_arrays(sizes, ty, l, u, v, c=cst if with_c else None)
        _prove_both_ways(B, O, circ)
        _verify_like_oracle(B, O, circ)
        rep = circ.replicate(40)
        _prove_both_ways(B, O, rep, flat_circ=rep.expand())


def test_negative_and_large_inputs_like_reference(B, O):
    """prover.cpp:30-36 loads inputs as F((long long) x): x < 0 means p + x (fieldElement.cpp:24-27). The device maps
    them the same way (k_load_inputs); the circuit-level setters only take canonical values."""
    circ = B.Circuit.random(4, 5, 21)
    inp = circ.inputs().copy()
    raw = inp.copy()
    raw[0] = np.uint64((1 << 64) - 5)            # -5
    raw[1] = np.uint64((1 << 64) - (B.P - 1))    # -(p - 1)  ->  1
    raw[2] = np.uint64(0)
    raw[3] = np.uint64(B.P - 1)
    flat = circ.flat()
    flat["inputs"] = raw.copy()
    want, _, _ = O.OracleCircuit(flat).prove()
    p = B.Prover(circ)
    got = p.prove(inputs=raw, challenges=circ.draw_challenges())
    _assert_same(got, want, "negative inputs")
    p.close()
    with pytest.raises(B.VpError):
        circ.set_inputs(raw)                     # the host-side circuit only takes values < p


def test_noncanonical_challenges_rejected(B):
    circ = B.Circuit.random(3, 4, 2)
    p = B.Prover(circ)
    ch = circ.draw_challenges()
    bad = ch.copy()
    bad[3]["im"] = B.P
    with pytest.raises(B.VpError):
        p.set_challenges(bad)
    with pytest.raises(B.VpError):
        p.prove(inputs=circ.inputs(), challenges=bad)
    p.set_challenges(ch)                         # the context is still usable
    p.prove()
    p.close()


# ------------------------------------------------------------------ BASELINE.json's full sizes against the REFERENCE
# tests/golden/full_size.json holds SHA-256 hashes of transcripts the unmodified reference prover produced at the
# benchmark sizes (tests/golden/make_golden_full.py, run once in the build container: minutes of CPU, tens of GB).
def _full_size_golden(name):
    import json
    import os
    import helpers as H
    path = os.path.join(H.GOLDEN, "full_size.json")
    if not os.path.exists(path):
        pytest.skip("tests/golden/full_size.json missing")
    g = json.load(open(path))
    if name not in g:
        pytest.skip(f"{name} not in full_size.json")
    return g[name]


def _sha(tr):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(tr).tobytes()).hexdigest()


def test_full_size_c3_transcript_hash_equals_reference(B, sha_circuit):
    """BASELINE.json configs[2], SHA256_64 x 1024: the GPU transcript hashes to what the reference prover produced"""
    g = _full_size_golden("sha256_64_x1024")
    rep = sha_circuit.replicate(1024)
    assert rep.total_gates == g["gates"] and rep.transcript_len == g["transcript_len"]
    p = B.Prover(rep)
    tr = p.prove(inputs=rep.inputs(), challenges=rep.draw_challenges())
    assert [int(tr[0]["re"]), int(tr[0]["im"])] == g["vres"]
    assert [int(tr[-1]["re"]), int(tr[-1]["im"])] == g["input_mle"]
    assert _sha(tr) == g["transcript_sha256"]
    p.close()


@pytest.mark.parametrize("name,n_layers,log_size", [("random_65x14", 65, 14), ("random_65x20", 65, 20)])
def test_c4_shape_transcript_hash_equals_reference(B, name, n_layers, log_size):
    """BASELINE.json configs[3]: 65 layers of random add/mul gates with operands from any earlier layer"""
    g = _full_size_golden(name)
    circ = B.Circuit.random(n_layers, log_size, 7)
    assert circ.total_gates == g["gates"] and circ.transcript_len == g["transcript_len"]
    p = B.Prover(circ)
    tr = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
    assert _sha(tr) == g["transcript_sha256"]
    p.close()


# ------------------------------------------------------------------ polynomial commitment, commit phase (SURVEY 8(f) N1)
def _pc_tools():
    import importlib.util
    import json
    import os
    import helpers as H
    spec = importlib.util.spec_from_file_location("make_golden_pc", os.path.join(H.GOLDEN, "make_golden_pc.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    with open(os.path.join(H.GOLDEN, "pc_commit.json")) as f:
        return m, json.load(f)


@pytest.mark.parametrize("name", ["random_6_1", "random_7_2", "random_9_3", "random_10_4", "random_11_5", "random_12_6", "sha256_64", "sha256_64_x16"])
def test_pc_commit_matches_reference_golden(B, O, name):
    """device commit (inverse NTT per slice, 32 coset NTTs, SHA3 leaf chains, Merkle tree) == what the reference's
    commit_private_array produced (root + hashes of every array), and == the oracle element by element"""
    mk, golden = _pc_tools()
    a, b = mk.case_array(B, O, name)
    got = B.pc_commit(a, b)
    g = golden[name]
    d = mk.digest_of(got)
    assert d["root"] == g["root"]
    if d["l_eval_sha256"] != g["l_eval_sha256"]:
        want = O.pc_commit_private(a, b)
        _assert_same(got["l_eval"], want["l_eval"], "l_eval")
    for k in ("l_eval_sha256", "leaf_sha256", "tree_sha256"):
        assert d[k] == g[k], k


def test_pc_commit_long_transforms_vs_oracle(B, O):
    """slices longer than the 2^11 points a block holds in shared memory (extra global stages): 2^18 and 2^19 inputs"""
    rng = np.random.default_rng(12)
    for b in (18, 19):
        a = _rand_fe(B, rng, (1 << b) - 1234)          # ragged: the tail is zero padding
        got = B.pc_commit(a, b)
        want = O.pc_commit_private(a, b)
        _assert_same(got["l_eval"], want["l_eval"], f"l_eval 2^{b}")
        assert got["root"] == want["root"] and (got["leaf_hash"] == want["leaf_hash"]).all() and (got["tree"][32:] == want["tree"][32:]).all()


def test_commit_private_through_the_context(B, O, sha_circuit):
    """prover::commit_private (prover.cpp:524-530) through the context: circuitValue[0] of SHA256_64 (x1 and x16)"""
    _, golden = _pc_tools()
    for circ, name in ((sha_circuit, "sha256_64"), (sha_circuit.replicate(16), "sha256_64_x16")):
        p = B.Prover(circ)
        root = p.commit_private()
        assert root.hex() == golden[name]["root"]
        p.evaluate()
        assert p.commit_private() == root               # also after evaluate()
        ex = p.commit_export()
        assert ex["tree"][32:64].tobytes() == root
        with pytest.raises(B.VpError):
            p.commit_private(mask=B.fe_array([(1, 0)]))  # only the GKR prover's zero mask
        p.close()


# ------------------------------------------------------------------ Fiat-Shamir mode (SURVEY 8(f) N4)
def test_fiat_shamir_mode_matches_oracle(B, O, sha_circuit):
    """vp_prove_fs: challenges hashed from the transcript (transcriptCache restated) -- transcript and challenges equal
    the oracle's FS prover; both verifiers accept it and reject a tampered or re-seeded one"""
    seed = bytes((7 * i + 1) % 256 for i in range(32))
    for circ, flat in ((B.Circuit.random(5, 6, 3), None), (sha_circuit, None), (_all_types_circuit(B, 11, with_assert=True).replicate(9), "expand")):
        f = circ.expand() if flat else circ
        oc = O.OracleCircuit(f.flat())
        want_tr, want_ch = oc.prove_fs(seed)
        p = B.Prover(circ)
        tr, ch = p.prove_fs(seed)
        _assert_same(ch, want_ch, "FS challenges")
        _assert_same(tr, want_tr, "FS transcript")
        assert oc.verify_fs(seed, tr) == (True, 0, 0)
        assert p.verify_fs(seed, tr) == (True, 0, 0)
        bad = tr.copy()
        bad[5]["im"] = (int(bad[5]["im"]) + 1) % B.P
        assert not p.verify_fs(seed, bad)[0] and not oc.verify_fs(seed, bad)[0]
        assert not p.verify_fs(bytes(32), tr)[0]
        p.close()


def test_pc_commit_c3_size_matches_reference(B, O):
    """the commit phase at the C3 benchmark size (input layer of SHA256_64 x 1024: 7.4 M values, 2^23 padded, slices of 2^17
    points: six global NTT stages on top of the shared-memory ones) against what the reference produced in 135 s"""
    import hashlib
    mk, golden = _pc_tools()
    if "sha256_64_x1024" not in golden:
        pytest.skip("no full-size commitment in pc_commit.json")
    a, b = mk.case_array(B, O, "sha256_64_x1024")
    got = B.pc_commit(a, b, want_l_eval=False)
    g = golden["sha256_64_x1024"]
    assert got["root"].hex() == g["root"]
    assert hashlib.sha256(got["leaf_hash"].tobytes()).hexdigest() == g["leaf_sha256"]
    assert hashlib.sha256(got["tree"][32:].tobytes()).hexdigest() == g["tree_sha256"]


@pytest.mark.parametrize("name", ["random_6_1", "random_9_3", "random_10_4", "random_12_6", "sha256_64"])
def test_pc_commit_public_matches_reference_golden(B, O, name):
    """device commit_public (public array encoded, l*q coefficients, quotient h extended, virtual oracle, second Merkle
    commitment) == what the reference's commit_public_array produced"""
    import importlib.util
    import json
    import os
    import helpers as H
    spec = importlib.util.spec_from_file_location("make_golden_pc_public", os.path.join(H.GOLDEN, "make_golden_pc_public.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    with open(os.path.join(H.GOLDEN, "pc_commit_public.json")) as f:
        g = json.load(f)[name]
    a, q, b = mk.case_arrays(B, O, name)
    got = B.pc_commit_public(a, q, b)
    d = mk.digest_of(got)
    if d["h_eval_sha256"] != g["h_eval_sha256"] or d["vow_sha256"] != g["vow_sha256"]:
        want = O.pc_commit_public(a, q, b)
        _assert_same(got["all_sum"], want["all_sum"], "all_sum")
        _assert_same(got["h_eval"], want["h_eval"], "h_eval")
        _assert_same(got["vow"], want["vow"], "virtual oracle")
    for k in ("root_h", "all_sum_sha256", "h_eval_sha256", "vow_sha256"):
        assert d[k] == g[k], k


def test_pc_commit_public_long_transforms_vs_oracle(B, O):
    """2^18 inputs: slices of 2^12 points, l*q transforms of 2^13 (global stages in both directions)"""
    rng = np.random.default_rng(31)
    b = 18
    a, q = _rand_fe(B, rng, (1 << b) - 5), _rand_fe(B, rng, 1 << b)
    got = B.pc_commit_public(a, q, b)
    want = O.pc_commit_public(a, q, b)
    _assert_same(got["all_sum"], want["all_sum"], "all_sum")
    _assert_same(got["h_eval"], want["h_eval"], "h_eval")
    _assert_same(got["vow"], want["vow"], "virtual oracle")
    assert got["root_h"] == want["root_h"]


def _fri_tools():
    import importlib.util
    import json
    import os
    import helpers as H
    spec = importlib.util.spec_from_file_location("make_golden_pc_fri", os.path.join(H.GOLDEN, "make_golden_pc_fri.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    with open(os.path.join(H.GOLDEN, "pc_fri.json")) as f:
        return mk, json.load(f)


@pytest.mark.parametrize("name", ["random_9_3", "random_10_4", "random_12_6", "sha256_64", "random_16_9"])
def test_pc_fri_commit_phase_matches_reference_golden(B, O, name):
    """device FRI commit phase (fold, leaf chains, tree per level) == what the reference's fri::commit_phase_step produced
    from its own virtual oracle: every level's root, all codewords, all trees"""
    mk, golden = _fri_tools()
    g = golden[name]
    a, q, b, r = mk.case_inputs(B, O, name)
    got = B.pc_fri(a, q, b, r)
    assert got["root_l"].hex() == g["root_l"] and got["root_h"].hex() == g["root_h"]
    d = mk.digest_of(got["roots"], got["codes"], got["trees"])
    if d["codes_sha256"] != g["codes_sha256"] and b <= 13:
        want = O.pc_fri_commit_phase(O.pc_commit_public(a, q, b)["vow"], b - 1, r)
        for l, (x, y) in enumerate(zip(got["codes"], want["codes"])):
            _assert_same(x, y, "codewords of level %d" % l)
    for k in ("roots", "codes_sha256", "trees_sha256", "final_sha256"):
        assert d[k] == g[k], k


def test_pc_fri_on_context_stepwise_and_restart(B, O, sha_circuit):
    """the context path the drop-in prover uses: commit_private, commit_public, then the steps one by one == all at once ==
    the oracle; exported levels equal the oracle's; too many steps / steps before commit_public are refused"""
    rng = np.random.default_rng(12)
    c = sha_circuit
    b = c.bit_length(0)
    p = B.Prover(c)
    p.evaluate()
    with pytest.raises(B.VpError):
        p.fri_commit_steps(_rand_fe(B, rng, 1))              # no commitment yet
    p.commit_private()
    with pytest.raises(B.VpError):
        p.fri_commit_steps(_rand_fe(B, rng, 1))              # no virtual oracle yet
    def interleaved(ev, N):   # fri.cpp:69-96: [(j << 7) | (slice << 1) | h] = codeword[slice][j + h N/2]
        return np.ascontiguousarray(ev[:64 * N].reshape(64, 2, N // 2).transpose(2, 0, 1)).reshape(-1)
    N = 1 << (b - 1)
    _assert_same(p.commit_export_interleaved(0), interleaved(p.commit_export()["l_eval"], N), "interleaved codewords of the first commitment")
    q = O.beta_table(_rand_fe(B, rng, b))
    root_h, _ = p.commit_public(q)
    a_in = np.zeros(c.num_inputs, B.F_DTYPE)
    a_in["re"] = c.inputs()
    _assert_same(p.commit_export_interleaved(1), interleaved(O.pc_commit_public(a_in, q, b)["h_eval"], N), "interleaved codewords of the second commitment")
    r = _rand_fe(B, rng, b - 6)
    assert p.fri_steps == b - 6
    one_by_one = [p.fri_commit_steps(r[k:k + 1])[0] for k in range(len(r))]
    with pytest.raises(B.VpError):
        p.fri_commit_steps(r[:1])                             # finished: 32 points per slice left
    p.fri_restart()
    at_once = p.fri_commit_steps(r)
    assert one_by_one == at_once
    a = np.zeros(c.num_inputs, B.F_DTYPE)
    a["re"] = c.inputs()
    pub = O.pc_commit_public(a, q, b)
    assert pub["root_h"] == root_h
    want = O.pc_fri_commit_phase(pub["vow"], b - 1, r)
    assert at_once == want["roots"]
    for lvl in (0, len(r) - 1):
        code, tree = p.fri_export_level(lvl)
        _assert_same(code, want["codes"][lvl], "level %d" % lvl)
        assert tree[32:] == want["trees"][lvl][32:]
    bad = r.copy()
    bad[0]["re"] = (1 << 61) - 1
    p.fri_restart()
    with pytest.raises(B.VpError):
        p.fri_commit_steps(bad)                               # not canonical
    p.close()


def test_pc_fri_full_size_roots_equal_reference(B, O):
    """BASELINE size: the 7.4 M inputs of SHA256_64 x 1024 (2^23 padded): every FRI level's root and the final codewords
    equal the reference's (golden made by make_golden_pc_fri.py --full)"""
    mk, golden = _fri_tools()
    if "sha256_64_x1024" not in golden:
        pytest.skip("no full-size case in pc_fri.json")
    g = golden["sha256_64_x1024"]
    a, q, b, r = mk.case_inputs(B, O, "sha256_64_x1024")
    got = B.pc_fri(a, q, b, r, want_arrays=False)
    assert got["root_l"].hex() == g["root_l"] and got["root_h"].hex() == g["root_h"]
    assert [x.hex() for x in got["roots"]] == g["roots"]


# ------------------------------------------------------------------ the commitment's inner GKR (fft_circuit_GKR, SURVEY 8(f) N4)
@pytest.mark.parametrize("name", ["lg1_seed3", "lg2_seed5", "lg5_seed77", "lg7_seed3396", "lg10_seed11", "lg13_seed2024"])
def test_fft_gkr_matches_reference_golden_and_oracle(B, O, name):
    """device fft_gkr: layer values, running claims, proof size, verdict == the reference's (golden); every round polynomial ==
    the oracle's (which the reference does not expose: pinned through the claim chain, see fftgkr_oracle.c)"""
    import json
    import os
    import helpers as H
    import test_oracle as T
    with open(os.path.join(H.GOLDEN, "fft_gkr.json")) as f:
        g = json.load(f)[name]
    lg = g["lg"]
    rnd = O.draw_challenges(O.fft_gkr_rnd_count(lg), seed=g["seed"])
    assert B.fft_gkr_rnd_count(lg) == len(rnd)
    got = B.fft_gkr(lg, rnd)
    T.fft_gkr_check_against_golden(got, g)
    want = O.fft_gkr(lg, rnd, want_layers=False)
    _assert_same(got["polys"].reshape(-1), want["polys"].reshape(-1), "round polynomials")
    _assert_same(got["claims"], want["claims"], "claims")


def test_fft_gkr_full_size_matches_reference_golden(B, O):
    """lg = 17: the inner GKR of a commitment to 2^23 values (BASELINE's 1024-instance circuit); reference: 6.5 s on one core"""
    import json
    import os
    import helpers as H
    import test_oracle as T
    with open(os.path.join(H.GOLDEN, "fft_gkr.json")) as f:
        g = json.load(f)["lg17_seed7"]
    rnd = O.draw_challenges(O.fft_gkr_rnd_count(17), seed=g["seed"])
    T.fft_gkr_check_against_golden(B.fft_gkr(17, rnd), g)


def test_fft_gkr_argument_checks(B, O):
    rnd = O.draw_challenges(O.fft_gkr_rnd_count(4), seed=1)
    with pytest.raises(B.VpError):
        B.fft_gkr(4, rnd[:-1])                       # one random element short
    bad = rnd.copy()
    bad[7]["im"] = (1 << 61) - 1
    with pytest.raises(B.VpError):
        B.fft_gkr(4, bad)                            # not canonical
    with pytest.raises(B.VpError):
        B.fft_gkr(0, rnd)
    B.fft_gkr_release()                              # frees the cached sumcheck objects; the next call recreates them
    assert B.fft_gkr(4, rnd)["ok"]


def test_random_pws_campaign_sample():
    """A slice of tools/gpu_diff_campaign.py (seeded random .pws circuits x K instances: whole proof, method by method, lane
    settings, verifier verdicts -- all against the oracle); profiles/r2f_gpu_diff_campaign.txt is the 1896-circuit run."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gpu_diff_campaign.py"), "50001", "8"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    last = r.stdout.strip().splitlines()[-1]
    assert last.startswith("gpu_diff_campaign:") and last.endswith(": 0 mismatches"), r.stdout[-2000:]
    assert int(last.split()[1]) >= 10, last


def test_device_verifier_gives_the_reference_verifiers_verdict_on_tampered_messages(B, O):
    """vp_verify against what the UNMODIFIED reference verifier answered (tests/golden/verifier_verdicts.json, recorded by
    tools/diff_reference_verifier.py): every third message of the six golden small circuits altered one at a time -- same
    accept / failing check / layer, incl. non-zero claims for empty dad subsets (rejected at the Liu phase of the source layer)."""
    import test_oracle as T
    n = 0
    for name, circ, oc, tr, cases in T.verifier_verdict_cases(B, O, stride=3):
        p = B.Prover(circ, device=0)
        got = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
        _assert_same(got, tr, name)
        assert p.verify(tr) == (True, 0, 0)
        for k, want in cases:
            assert tuple(p.verify(T.tampered(B, tr, k))) == want, (name, k)
            n += 1
        p.close()
    assert n > 700


def test_device_prover_and_verifier_equal_the_reference_on_all_gate_types(B, O):
    """The circuits of tests/golden/verifier_verdicts_alltypes.json.xz (all gate types, real / complex constants, assert gates)
    on the device: transcript == what the UNMODIFIED reference verifier accepted (hash recorded from that run), and vp_verify
    gives the stock verifier's verdict on every sixth message altered."""
    import hashlib
    import test_oracle as T
    n = 0
    for seed, circ, oc, tr, cases in T.alltypes_verdict_cases(B, O, stride=3):
        p = B.Prover(circ, device=0)
        got = p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
        _assert_same(got, tr, f"all-types circuit {seed}")
        assert p.verify(got) == (True, 0, 0)
        for k, want in cases:
            assert tuple(p.verify(T.tampered(B, tr, k))) == want, (seed, k)
            n += 1
        p.close()
        p = B.Prover(circ, device=0)
        _assert_same(B.prove_interactive(p, circ), tr, f"all-types circuit {seed}, method by method")
        p.close()
    assert n > 450


@pytest.mark.parametrize("name", ["small_allops", "small_chain", "small_notquirk", "small_random_a", "small_random_b", "small_random_c",
                                  "sha256_64_x2"])
def test_proof_size_equals_the_reference_statistics_line(B, O, sha_pws_text, name):
    """prover::proofSize() (prover.cpp:553-555, printed by main.cpp as `proof size = ... kb`) through the method-by-method API:
    the value the UNMODIFIED reference printed for the golden circuits (tests/golden/*.stats.txt), incl. the 16 bytes it counts for
    every EMPTY dad subset (the INT_MIN quirk)."""
    import re
    import helpers as H
    import test_oracle as T
    circ = T._case_circuit(B, name, sha_pws_text)
    want = float(re.search(r"proof size = ([0-9.]+) kb", H.golden_text(name + ".stats.txt")).group(1))
    p = B.Prover(circ)
    B.prove_interactive(p, circ)
    assert abs(p.proofSize() - want) < 1e-9, (p.proofSize(), want)
    p.close()
