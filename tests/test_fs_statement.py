"""Statement-bound Fiat-Shamir proofs (include/virgo_b200.h, DESIGN.md section 7): a pure-Python restatement of the statement
digest (vector root R, circuit bytes, statement) checked on hand-built cases and against the device, the bound proof
checked bit for bit against the oracle's prove_fs(statement) and the library's vp_prove_fs(statement), and the bound
verifier's verdicts."""
import copy
import hashlib
import importlib.util
import lzma
import os
import random
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
P = (1 << 61) - 1
F_DTYPE = np.dtype([("re", "<u8"), ("im", "<u8")])
GATE = np.dtype([("ty", "u1"), ("is_assert", "u1"), ("l", "<i4"), ("u", "<u4"), ("v", "<u4"), ("lv", "<u4"), ("c_re", "<u8"),
                 ("c_im", "<u8")])   # packed: 34 bytes
MUL, ADD, SUB, ANTISUB, NAAB, ANTINAAB, INPUT, MULC, ADDC, XOR, NOT, COPY = range(12)


# ------------------------------------------------------------------ the restatement
def H(b):
    return hashlib.sha3_256(b).digest()


def vector_root(data):
    """R(bytes): zero-padded to 2^k 64-byte leaves, leaf = H(block), node = H(left | right), root = node 1"""
    leaves = max(1, -(-len(data) // 64))
    k = 0
    while (1 << k) < leaves:
        k += 1
    data = bytes(data) + bytes(64 * (1 << k) - len(data))
    level = [H(data[64 * j:64 * j + 64]) for j in range(1 << k)]
    while len(level) > 1:
        level = [H(level[2 * i] + level[2 * i + 1]) for i in range(len(level) // 2)]
    return level[0]


def describe(circ):
    """what the export functions return: layer sizes, template gates of layers >= 1, dad subsets"""
    n = circ.n_layers
    return dict(n=n, K=circ.instances, sizes=[circ.layer_size(i) for i in range(n)],
                gates=[None] + [circ.export_layer(i) for i in range(1, n)],
                dads=[[circ.export_dad(i, s) for s in range(i)] for i in range(n)])


def circuit_bytes(d):
    out = [b"VPCIRC01", struct.pack("<QQ", d["n"], d["K"])] + [struct.pack("<Q", s) for s in d["sizes"]]
    for i in range(1, d["n"]):
        L = d["gates"][i]
        g = np.zeros(d["sizes"][i], GATE)
        for k in ("ty", "is_assert", "l", "u", "v", "lv"):
            g[k] = L[k]
        g["c_re"], g["c_im"] = L["c"]["re"], L["c"]["im"]
        out.append(g.tobytes())
    for i in range(1, d["n"]):
        for s in range(i):
            ids = np.ascontiguousarray(d["dads"][i][s], dtype="<u4")
            out.append(struct.pack("<Q", len(ids)) + ids.tobytes())
    return b"".join(out)


def field_bytes(values):
    return np.ascontiguousarray(values, dtype=F_DTYPE).tobytes()


def statement(circuit_digest, inputs, outputs, context):
    """inputs / outputs: field-element arrays"""
    return H(b"VPSTMT01" + circuit_digest + struct.pack("<Q", len(inputs)) + vector_root(field_bytes(inputs)) +
             struct.pack("<Q", len(outputs)) + vector_root(field_bytes(outputs)) + bytes(context))


def digests(circ, inputs, outputs, context):
    cd = vector_root(circuit_bytes(describe(circ)))
    return dict(circuit=cd, inputs=vector_root(field_bytes(inputs)), outputs=vector_root(field_bytes(outputs)),
                statement=statement(cd, inputs, outputs, context))


def oracle_values(O, circ):
    """(inputs, outputs) as field elements, evaluated by the CPU oracle on the materialised circuit"""
    f = (circ.expand() if circ.instances > 1 else circ).flat()
    vals = O.OracleCircuit(f).evaluate()
    off = f["gate_off"]
    return vals[:int(off[1])], vals[int(off[-2]):]


# ------------------------------------------------------------------ circuits
def all_types_circuit(B, seed, n_layers=5, max_size=24, complex_consts=True, with_assert=True, sizes=None):
    """random layered circuit over all gate types (Addc / Mulc with complex constants, zero-valued assert gates); `sizes`
    fixes the layer sizes (1-gate layers included)"""
    rng = np.random.default_rng(seed)
    if sizes is None:
        sizes = [int(rng.integers(3, max_size))] + [int(rng.integers(2, max_size)) for _ in range(n_layers - 1)]
    n_layers = len(sizes)
    ty, l, u, v, c, asr = [], [], [], [], [], []
    for g in range(sizes[0]):
        ty.append(INPUT); l.append(-1); u.append(int(rng.integers(0, 1 << 31))); v.append(0); c.append((0, 0)); asr.append(0)
    kinds = [MUL, ADD, SUB, ANTISUB, NAAB, ANTINAAB, MULC, ADDC, XOR, NOT, COPY]
    for i in range(1, n_layers):
        for g in range(sizes[i]):
            t = kinds[int(rng.integers(0, len(kinds)))]
            uu, cc, a = int(rng.integers(0, sizes[i - 1])), (0, 0), 0
            if t in (MULC, ADDC):
                cc = (int(rng.integers(1, P)), int(rng.integers(0, P)) if complex_consts else 0)
            if t in (NOT, COPY, MULC, ADDC):
                ll, vv = -1, 0
            else:
                ll = int(rng.integers(0, i))
                vv = int(rng.integers(0, sizes[ll]))
            if with_assert and g == 0 and sizes[i] > 1:   # Sub(x, x) == 0: a legal assert gate
                t, ll, vv, cc, a = SUB, i - 1, uu, (0, 0), 1
            ty.append(t); l.append(ll); u.append(uu); v.append(vv); c.append(cc); asr.append(a)
    cst = np.zeros(len(c), F_DTYPE)
    cst["re"] = [x[0] for x in c]
    cst["im"] = [x[1] for x in c]
    return B.Circuit.from_arrays(sizes, ty, l, u, v, c=cst, is_assert=asr if with_assert else None)


def one_gate_layers_circuit(B, seed):
    return all_types_circuit(B, seed, complex_consts=False, with_assert=False, sizes=[5, 1, 3, 1, 1, 2, 1])


def _make_golden():
    spec = importlib.util.spec_from_file_location("make_golden_fs", os.path.join(GOLDEN, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg


def _golden_pws(B, name):
    with lzma.open(os.path.join(GOLDEN, f"{name}.pws.xz"), "rb") as f:
        return B.Circuit.from_pws_text(f.read())


CONTEXT = bytes((3 * i + 5) % 256 for i in range(32))


# ------------------------------------------------------------------ CPU
def test_vector_root_hand_built():
    """one leaf, two leaves, a non-power-of-two leaf count and a length that is not a multiple of 64"""
    a = bytes(range(64))
    assert vector_root(a) == H(a)
    assert vector_root(b"") == H(bytes(64))
    assert vector_root(b"\x01") == H(b"\x01" + bytes(63))
    b = bytes((7 * i) % 251 for i in range(128))
    assert vector_root(b) == H(H(b[:64]) + H(b[64:]))
    c = bytes((5 * i + 1) % 253 for i in range(3 * 64))
    l = [H(c[:64]), H(c[64:128]), H(c[128:]), H(bytes(64))]
    assert vector_root(c) == H(H(l[0] + l[1]) + H(l[2] + l[3]))
    d = c[:150]   # 2.3 blocks: the third block zero-padded, a fourth zero leaf
    l = [H(d[:64]), H(d[64:128]), H(d[128:] + bytes(64 - 22)), H(bytes(64))]
    assert vector_root(d) == H(H(l[0] + l[1]) + H(l[2] + l[3]))
    assert len(b"VPSTMT01" + bytes(32) + bytes(8) + bytes(32) + bytes(8) + bytes(32) + bytes(32)) == 152


def test_circuit_bytes_layout(B):
    circ = all_types_circuit(B, 21)
    d = describe(circ)
    raw = circuit_bytes(d)
    n = d["n"]
    assert raw[:8] == b"VPCIRC01" and struct.unpack_from("<QQ", raw, 8) == (n, 1)
    assert list(struct.unpack_from(f"<{n}Q", raw, 24)) == d["sizes"]
    o = 24 + 8 * n
    g = np.frombuffer(raw, GATE, count=d["sizes"][1], offset=o)
    assert GATE.itemsize == 34 and (g["ty"] == d["gates"][1]["ty"]).all() and (g["c_im"] == d["gates"][1]["c"]["im"]).all()
    o += 34 * sum(d["sizes"][1:])
    assert struct.unpack_from("<Q", raw, o)[0] == len(d["dads"][1][0])
    assert len(raw) == o + sum(8 + 4 * len(d["dads"][i][s]) for i in range(1, n) for s in range(i))
    rep = circ.replicate(3)
    assert circuit_bytes(describe(rep))[:40] == b"VPCIRC01" + struct.pack("<QQ", n, 3) + raw[24:40]   # template + K


def test_digest_word_reduction_edge_words(tmp_path):
    """fp_mod (field.cuh, the device's digest-word reduction) == x % p for every 64-bit x, compiled for the host"""
    src = tmp_path / "fs_mod.cpp"
    src.write_text('#include "%s"\nextern "C" void h_mod(const vp::u64* x, vp::u64* o, int n) { for (int i = 0; i < n; ++i) o[i] = vp::fp_mod(x[i]); }\n'
                   % os.path.join(ROOT, "virgo-plus_b200", "csrc", "field.cuh"))
    so = tmp_path / "fs_mod.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", str(src), "-o", str(so)])
    import ctypes
    lib = ctypes.CDLL(str(so))
    edge = [0, P - 1, P, P + 1, 2 * P, (1 << 64) - (1 << 61) - 1, (1 << 64) - (1 << 61), 8 * P, (1 << 64) - 1, 7 * P + 6, 8 * P + 7,
            (1 << 63), (1 << 61), (1 << 62) - 1]
    rng = random.Random(5)
    words = np.array(edge + [rng.getrandbits(64) for _ in range(5000)], np.uint64)
    out = np.zeros_like(words)
    lib.h_mod(words.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), len(words))
    want = np.array([int(x) % P for x in words], np.uint64)
    assert (out == want).all(), [(int(w), int(o)) for w, o in zip(words, out) if int(o) != int(w) % P][:5]


def test_statement_binds_every_part_and_the_oracle_proof(B, O):
    """the statement changes with one input, one output, every single gate field, one dad_id entry, K and one context byte;
    the oracle's prove_fs(statement) is accepted under the statement and rejected under every changed one"""
    circ = all_types_circuit(B, 31).replicate(2)
    inputs, outputs = oracle_values(O, circ)
    d0 = describe(circ)
    cd0 = vector_root(circuit_bytes(d0))
    s0 = statement(cd0, inputs, outputs, CONTEXT)

    def with_desc(fn):
        d = copy.deepcopy(d0)
        fn(d)
        return statement(vector_root(circuit_bytes(d)), inputs, outputs, CONTEXT)

    changed = {}
    x = inputs.copy(); x[len(x) // 2]["re"] = (int(x[len(x) // 2]["re"]) + 1) % P
    changed["input"] = statement(cd0, x, outputs, CONTEXT)
    y = outputs.copy(); y[-1]["im"] = (int(y[-1]["im"]) + 1) % P
    changed["output"] = statement(cd0, inputs, y, CONTEXT)
    layer = 2
    for field in ("ty", "is_assert", "l", "u", "v", "lv"):
        def bump(d, field=field):
            d["gates"][layer][field][1] += 1
        changed[f"gate.{field}"] = with_desc(bump)
    for part in ("re", "im"):
        def bump_c(d, part=part):
            d["gates"][layer]["c"][part][1] += 1
        changed[f"gate.c.{part}"] = with_desc(bump_c)
    src = next((i, s) for i in range(1, d0["n"]) for s in range(i) if len(d0["dads"][i][s]))

    def bump_dad(d):
        d["dads"][src[0]][src[1]][0] += 1
    changed["dad_id"] = with_desc(bump_dad)
    rep3 = all_types_circuit(B, 31).replicate(3)
    changed["K"] = statement(vector_root(circuit_bytes(describe(rep3))), inputs, outputs, CONTEXT)
    ctx = bytearray(CONTEXT); ctx[31] ^= 1
    changed["context"] = statement(cd0, inputs, outputs, bytes(ctx))
    assert len(set(changed.values()) | {s0}) == len(changed) + 1, "two statements collide"
    oc = O.OracleCircuit(circ.expand().flat())
    tr, _ = oc.prove_fs(s0)
    assert oc.verify_fs(s0, tr) == (True, 0, 0)
    for what, s in changed.items():
        assert not oc.verify_fs(s, tr)[0], f"a proof under the statement verified with a changed {what}"


# ------------------------------------------------------------------ GPU
def _gpu_cases(B, sha_circuit):
    yield "sha256_64", sha_circuit
    yield "sha256_64_x3", sha_circuit.replicate(3)
    yield "sha256_64_x33", sha_circuit.replicate(33)
    for name in ("small_allops", "small_chain", "small_notquirk", "small_random_a", "small_random_b", "small_random_c"):
        yield name, _golden_pws(B, name)
    yield "all_types_x5", all_types_circuit(B, 41).replicate(5)
    yield "one_gate_layers", one_gate_layers_circuit(B, 43)


def _bump(tr, k, part="re"):
    t = tr.copy()
    t[k][part] = (int(t[k][part]) + 1) % P
    return t


@pytest.mark.gpu
def test_statement_digest_matches_python(B, O, sha_circuit):
    for name, circ in _gpu_cases(B, sha_circuit):
        p = B.Prover(circ)
        got = p.statement_digest(CONTEXT)
        n = circ.n_layers
        inputs, outputs = p.values(0), p.values(n - 1)
        if circ.total_gates < 2_000_000:
            want_in, want_out = oracle_values(O, circ)
            assert (inputs == want_in).all() and (outputs == want_out).all(), name
        want = digests(circ, inputs, outputs, CONTEXT)
        for k in ("circuit", "inputs", "outputs", "statement"):
            assert got[k] == want[k], f"{name}: {k} digest differs"
        assert p.statement_digest(bytes(32))["statement"] == digests(circ, inputs, outputs, bytes(32))["statement"], name
        p.close()


@pytest.mark.gpu
def test_prove_fs_bound_matches_oracle_and_prove_fs(B, O, sha_circuit):
    for name, circ in _gpu_cases(B, sha_circuit):
        p = B.Prover(circ)
        tr, ch, st = p.prove_fs_bound(CONTEXT)
        assert st == p.statement_digest(CONTEXT)["statement"], name
        tr2, ch2 = p.prove_fs(st)
        assert (tr == tr2).all() and (ch == ch2).all(), f"{name}: vp_prove_fs(statement) != vp_prove_fs_bound"
        oc = O.OracleCircuit((circ.expand() if circ.instances > 1 else circ).flat())
        want_tr, want_ch = oc.prove_fs(st)
        assert (tr == want_tr).all(), f"{name}: transcript != oracle prove_fs(statement)"
        assert (ch == want_ch).all(), f"{name}: challenges != oracle prove_fs(statement)"
        assert p.verify_fs_bound(CONTEXT, p.values(circ.n_layers - 1), tr) == (True, 0, 0), name
        p.close()


@pytest.mark.gpu
def test_prove_fs_bound_random_pws_sample(B, O):
    """a seeded sample of tools/gpu_diff_campaign.py's random .pws circuits (1-gate layers, every parser gate type) x K"""
    mg = _make_golden()
    for seed in range(900, 912):
        rng = random.Random(seed * 104729)
        n_in = rng.choice([3, 8, 17, 64, 200, 257, 1000])
        n_g = rng.choice([1, 2, 7, 30, 120, 500, 2000])
        K = rng.choice([1, 1, 2, 3, 5, 8, 13, 33])
        circ = B.Circuit.from_pws_text(mg.random_pws(seed, n_in, n_g))
        if K > 1:
            circ = circ.replicate(K)
        p = B.Prover(circ)
        tr, ch, st = p.prove_fs_bound(CONTEXT)
        want_tr, want_ch = O.OracleCircuit((circ.expand() if K > 1 else circ).flat()).prove_fs(st)
        assert (tr == want_tr).all() and (ch == want_ch).all(), f"seed {seed}"
        assert p.verify_fs_bound(CONTEXT, p.values(circ.n_layers - 1), tr) == (True, 0, 0), f"seed {seed}"
        p.close()


def _message_positions(circ):
    """transcript index of Vres, a phase-1 / phase-2 / Liu coefficient, claim_u, claims_v, claim_liu and the input MLE"""
    n = circ.n_layers
    ti, pos = 1, {"Vres": 0}
    for i in range(n - 1, 0, -1):
        pb, m = circ.bit_length(i - 1), circ.max_dad_bit_length(i)
        if pb > 0 and "phase1" not in pos:
            pos["phase1"] = ti + 1
        ti += 3 * pb
        pos.setdefault("claim_u", ti)
        ti += 1
        if m != -1:
            if m > 0 and "phase2" not in pos:
                pos["phase2"] = ti + 2
            ti += 3 * m
            pos.setdefault("claims_v", ti + i - 1)
            ti += i
        if pb > 0 and "liu" not in pos:
            pos["liu"] = ti
        ti += 3 * pb
        pos.setdefault("claim_liu", ti)
        ti += 1
    pos["input_mle"] = ti
    assert ti + 1 == circ.transcript_len
    return pos


@pytest.mark.gpu
def test_verify_fs_bound_verdicts(B, sha_circuit):
    for circ in (sha_circuit, all_types_circuit(B, 51).replicate(4)):
        n = circ.n_layers
        p = B.Prover(circ)
        tr, _, st = p.prove_fs_bound(CONTEXT)
        outputs = p.values(n - 1)
        v = B.Prover(circ)                      # the verifier's own context: same circuit, same inputs
        assert v.verify_fs_bound(CONTEXT, outputs, tr) == (True, 0, 0)
        pos = _message_positions(circ)
        assert set(pos) == {"Vres", "phase1", "phase2", "liu", "claim_u", "claims_v", "claim_liu", "input_mle"}
        for what, k in pos.items():
            ok, code, _ = v.verify_fs_bound(CONTEXT, outputs, _bump(tr, k))
            assert not ok, f"+1 on {what} accepted"
            if what == "Vres":
                assert code == 8
        ctx = bytearray(CONTEXT); ctx[0] ^= 0x80
        assert not v.verify_fs_bound(bytes(ctx), outputs, tr)[0]
        assert v.verify_fs_bound(CONTEXT, _bump(outputs, len(outputs) // 3, "im"), tr)[:2] == (False, 8)
        x = circ.inputs().copy()
        x[1] = (int(x[1]) + 1) % P
        w = B.Prover(circ)
        w.set_inputs(x)
        assert not w.verify_fs_bound(CONTEXT, outputs, tr)[0]
        w.close()
        unrelated, _ = p.prove_fs(bytes(range(32)))
        assert not v.verify_fs_bound(CONTEXT, outputs, unrelated)[0]
        bad = tr.copy()
        bad[3]["re"] = P
        assert v.verify_fs_bound(CONTEXT, outputs, bad)[:2] == (False, 7)
        with pytest.raises(B.VpError):
            v.verify_fs_bound(CONTEXT, outputs[:-1], tr)
        o = outputs.copy(); o[0]["re"] = P
        with pytest.raises(B.VpError):
            v.verify_fs_bound(CONTEXT, o, tr)
        p.close()
        v.close()


@pytest.mark.gpu
def test_bound_proof_leaves_the_context_consistent(B, sha_circuit):
    """vp_prove -> vp_prove_fs_bound -> vp_prove -> vp_prove_fs on one context == each on a fresh context; lanes 1 and 6
    give the same Fiat-Shamir bits; no per-round launches"""
    circ = sha_circuit.replicate(3)
    inputs, chal = circ.inputs(), circ.draw_challenges()

    def fresh(fn):
        q = B.Prover(circ)
        r = fn(q)
        q.close()
        return r

    want_prove = fresh(lambda q: q.prove(inputs=inputs, challenges=chal))
    want_bound = fresh(lambda q: q.prove_fs_bound(CONTEXT))
    seed = bytes(range(1, 33))
    want_fs = fresh(lambda q: q.prove_fs(seed))
    p = B.Prover(circ)
    assert (p.prove(inputs=inputs, challenges=chal) == want_prove).all()
    tr, ch, st = p.prove_fs_bound(CONTEXT)
    assert (tr == want_bound[0]).all() and (ch == want_bound[1]).all() and st == want_bound[2]
    assert p.verify(tr) == (True, 0, 0)        # the context holds the challenges the proof drew
    assert (p.prove(inputs=inputs, challenges=chal) == want_prove).all()
    tr2, ch2 = p.prove_fs(seed)
    assert (tr2 == want_fs[0]).all() and (ch2 == want_fs[1]).all()
    for lanes in (1, 6):
        p.set_lanes(lanes)
        t, c, s = p.prove_fs_bound(CONTEXT)
        assert (t == want_bound[0]).all() and (c == want_bound[1]).all() and s == st, lanes
    # launches: at most a one-lane vp_prove plus 4 per layer plus 8
    p.set_lanes(1)
    p.prove(inputs=inputs, challenges=chal)
    base = p.last_prove_launches
    p.prove_fs_bound(CONTEXT)
    n = circ.n_layers
    assert p.last_prove_launches <= base + 4 * n + 8, (p.last_prove_launches, base)
    stamps = p.fs_round_stamps()
    rounds = sum(2 * circ.bit_length(i - 1) + max(circ.max_dad_bit_length(i), 0) for i in range(1, n))
    assert stamps.shape == (rounds, 4) and (np.diff(stamps.astype(np.int64), axis=1) >= 0).all()
    p.close()


@pytest.mark.gpu
def test_statement_and_bound_proof_at_c3_size(B, sha_circuit):
    """SHA256_64 x 1024 (the C3 benchmark shape): the digests equal the restatement over vp_get_values, the device
    verifier accepts the bound proof and rejects it with one changed element"""
    circ = sha_circuit.replicate(1024)
    p = B.Prover(circ)
    got = p.statement_digest(CONTEXT)
    n = circ.n_layers
    outputs = p.values(n - 1)
    want = digests(circ, p.values(0), outputs, CONTEXT)
    assert got == want
    tr, _, st = p.prove_fs_bound(CONTEXT)
    assert st == want["statement"]
    assert p.verify_fs_bound(CONTEXT, outputs, tr) == (True, 0, 0)
    assert not p.verify_fs_bound(CONTEXT, outputs, _bump(tr, len(tr) // 2))[0]
    p.close()
