"""Aggregate statement-bound proofs (vp_prove_fs_aggregate, include/virgo_b200.h): one Fiat-Shamir proof of B statements of
one circuit, statement b being instances [b K, (b + 1) K) with its own context. A pure-Python restatement of the aggregate
checked on hand-built statements; on the device, every statement equal to the single bound statement of a K-instance
context holding its inputs, the proof bit for bit vp_prove_fs(aggregate) and the oracle's prove_fs(aggregate), and the
verifier's verdicts."""
import ctypes
import random
import struct

import numpy as np
import pytest

from test_fs_batch import _assert_circuit
from test_fs_statement import (CONTEXT, F_DTYPE, P, H, _bump, _golden_pws, _make_golden, _message_positions, all_types_circuit,
                               circuit_bytes, describe, one_gate_layers_circuit, statement, vector_root)

VP_ERR_ARG, VP_ERR_ASSERT = -1, -4


# ------------------------------------------------------------------ the restatement
def aggregate(statements):
    """H("VPAGGR01" | u64 B | R(statement_0 | ... | statement_{B-1})): 48 bytes hashed"""
    statements = [bytes(s) for s in statements]
    assert all(len(s) == 32 for s in statements)
    return H(b"VPAGGR01" + struct.pack("<Q", len(statements)) + vector_root(b"".join(statements)))


def k_circuit(template, K):
    """template + K: the circuit of a statement of K instances (the template itself when K = 1)"""
    return template.replicate(K) if K > 1 else template


def statements_of(template, inputs, outputs, B, contexts):
    """statement b over slice b of the inputs / outputs (field-element arrays of the whole N-instance circuit)"""
    K_circ = k_circuit(template, len(inputs) // B // template.layer_size(0))
    cd = vector_root(circuit_bytes(describe(K_circ)))
    ni, no = len(inputs) // B, len(outputs) // B
    return [statement(cd, inputs[b * ni:(b + 1) * ni], outputs[b * no:(b + 1) * no], contexts[b]) for b in range(B)]


def _contexts(n, seed):
    rng = random.Random(seed)
    return [bytes(rng.randrange(256) for _ in range(32)) for _ in range(n)]


# ------------------------------------------------------------------ CPU
def test_aggregate_restatement_hand_built():
    s = [bytes((7 * i + 11 * b + 1) % 256 for i in range(32)) for b in range(3)]
    head = lambda n: b"VPAGGR01" + struct.pack("<Q", n)
    assert len(head(1) + bytes(32)) == 48
    # B = 1: one 64-byte leaf, the statement zero-padded
    assert aggregate(s[:1]) == H(head(1) + H(s[0] + bytes(32)))
    # B = 2: the two statements fill one leaf
    assert aggregate(s[:2]) == H(head(2) + H(s[0] + s[1]))
    # B = 3: two leaves, the second zero-padded
    assert aggregate(s) == H(head(3) + H(H(s[0] + s[1]) + H(s[2] + bytes(32))))
    # domain-separated from the statement itself
    assert aggregate(s[:1]) != s[0]
    # B is hashed: [s0] and [s0, 0^32] have the same vector root
    assert vector_root(s[0]) == vector_root(s[0] + bytes(32))
    assert aggregate(s[:1]) != aggregate([s[0], bytes(32)])
    # order and every byte of every statement
    assert aggregate([s[1], s[0], s[2]]) != aggregate(s)
    assert aggregate([s[0], s[2], s[1]]) != aggregate(s)
    for b in range(3):
        for i in (0, 17, 31):
            t = [bytearray(x) for x in s]
            t[b][i] ^= 1
            assert aggregate(t) != aggregate(s), (b, i)


class _Circuit:   # the shape of a 6-instance circuit, without the library
    instances = 6
    n_layers = 3
    transcript_len = 40
    challenge_count = 20

    def layer_size(self, i):
        return (5, 4, 2)[i]


def test_aggregate_binding_rejects_bad_arguments_before_the_library(B, monkeypatch):
    p = B.Prover.__new__(B.Prover)   # no device context: the checks must fire before any library call
    p.circuit, p.h = _Circuit(), None
    called = []

    def no_lib():
        called.append(1)
        raise AssertionError("library called")

    monkeypatch.setattr(B, "lib", no_lib)
    ctx3 = [bytes(32)] * 3
    out = np.zeros(6 * 2, F_DTYPE)
    tr = np.zeros(40, F_DTYPE)
    for fn in (lambda Bn, c: p.aggregate_digest(Bn, c), lambda Bn, c: p.prove_fs_aggregate(Bn, c),
               lambda Bn, c: p.verify_fs_aggregate(Bn, c, out, tr)):
        with pytest.raises(ValueError):
            fn(3, [bytes(32)] * 2)                    # two contexts for three statements
        with pytest.raises(ValueError):
            fn(3, [bytes(32)] * 2 + [bytes(31)])      # a short context
        with pytest.raises(ValueError):
            fn(3, np.zeros((3, 31), np.uint8))        # context array of the wrong shape
        with pytest.raises(ValueError):
            fn(4, [bytes(32)] * 4)                    # 4 does not divide 6
        with pytest.raises(ValueError):
            fn(0, [])                                 # B = 0
        with pytest.raises(ValueError):
            fn(12, [bytes(32)] * 12)                  # more statements than instances
        with pytest.raises(ValueError):
            fn(2.0, [bytes(32)] * 2)                  # not an integer
    with pytest.raises(ValueError):
        p.verify_fs_aggregate(3, ctx3, out[:-1], tr)                   # short outputs
    with pytest.raises(ValueError):
        p.verify_fs_aggregate(3, ctx3, out.reshape(3, 4), tr)          # outputs of the wrong shape
    with pytest.raises(ValueError):
        p.verify_fs_aggregate(3, ctx3, np.zeros(12, np.uint64), tr)    # outputs that are not field elements
    with pytest.raises(ValueError):
        p.verify_fs_aggregate(3, ctx3, out, tr[:-1])                   # short transcript
    with pytest.raises(ValueError):
        p.verify_fs_aggregate(3, ctx3, out, np.zeros((2, 20), F_DTYPE))   # transcript of the wrong shape
    assert not called


# ------------------------------------------------------------------ GPU
def _cases(B, sha_circuit):
    """(name, template, N, statement counts B | N) at sizes the oracle proves"""
    for N in (1, 2, 3, 8):
        yield f"sha256_64_x{N}", sha_circuit, N, [d for d in range(1, N + 1) if N % d == 0]
    for name in ("small_allops", "small_chain"):
        yield f"{name}_x6", _golden_pws(B, name), 6, [2, 3, 6]
    yield "all_types_x6", all_types_circuit(B, 61), 6, [1, 2, 3, 6]
    yield "one_gate_layers_x4", one_gate_layers_circuit(B, 63), 4, [1, 2, 4]
    mg = _make_golden()
    for seed in range(920, 926):
        rng = random.Random(seed * 7919)
        n_in = rng.choice([3, 8, 17, 64, 200, 257])
        n_g = rng.choice([1, 2, 7, 30, 120, 500])
        N = rng.choice([2, 3, 4, 6])
        yield f"random_pws_{seed}_x{N}", B.Circuit.from_pws_text(mg.random_pws(seed, n_in, n_g)), N, \
            sorted({rng.choice([d for d in range(1, N + 1) if N % d == 0]) for _ in range(2)})


def _single_statement(B, template, K, inputs, context):
    """vp_statement_digest on a fresh context of template + K holding `inputs`"""
    q = B.Prover(k_circuit(template, K))
    q.set_inputs(inputs)
    s = q.statement_digest(context)["statement"]
    q.close()
    return s


@pytest.mark.gpu
def test_aggregate_statements_and_proof(B, O, sha_circuit):
    for name, template, N, Bs in _cases(B, sha_circuit):
        circ = k_circuit(template, N)
        x = np.asarray(circ.inputs(), dtype=np.uint64)
        S0, n = template.layer_size(0), circ.n_layers
        oc = O.OracleCircuit((circ.expand() if N > 1 else circ).flat())
        p = B.Prover(circ)
        p.evaluate()
        vals_in, vals_out = p.values(0), p.values(n - 1)
        for Bn in Bs:
            K = N // Bn
            ctx = _contexts(Bn, 1000 * N + Bn)
            st, agg = p.aggregate_digest(Bn, ctx)
            want = statements_of(template, vals_in, vals_out, Bn, ctx)
            for b in range(Bn):
                assert st[b].tobytes() == want[b], f"{name} B={Bn}: statement {b} != restatement"
                assert st[b].tobytes() == _single_statement(B, template, K, x[b * K * S0:(b + 1) * K * S0], ctx[b]), \
                    f"{name} B={Bn}: statement {b} != vp_statement_digest of a K-instance context"
            assert agg == aggregate(want), f"{name} B={Bn}: aggregate"
            tr, ch, st2, agg2 = p.prove_fs_aggregate(Bn, ctx)
            assert (st2 == st).all() and agg2 == agg, f"{name} B={Bn}"
            tr1, ch1 = p.prove_fs(agg)
            assert (tr == tr1).all() and (ch == ch1).all(), f"{name} B={Bn}: != vp_prove_fs(aggregate)"
            want_tr, want_ch = oc.prove_fs(agg)
            assert (tr == want_tr).all() and (ch == want_ch).all(), f"{name} B={Bn}: != oracle prove_fs(aggregate)"
            assert p.verify_fs_aggregate(Bn, ctx, vals_out, tr) == (True, 0, 0), f"{name} B={Bn}"
        p.close()


def _raw(B, fn, *args):
    """a library call past the binding's own checks, through the binding's error path -> the VpError's status"""
    with pytest.raises(B.VpError) as e:
        B._ck(getattr(B.lib(), fn)(*args))
    return e.value.code


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.mark.gpu
def test_aggregate_verdicts(B, sha_circuit):
    for circ, Bn in ((sha_circuit.replicate(8), 4), (all_types_circuit(B, 51).replicate(6), 3)):
        N, n = circ.instances, circ.n_layers
        K, S0, So = N // Bn, circ.layer_size(0), circ.layer_size(n - 1)
        ctx = _contexts(Bn, 77)
        p = B.Prover(circ)
        tr, ch, st, agg = p.prove_fs_aggregate(Bn, ctx)
        outputs = p.values(n - 1)
        v = B.Prover(circ)   # the verifier's own context: same circuit, same inputs
        assert v.verify_fs_aggregate(Bn, ctx, outputs, tr) == (True, 0, 0)
        pos = _message_positions(circ)
        for what, k in pos.items():
            ok, code, _ = v.verify_fs_aggregate(Bn, ctx, outputs, _bump(tr, k))
            assert not ok, f"+1 on {what} accepted"
            if what == "Vres":
                assert code == 8
        for b in (0, Bn - 1):
            c = [bytearray(x) for x in ctx]
            c[b][5] ^= 0x10
            assert not v.verify_fs_aggregate(Bn, [bytes(x) for x in c], outputs, tr)[0], f"context {b} flipped"
        swapped = list(ctx)
        swapped[0], swapped[1] = swapped[1], swapped[0]
        assert not v.verify_fs_aggregate(Bn, swapped, outputs, tr)[0], "contexts swapped"
        x = np.asarray(circ.inputs(), dtype=np.uint64)
        a, b_ = x[:K * S0].copy(), x[K * S0:2 * K * S0].copy()
        assert (a != b_).any()
        y = x.copy()
        y[:K * S0], y[K * S0:2 * K * S0] = b_, a
        w = B.Prover(circ)
        w.set_inputs(y)
        assert not w.verify_fs_aggregate(Bn, ctx, outputs, tr)[0], "input slices swapped"
        w.close()
        o = outputs.copy()
        o[(Bn - 1) * K * So]["re"] = (int(o[(Bn - 1) * K * So]["re"]) + 1) % P
        assert not v.verify_fs_aggregate(Bn, ctx, o, tr)[0], "one statement's output changed"
        for other in (d for d in range(1, N + 1) if N % d == 0 and d != Bn):
            assert not v.verify_fs_aggregate(other, _contexts(other, 77), outputs, tr)[0], f"accepted with B = {other}"
        bad = tr.copy()
        bad[3]["im"] = P
        assert v.verify_fs_aggregate(Bn, ctx, outputs, bad)[:2] == (False, 7)
        # argument errors from the library itself (past the binding's checks) raise VpError(VP_ERR_ARG)
        c = np.frombuffer(b"".join(ctx), np.uint8).copy()
        a_, c_, l_ = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
        refs = (ctypes.byref(a_), ctypes.byref(c_), ctypes.byref(l_))
        big = np.zeros(70000 * 32, np.uint8)
        non_div = next(d for d in range(2, N + 2) if N % d)
        for Bx, cx in ((0, c), (non_div, big), (70000, big)):
            assert _raw(B, "vp_verify_fs_aggregate", v.h, Bx, _vp(cx), _vp(outputs), outputs.size, _vp(tr), tr.size, *refs) == VP_ERR_ARG
            assert _raw(B, "vp_aggregate_digest", v.h, Bx, _vp(cx), None, _vp(np.zeros(32, np.uint8))) == VP_ERR_ARG
        assert _raw(B, "vp_verify_fs_aggregate", v.h, Bn, _vp(c), _vp(outputs), outputs.size - 1, _vp(tr), tr.size, *refs) == VP_ERR_ARG
        assert _raw(B, "vp_verify_fs_aggregate", v.h, Bn, _vp(c), _vp(outputs), outputs.size, _vp(tr), tr.size - 1, *refs) == VP_ERR_ARG
        o = outputs.copy()
        o[0]["im"] = P
        assert _raw(B, "vp_verify_fs_aggregate", v.h, Bn, _vp(c), _vp(o), o.size, _vp(tr), tr.size, *refs) == VP_ERR_ARG
        t = np.zeros(len(tr), F_DTYPE)
        assert _raw(B, "vp_prove_fs_aggregate", p.h, Bn, _vp(c), _vp(t), t.size - 1, None, 0, None, None) == VP_ERR_ARG
        assert _raw(B, "vp_prove_fs_aggregate", p.h, Bn, _vp(c), _vp(t), t.size, _vp(ch), ch.size - 1, None, None) == VP_ERR_ARG
        assert _raw(B, "vp_prove_fs_aggregate", p.h, non_div, _vp(big), _vp(t), t.size, None, 0, None, None) == VP_ERR_ARG
        # ... and the contexts still prove and verify
        tr2, ch2, st2, agg2 = p.prove_fs_aggregate(Bn, ctx)
        assert (tr2 == tr).all() and (ch2 == ch).all() and (st2 == st).all() and agg2 == agg
        assert v.verify_fs_aggregate(Bn, ctx, outputs, tr) == (True, 0, 0)
        p.close()
        v.close()


@pytest.mark.gpu
def test_aggregate_proof_leaves_the_context_consistent(B, sha_circuit):
    """vp_prove -> vp_prove_fs_aggregate -> vp_prove -> vp_prove_fs_bound on one context == each on a fresh context; lanes 1
    and 6 give the same aggregate bits; vp_verify accepts the aggregate proof with the challenges it left resident"""
    circ = sha_circuit.replicate(6)
    inputs, chal = circ.inputs(), circ.draw_challenges()
    ctx = _contexts(3, 5)

    def fresh(fn):
        q = B.Prover(circ)
        r = fn(q)
        q.close()
        return r

    want_prove = fresh(lambda q: q.prove(inputs=inputs, challenges=chal))
    want_agg = fresh(lambda q: q.prove_fs_aggregate(3, ctx))
    want_bound = fresh(lambda q: q.prove_fs_bound(CONTEXT))
    p = B.Prover(circ)
    assert (p.prove(inputs=inputs, challenges=chal) == want_prove).all()
    tr, ch, st, agg = p.prove_fs_aggregate(3, ctx)
    assert (tr == want_agg[0]).all() and (ch == want_agg[1]).all() and (st == want_agg[2]).all() and agg == want_agg[3]
    assert p.verify(tr) == (True, 0, 0)
    assert p.last_prove_launches > 0 and p.last_prove_ms > 0
    assert (p.prove(inputs=inputs, challenges=chal) == want_prove).all()
    tr2, ch2, st2 = p.prove_fs_bound(CONTEXT)
    assert (tr2 == want_bound[0]).all() and (ch2 == want_bound[1]).all() and st2 == want_bound[2]
    for lanes in (1, 6):
        p.set_lanes(lanes)
        t, c, s, a = p.prove_fs_aggregate(3, ctx)
        assert (t == tr).all() and (c == ch).all() and (s == st).all() and a == agg, lanes
    p.close()


@pytest.mark.gpu
def test_aggregate_assert_failure(B):
    circ = _assert_circuit(B).replicate(4)
    rng = np.random.default_rng(9)
    x = rng.integers(0, P, size=circ.num_inputs, dtype=np.uint64)
    x[1::4] = x[0::4]   # every instance's assert holds ...
    p = B.Prover(circ)
    p.set_inputs(x)
    ctx = _contexts(2, 3)
    tr, _, _, agg = p.prove_fs_aggregate(2, ctx)
    assert p.verify_fs_aggregate(2, ctx, p.values(circ.n_layers - 1), tr) == (True, 0, 0)
    y = x.copy()
    y[3 * 4 + 1] = (int(y[3 * 4]) + 1) % P   # ... except instance 3's, in statement 1
    p.set_inputs(y)
    with pytest.raises(B.VpError) as e:
        p.prove_fs_aggregate(2, ctx)
    assert e.value.code == VP_ERR_ASSERT
    p.set_inputs(x)
    tr2, _, _, agg2 = p.prove_fs_aggregate(2, ctx)
    assert (tr2 == tr).all() and agg2 == agg
    p.close()


@pytest.mark.gpu
def test_aggregate_at_c3_size(B, sha_circuit):
    """SHA256_64 x 1024 (the C3 benchmark shape) with K = 1 and K = 16 per statement: the aggregate equals the restatement
    over vp_get_values, sampled statements equal vp_statement_digest of a K-instance context, the verifier accepts the
    proof and rejects it with one changed element"""
    circ = sha_circuit.replicate(1024)
    n, S0 = circ.n_layers, sha_circuit.layer_size(0)
    p = B.Prover(circ)
    p.evaluate()
    x = np.asarray(circ.inputs(), dtype=np.uint64)
    vals_in, vals_out = p.values(0), p.values(n - 1)
    for Bn in (1024, 64):
        K = 1024 // Bn
        ctx = _contexts(Bn, Bn)
        st, agg = p.aggregate_digest(Bn, ctx)
        want = statements_of(sha_circuit, vals_in, vals_out, Bn, ctx)
        assert [s.tobytes() for s in st] == want and agg == aggregate(want), Bn
        for b in (0, 1, Bn - 1):
            assert st[b].tobytes() == _single_statement(B, sha_circuit, K, x[b * K * S0:(b + 1) * K * S0], ctx[b]), (Bn, b)
        tr, _, st2, agg2 = p.prove_fs_aggregate(Bn, ctx)
        assert agg2 == agg and (st2 == st).all()
        assert p.verify_fs_aggregate(Bn, ctx, vals_out, tr) == (True, 0, 0)
        assert not p.verify_fs_aggregate(Bn, ctx, vals_out, _bump(tr, len(tr) // 2))[0]
    p.close()
