"""vp_prove_fs_bound_batch: B independent statement-bound proofs of one circuit in one device pass.

Every proof of a batch must be, bit for bit, the single proof vp_prove_fs_bound gives after vp_set_inputs(inputs_b) with
context b; the batch must not disturb the context's resident state and must not launch more kernels as B grows."""
import random

import numpy as np
import pytest

from test_fs_statement import ADD, CONTEXT, F_DTYPE, INPUT, P, SUB, _golden_pws, _make_golden, all_types_circuit, one_gate_layers_circuit


def _contexts(B_, seed):
    rng = random.Random(seed)
    return [bytes(rng.randrange(256) for _ in range(32)) for _ in range(B_)]


def _inputs(circ, n, seed):
    """n distinct seeded input vectors. Bits are flipped in a few places of the circuit's own inputs, which keeps 0/1
    inputs 0/1 (the circuits' assert gates hold for any value)."""
    base = np.asarray(circ.inputs(), dtype=np.uint64)
    rng = np.random.default_rng(seed)
    out = np.repeat(base[None, :], n, axis=0)
    for b in range(n):
        idx = rng.choice(len(base), size=min(8, len(base)), replace=False)
        for i in idx:
            x = int(out[b, i])
            out[b, i] = 1 - x if x in (0, 1) else int(rng.integers(0, P))
    return out


def _singles(B, circ, inputs, contexts):
    p = B.Prover(circ)
    res = []
    for x, c in zip(inputs, contexts):
        p.set_inputs(x)
        res.append(p.prove_fs_bound(c))
    p.close()
    return res


def _check_batch(B, circ, sizes, seed, name):
    p = B.Prover(circ)
    for n in sizes:
        x = _inputs(circ, n, seed + n)
        ctx = _contexts(n, seed + n)
        tr, ch, st = p.prove_fs_bound_batch(x, ctx)
        assert tr.shape == (n, circ.transcript_len) and ch.shape == (n, circ.challenge_count) and st.shape == (n, 32)
        for b, (tr1, ch1, st1) in enumerate(_singles(B, circ, x, ctx)):
            assert st[b].tobytes() == st1, f"{name} B={n}: statement {b}"
            assert (tr[b] == tr1).all(), f"{name} B={n}: transcript {b}"
            assert (ch[b] == ch1).all(), f"{name} B={n}: challenges {b}"
    p.close()


def _batch_cases(B, sha_circuit):
    yield "sha256_64", sha_circuit
    yield "sha256_64_x3", sha_circuit.replicate(3)
    for name in ("small_allops", "small_chain", "small_notquirk", "small_random_a", "small_random_b", "small_random_c"):
        yield name, _golden_pws(B, name)
    yield "all_types", all_types_circuit(B, 41)
    yield "all_types_x5", all_types_circuit(B, 41).replicate(5)
    yield "one_gate_layers", one_gate_layers_circuit(B, 43)
    mg = _make_golden()
    for seed in (901, 905):
        rng = random.Random(seed * 104729)
        n_in = rng.choice([3, 8, 17, 64, 200, 257, 1000])
        n_g = rng.choice([1, 2, 7, 30, 120, 500, 2000])
        yield f"random_pws_{seed}", B.Circuit.from_pws_text(mg.random_pws(seed, n_in, n_g)).replicate(2)


# ------------------------------------------------------------------ CPU
def test_batch_binding_rejects_bad_shapes_before_the_library(B, sha_circuit, monkeypatch):
    n_in = sha_circuit.layer_size(0) * sha_circuit.instances

    class _Circuit:   # the shape of sha_circuit, without the library
        instances = sha_circuit.instances
        transcript_len = sha_circuit.transcript_len
        challenge_count = sha_circuit.challenge_count

        def layer_size(self, i):
            return n_in // self.instances

    p = B.Prover.__new__(B.Prover)   # no device context: the checks must fire before any library call
    p.circuit, p.h = _Circuit(), None
    called = []

    def no_lib():
        called.append(1)
        raise AssertionError("library called")

    monkeypatch.setattr(B, "lib", no_lib)
    good = np.zeros((2, n_in), np.uint64)
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(np.zeros(n_in, np.uint64), [bytes(32)])            # 1-D inputs
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(np.zeros((2, n_in - 1), np.uint64), [bytes(32)] * 2)   # short rows
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(np.zeros((0, n_in), np.uint64), [])                # B = 0
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(good.astype(np.float64), [bytes(32)] * 2)          # not integers
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(good, [bytes(32)])                                 # one context for two statements
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(good, [bytes(32), bytes(31)])                      # a short context
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(good, np.zeros((2, 31), np.uint8))                 # context array of the wrong shape
    with pytest.raises(ValueError):
        p.prove_fs_bound_batch(good, np.zeros((2, 32), np.int32))                 # context array of the wrong type
    assert not called


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_batch_is_bit_identical_to_single_proofs(B, sha_circuit):
    for name, circ in _batch_cases(B, sha_circuit):
        _check_batch(B, circ, (1, 2, 3, 7, 64), 17, name)


@pytest.mark.gpu
def test_batch_matches_the_oracle(B, O, sha_circuit):
    circ = all_types_circuit(B, 47).replicate(3)
    x, ctx = _inputs(circ, 5, 3), _contexts(5, 3)
    p = B.Prover(circ)
    tr, ch, st = p.prove_fs_bound_batch(x, ctx)
    p.close()
    for b in range(5):
        circ.set_inputs(x[b])
        want_tr, want_ch = O.OracleCircuit(circ.expand().flat()).prove_fs(st[b].tobytes())
        assert (tr[b] == want_tr).all() and (ch[b] == want_ch).all(), f"statement {b}"


@pytest.mark.gpu
def test_batch_larger_than_the_phase_grid_runs_in_chunks(B, sha_circuit):
    n = 600   # > 148 SMs x 2 co-resident blocks of the phase kernel on a B200, and > 512
    x, ctx = _inputs(sha_circuit, n, 5), _contexts(n, 5)
    p = B.Prover(sha_circuit)
    tr, ch, st = p.prove_fs_bound_batch(x, ctx)
    p.close()
    sample = [0, 1, 295, 296, 297, 591, 592, 599]
    singles = _singles(B, sha_circuit, x[sample], [ctx[b] for b in sample])
    for b, (tr1, ch1, st1) in zip(sample, singles):
        assert st[b].tobytes() == st1 and (tr[b] == tr1).all() and (ch[b] == ch1).all(), f"statement {b}"


@pytest.mark.gpu
def test_batch_statements_are_independent(B, sha_circuit):
    x = _inputs(sha_circuit, 1, 9)
    xs = np.repeat(x, 3, axis=0)
    ctx = [CONTEXT, CONTEXT, bytes(32)]
    p = B.Prover(sha_circuit)
    tr, ch, st = p.prove_fs_bound_batch(xs, ctx)
    assert st[0].tobytes() == st[1].tobytes() and (tr[0] == tr[1]).all() and (ch[0] == ch[1]).all()
    assert st[0].tobytes() != st[2].tobytes() and not (tr[0] == tr[2]).all()
    p.close()


@pytest.mark.gpu
def test_verifier_accepts_each_proof_of_a_batch(B, sha_circuit):
    n = 8
    x, ctx = _inputs(sha_circuit, n, 11), _contexts(n, 11)
    p = B.Prover(sha_circuit)
    tr, _, _ = p.prove_fs_bound_batch(x, ctx)
    outs = []
    v = B.Prover(sha_circuit)
    for b in range(n):
        v.set_inputs(x[b])
        v.evaluate()
        outs.append(v.values(sha_circuit.n_layers - 1))
        assert v.verify_fs_bound(ctx[b], outs[b], tr[b]) == (True, 0, 0), f"statement {b}"
    bad = tr.copy()
    bad["re"][3, 5] = (int(bad["re"][3, 5]) + 1) % P
    for b in (2, 3, 4):
        v.set_inputs(x[b])
        ok = v.verify_fs_bound(ctx[b], outs[b], bad[b])[0]
        assert ok == (b != 3), f"statement {b}"
    v.close()
    p.close()


def _same(a, b):
    return all((x == y).all() if hasattr(x, "all") else x == y for x, y in zip(a, b))


@pytest.mark.gpu
def test_batch_leaves_the_context_untouched(B, sha_circuit):
    circ = sha_circuit.replicate(3)
    inputs, chal = circ.inputs(), circ.draw_challenges()
    p = B.Prover(circ)
    fs0 = p.prove_fs_bound(CONTEXT)
    vals0 = p.values(circ.n_layers - 1)
    p.prove_fs_bound_batch(_inputs(circ, 4, 13), _contexts(4, 13))
    assert (p.values(circ.n_layers - 1) == vals0).all()
    assert p.verify(fs0[0]) == (True, 0, 0)   # the resident challenges are still those of the last single proof
    assert _same(p.prove_fs_bound(CONTEXT), fs0)
    tr0 = p.prove(inputs=inputs, challenges=chal)
    ver0 = p.verify(tr0)
    p.prove_fs_bound_batch(_inputs(circ, 3, 14), _contexts(3, 14))
    assert p.verify(tr0) == ver0 == (True, 0, 0)
    assert (p.prove(inputs=inputs, challenges=chal) == tr0).all()
    assert _same(p.prove_fs_bound(CONTEXT), fs0)
    p.close()


# the batch adds no launch per statement; it may add this many over a single bound proof (the contexts' upload is a copy)
EXTRA_LAUNCHES = 0


@pytest.mark.gpu
def test_batch_launches_do_not_grow_with_B(B, sha_circuit):
    p = B.Prover(sha_circuit)
    p.prove_fs_bound(CONTEXT)
    p.prove_fs_bound(CONTEXT)
    single = p.last_prove_launches
    counts = {}
    for n in (1, 8, 1, 8):
        p.prove_fs_bound_batch(_inputs(sha_circuit, n, 1), _contexts(n, 1))
        counts[n] = p.last_prove_launches
    assert counts[8] == counts[1]
    assert counts[1] <= single + EXTRA_LAUNCHES
    p.close()


def _assert_circuit(B):
    """layer 1 gate 0 = Sub(x0, x1) is an assert gate: it holds exactly when the first two inputs are equal"""
    sizes = [4, 2]
    ty = [INPUT] * 4 + [SUB, ADD]
    l = [-1] * 4 + [0, 0]
    u = [7, 7, 3, 9, 0, 2]
    v = [0] * 4 + [1, 3]
    asr = [0] * 4 + [1, 0]
    return B.Circuit.from_arrays(sizes, ty, l, u, v, c=np.zeros(6, F_DTYPE), is_assert=asr)


@pytest.mark.gpu
def test_batch_errors_leave_the_context_usable(B):
    circ = _assert_circuit(B).replicate(2)
    n = 8
    rng = np.random.default_rng(4)
    xs = rng.integers(0, P, size=(n, circ.num_inputs), dtype=np.uint64)
    xs[:, 1::4] = xs[:, 0::4]   # every instance's assert holds ...
    p = B.Prover(circ)
    p.set_inputs(xs[0])
    ref = p.prove_fs_bound(CONTEXT)
    ctx = _contexts(n, 2)
    ctx_arr = np.frombuffer(b"".join(ctx), np.uint8)
    tr = np.zeros((n, circ.transcript_len), F_DTYPE)
    ch = np.zeros((n, circ.challenge_count), F_DTYPE)

    def raw(B_, x, n_inputs, cap, ch_cap):
        return B.lib().vp_prove_fs_bound_batch(p.h, B_, B._ptr(x), n_inputs, B._ptr(ctx_arr), B._ptr(tr), cap, B._ptr(ch), ch_cap, None)

    assert raw(n, xs, xs.size, tr.size, ch.size) == 0
    VP_ERR_ARG = raw(0, xs, 0, tr.size, ch.size)
    assert VP_ERR_ARG != 0
    assert raw(n, xs, xs.size - 1, tr.size, ch.size) == VP_ERR_ARG
    assert raw(n, xs, xs.size, tr.size - 1, ch.size) == VP_ERR_ARG
    assert raw(n, xs, xs.size, tr.size, ch.size - 1) == VP_ERR_ARG
    bad = xs.copy()
    bad[6, 2] = P
    with pytest.raises(B.VpError) as e:
        p.prove_fs_bound_batch(bad, ctx)
    assert e.value.code == VP_ERR_ARG
    broken = xs.copy()
    broken[5, 5] = (int(broken[5, 4]) + 1) % P   # ... except in instance 1 of statement 5
    broken[7, 1] = (int(broken[7, 0]) + 1) % P   # ... and statement 7: the error names the first
    with pytest.raises(B.VpError) as e:
        p.prove_fs_bound_batch(broken, ctx)
    assert e.value.code != VP_ERR_ARG and "statement 5:" in str(e.value)
    assert _same(p.prove_fs_bound(CONTEXT), ref)
    tr2, ch2, st2 = p.prove_fs_bound_batch(xs, ctx)
    assert (tr2 == tr).all() and (ch2 == ch).all()
    p.close()
