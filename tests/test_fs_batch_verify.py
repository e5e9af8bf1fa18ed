"""vp_verify_fs_bound_batch and vp_last_batch_outputs: B statement-bound proofs checked in one device pass, and the output
layers of a proving batch.

Verdict b of a batch must be exactly the single vp_verify_fs_bound verdict (accept, code, layer) on the same data, its
challenges those vp_fs_challenges derives; the batch must not disturb the context's resident state and must not launch
more kernels as B grows."""
import gc
import random

import numpy as np
import pytest

from test_fs_batch import _assert_circuit, _batch_cases, _contexts, _inputs, _same
from test_fs_statement import CONTEXT, F_DTYPE, P, _bump, _golden_pws, _make_golden, _message_positions, all_types_circuit


def _evaluated_outputs(B, circ, inputs):
    v = B.Prover(circ)
    out = []
    for x in inputs:
        v.set_inputs(x)
        v.evaluate()
        out.append(v.values(circ.n_layers - 1))
    v.close()
    return np.stack(out)


def _singles(B, circ, inputs, contexts, outputs, transcripts):
    """(accept, code, layer) of vp_verify_fs_bound for every statement, one call each"""
    v = B.Prover(circ)
    res = []
    for x, c, o, t in zip(inputs, contexts, outputs, transcripts):
        v.set_inputs(x)
        res.append(v.verify_fs_bound(c, o, t))
    v.close()
    return res


def _last_rounds(circ):
    """transcript index of the last round polynomial before layer n-1's final-value check (phase 2, or phase 1 when the
    layer has no phase 2) and of its last Liu round; None where the phase has no rounds"""
    n = circ.n_layers
    i = n - 1
    pb, m = circ.bit_length(i - 1), circ.max_dad_bit_length(i)
    ti = 1 + 3 * pb + 1   # Vres, phase 1, claim_u
    final = ti - 4 if pb > 0 else None
    if m != -1:
        if m > 0:
            final = ti + 3 * (m - 1)
        ti += 3 * m + i
    liu = ti + 3 * (pb - 1) if pb > 0 else None
    return final, liu


def _keep_sum(tr, k):
    """+1 on a and -1 on b of the round polynomial at k: q(0) + q(1) holds, q(r) does not"""
    t = tr.copy()
    t[k]["re"] = (int(t[k]["re"]) + 1) % P
    t[k + 1]["re"] = (int(t[k + 1]["re"]) + P - 1) % P
    return t


# ------------------------------------------------------------------ CPU
def test_batch_verify_binding_rejects_bad_shapes_before_the_library(B, sha_circuit, monkeypatch):
    n_in = sha_circuit.layer_size(0) * sha_circuit.instances
    n_out = sha_circuit.layer_size(sha_circuit.n_layers - 1) * sha_circuit.instances
    n_tr = sha_circuit.transcript_len

    class _Circuit:   # the shape of sha_circuit, without the library
        instances = 1
        n_layers = 2
        transcript_len = n_tr
        challenge_count = sha_circuit.challenge_count

        def layer_size(self, i):
            return n_in if i == 0 else n_out

    p = B.Prover.__new__(B.Prover)   # no device context: the checks must fire before any library call
    p.circuit, p.h = _Circuit(), None
    called = []

    def no_lib():
        called.append(1)
        raise AssertionError("library called")

    # A context or circuit of an earlier test that the cycle collector frees during the checks would reach the patched
    # lib() from its __del__: collect them before patching, and keep the collector off while the checks run.
    gc.collect()
    monkeypatch.setattr(B, "lib", no_lib)
    x, ctx = np.zeros((2, n_in), np.uint64), [bytes(32)] * 2
    out, tr = np.zeros((2, n_out), F_DTYPE), np.zeros((2, n_tr), F_DTYPE)
    bad = [
        (np.zeros(n_in, np.uint64), ctx[:1], out[:1], tr[:1]),           # 1-D inputs
        (np.zeros((0, n_in), np.uint64), [], out[:0], tr[:0]),           # B = 0
        (x.astype(np.float64), ctx, out, tr),                            # inputs not integers
        (x[:, :-1], ctx, out, tr),                                       # short input rows
        (x, ctx[:1], out, tr),                                           # one context for two statements
        (x, [bytes(32), bytes(31)], out, tr),                            # a short context
        (x, np.zeros((2, 32), np.int32), out, tr),                       # context array of the wrong type
        (x, ctx, out[:, :-1], tr),                                       # short output rows
        (x, ctx, out[:1], tr),                                           # outputs of one statement
        (x, ctx, out.reshape(-1), tr),                                   # 1-D outputs
        (x, ctx, np.zeros((2, n_out), np.uint64), tr),                   # outputs not field elements
        (x, ctx, out, tr[:, :-1]),                                       # short transcripts
        (x, ctx, out, np.zeros((3, n_tr), F_DTYPE)),                     # transcripts of three statements
        (x, ctx, out, np.zeros((2, 2 * n_tr), np.uint64)),               # transcripts not field elements
        (x, ctx, out, list(tr)),                                         # not an array
    ]
    gc.disable()
    try:
        for k, args in enumerate(bad):
            with pytest.raises(ValueError):
                p.verify_fs_bound_batch(*args)
            assert not called, f"case {k}"
    finally:
        gc.enable()


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_batch_outputs_are_each_statements_output_layer(B, sha_circuit):
    for name, circ in _batch_cases(B, sha_circuit):
        p = B.Prover(circ)
        for n in (1, 3, 64):
            x, ctx = _inputs(circ, n, 23 + n), _contexts(n, 23 + n)
            res = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
            assert len(res) == 4 and len(p.prove_fs_bound_batch(x, ctx)) == 3
            out = res[3]
            n_out = circ.layer_size(circ.n_layers - 1) * circ.instances
            assert out.shape == (n, n_out) and out.dtype == F_DTYPE
            assert (out == _evaluated_outputs(B, circ, x)).all(), f"{name} B={n}"
        p.close()


def _check_honest(B, circ, n, seed, name, sample=None):
    p = B.Prover(circ)
    x, ctx = _inputs(circ, n, seed), _contexts(n, seed)
    tr, ch, st, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    acc, code, layer, vch = p.verify_fs_bound_batch(x, ctx, out, tr, return_challenges=True)
    assert acc.dtype == bool and code.shape == layer.shape == (n,)
    assert acc.all() and not code.any() and not layer.any(), f"{name} B={n}: {np.flatnonzero(~acc)} rejected"
    assert (vch == ch).all(), f"{name} B={n}: replayed challenges != the prover's"
    for b in (range(n) if sample is None else sample):
        assert (vch[b] == circ.fs_challenges(st[b].tobytes(), tr[b])).all(), f"{name} B={n}: statement {b}"
    assert p.verify_fs_bound_batch(x, ctx, out, tr)[0].all()   # without challenges
    p.close()
    return x, ctx, out


@pytest.mark.gpu
def test_batch_verify_accepts_honest_batches(B, sha_circuit):
    for name, circ in _batch_cases(B, sha_circuit):
        for n in (1, 2, 3, 7, 64):
            _check_honest(B, circ, n, 31 + n, name)


@pytest.mark.gpu
def test_batch_of_600_outputs_and_verify(B, sha_circuit):
    sample = [0, 1, 295, 296, 297, 591, 592, 599]
    x, _, out = _check_honest(B, sha_circuit, 600, 7, "sha256_64", sample)
    assert (out[sample] == _evaluated_outputs(B, sha_circuit, x[sample])).all()


def _tamper_cases(B, sha_circuit):
    yield "sha256_64", sha_circuit
    for name in ("small_allops", "small_chain", "small_notquirk", "small_random_a", "small_random_b", "small_random_c"):
        yield name, _golden_pws(B, name)
    yield "all_types_x3", all_types_circuit(B, 41).replicate(3)
    rng = random.Random(905 * 104729)
    n_in, n_g = rng.choice([3, 8, 17, 64, 200, 257, 1000]), rng.choice([1, 2, 7, 30, 120, 500, 2000])
    yield "random_pws_905", B.Circuit.from_pws_text(_make_golden().random_pws(905, n_in, n_g))


@pytest.mark.gpu
def test_batch_verdicts_equal_single_verdicts_on_tampered_proofs(B, sha_circuit):
    codes = set()
    for name, circ in _tamper_cases(B, sha_circuit):
        pos = _message_positions(circ)
        final, liu_final = _last_rounds(circ)
        tampers = [(what, lambda s, k=k: s.update(tr=_bump(s["tr"], k))) for what, k in pos.items()]
        if final is not None:
            tampers.append(("final value", lambda s: s.update(tr=_keep_sum(s["tr"], final))))
        if liu_final is not None:
            tampers.append(("Liu final", lambda s: s.update(tr=_keep_sum(s["tr"], liu_final))))
        n_out = circ.layer_size(circ.n_layers - 1) * circ.instances

        def other_context(s):
            c = bytearray(s["ctx"]); c[0] ^= 0x80
            s.update(ctx=bytes(c))

        def other_inputs(s):
            x = s["x"].copy(); x[1] = (int(x[1]) + 1) % P
            s.update(x=x)

        def non_canonical(s):
            t = s["tr"].copy(); t[3]["re"] = P
            s.update(tr=t)

        tampers += [("output", lambda s: s.update(out=_bump(s["out"], n_out // 3, "im"))), ("context", other_context),
                    ("inputs", other_inputs), ("non-canonical", non_canonical)]
        n = 2 * len(tampers) + 1   # honest statements at even indices, a tampered one between every two
        p = B.Prover(circ)
        x, ctx = _inputs(circ, n, 61), _contexts(n, 61)
        tr, _, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
        x, tr, out, ctx = x.copy(), tr.copy(), out.copy(), list(ctx)
        for j, (what, f) in enumerate(tampers):
            b = 2 * j + 1
            s = dict(x=x[b], ctx=ctx[b], out=out[b], tr=tr[b])
            f(s)
            x[b], ctx[b], out[b], tr[b] = s["x"], s["ctx"], s["out"], s["tr"]
        acc, code, layer = p.verify_fs_bound_batch(x, ctx, out, tr)
        p.close()
        for b, want in enumerate(_singles(B, circ, x, ctx, out, tr)):
            what = "honest" if b % 2 == 0 else tampers[b // 2][0]
            assert (bool(acc[b]), int(code[b]), int(layer[b])) == want, f"{name}: statement {b} ({what})"
            assert want[0] == (b % 2 == 0), f"{name}: statement {b} ({what})"
            codes.add(want[1])
    assert codes >= set(range(1, 9)), f"fail codes hit: {sorted(codes)}"


@pytest.mark.gpu
def test_batch_verify_leaves_the_context_untouched(B, sha_circuit):
    circ = sha_circuit.replicate(3)
    inputs, chal = circ.inputs(), circ.draw_challenges()
    p = B.Prover(circ)
    fs0 = p.prove_fs_bound(CONTEXT)
    vals0 = p.values(circ.n_layers - 1)
    x, ctx = _inputs(circ, 4, 13), _contexts(4, 13)
    tr, _, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    assert p.verify_fs_bound_batch(x, ctx, out, tr)[0].all()
    assert (p.values(circ.n_layers - 1) == vals0).all()
    assert (p.transcript() == fs0[0]).all()
    assert p.verify(fs0[0]) == (True, 0, 0)   # the resident challenges are still those of the last single proof
    assert _same(p.prove_fs_bound(CONTEXT), fs0)
    tr0 = p.prove(inputs=inputs, challenges=chal)
    ver0 = p.verify(tr0)
    assert p.verify_fs_bound_batch(x, ctx, out, tr)[0].all()
    assert (p.transcript() == tr0).all()
    assert p.verify(tr0) == ver0 == (True, 0, 0)
    assert (p.prove(inputs=inputs, challenges=chal) == tr0).all()
    assert _same(p.prove_fs_bound(CONTEXT), fs0)
    p.close()


@pytest.mark.gpu
def test_batch_verify_launches_do_not_grow_with_B(B, sha_circuit):
    p = B.Prover(sha_circuit)
    args = {}
    for n in (1, 8):
        x, ctx = _inputs(sha_circuit, n, 1), _contexts(n, 1)
        tr, _, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
        args[n] = (x, ctx, out, tr)
    counts = {}
    for n in (1, 8, 1, 8):
        assert p.verify_fs_bound_batch(*args[n])[0].all()
        counts[n] = p.last_prove_launches
    assert counts[8] == counts[1] > 0
    p.close()


@pytest.mark.gpu
def test_batch_verify_errors_leave_the_context_usable(B):
    circ = _assert_circuit(B).replicate(2)
    n = 8
    rng = np.random.default_rng(4)
    xs = rng.integers(0, P, size=(n, circ.num_inputs), dtype=np.uint64)
    xs[:, 1::4] = xs[:, 0::4]   # every instance's assert holds
    ctx = _contexts(n, 2)
    p = B.Prover(circ)
    p.set_inputs(xs[0])
    ref = p.prove_fs_bound(CONTEXT)
    n_out = circ.layer_size(circ.n_layers - 1) * circ.instances
    outs = np.zeros(n * n_out, F_DTYPE)

    def last_outputs(cap=outs.size):
        return B.lib().vp_last_batch_outputs(p.h, B._ptr(outs), cap)

    VP_ERR_ARG = last_outputs()   # before any batch
    assert VP_ERR_ARG != 0
    tr, ch, _, out = p.prove_fs_bound_batch(xs, ctx, return_outputs=True)
    assert last_outputs() == 0 and (outs.reshape(n, n_out) == out).all()
    assert last_outputs(outs.size - 1) == VP_ERR_ARG

    ctx_arr = np.frombuffer(b"".join(ctx), np.uint8)
    acc, code, layer = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
    vch = np.zeros(ch.shape, F_DTYPE)

    def raw(B_, x=xs, n_in=xs.size, o=out, n_o=out.size, t=tr, n_t=tr.size, a=acc, ch_cap=vch.size):
        return B.lib().vp_verify_fs_bound_batch(p.h, B_, B._ptr(x), n_in, B._ptr(ctx_arr), B._ptr(o), n_o, B._ptr(t), n_t,
                                                B._ptr(a), B._ptr(code), B._ptr(layer), B._ptr(vch), ch_cap)

    assert raw(n) == 0 and acc.all() and (vch == ch).all()
    assert last_outputs() == VP_ERR_ARG   # a verifying batch ends the outputs' validity
    assert raw(0, n_in=0, n_o=0, n_t=0) == VP_ERR_ARG
    assert raw(n, n_in=xs.size - 1) == VP_ERR_ARG
    assert raw(n, n_o=out.size - 1) == VP_ERR_ARG
    assert raw(n, n_t=tr.size - 1) == VP_ERR_ARG
    assert raw(n, ch_cap=vch.size - 1) == VP_ERR_ARG
    assert raw(n, a=None) == VP_ERR_ARG
    bad = xs.copy()
    bad[6, 2] = P
    with pytest.raises(B.VpError) as e:
        p.verify_fs_bound_batch(bad, ctx, out, tr)
    assert e.value.code == VP_ERR_ARG and "statement 6" in str(e.value)
    o = out.copy()
    o[5, 1]["im"] = P
    with pytest.raises(B.VpError) as e:
        p.verify_fs_bound_batch(xs, ctx, o, tr)
    assert e.value.code == VP_ERR_ARG and "statement 5" in str(e.value)

    p.prove_fs_bound_batch(xs, ctx)
    assert last_outputs() == 0
    broken = xs.copy()
    broken[5, 5] = (int(broken[5, 4]) + 1) % P   # an assert fails in statement 5
    with pytest.raises(B.VpError):
        p.prove_fs_bound_batch(broken, ctx)
    assert last_outputs() == VP_ERR_ARG   # after a failed batch

    assert _same(p.prove_fs_bound(CONTEXT), ref)
    assert p.verify_fs_bound(CONTEXT, p.values(circ.n_layers - 1), ref[0]) == (True, 0, 0)
    acc2, code2, _ = p.verify_fs_bound_batch(xs, ctx, out, tr)
    assert acc2.all() and not code2.any()
    p.close()
