"""vp_prove_fs_bound_batch_dev and vp_verify_fs_bound_batch_dev: the batch calls on arrays in device memory (torch CUDA
tensors), queued on the caller's stream with a status or verdict per statement.

A proved statement must be, bit for bit, what the host-memory batch gives; every verdict apart from code 9 must be the
host-memory batch verifier's, so that k_verify_check is pinned against Engine::verify_check on every failure path; a
failing statement changes nothing else; the calls must not wait for the stream."""
import time

import numpy as np
import pytest

from test_fs_batch import _assert_circuit, _contexts, _inputs, _singles
from test_fs_batch_verify import _keep_sum, _last_rounds, _tamper_cases
from test_fs_statement import CONTEXT, F_DTYPE, P, _bump, _golden_pws, _message_positions, all_types_circuit


# ------------------------------------------------------------------ conversions
def _fe_tensor(a):
    """F_DTYPE [B, n] -> int64 CUDA tensor [B, n, 2] (re, im)"""
    import torch
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.view(np.int64).reshape(a.shape + (2,)).copy()).cuda()


def _fe_array(t):
    """int64 tensor [B, n, 2] -> F_DTYPE [B, n]"""
    a = np.ascontiguousarray(t.cpu().numpy())
    return a.view(F_DTYPE).reshape(a.shape[:-1])


def _dev_inputs(x, ctx):
    import torch
    x = torch.from_numpy(np.ascontiguousarray(x).view(np.int64).copy()).cuda()
    c = torch.from_numpy(np.frombuffer(b"".join(ctx), np.uint8).reshape(len(ctx), 32).copy()).cuda()
    return x, c


def _prove_dev(p, x, ctx):
    """device prove with every optional array -> (tr, ch, st, out, status) as host arrays"""
    import torch
    tr, ch, st, out, status = p.prove_fs_bound_batch_cuda(*_dev_inputs(x, ctx), challenges=True, outputs=True)
    torch.cuda.synchronize()
    return _fe_array(tr), _fe_array(ch), st.cpu().numpy(), _fe_array(out), status.cpu().numpy()


def _verify_dev(p, x, ctx, out, tr):
    import torch
    xi, c = _dev_inputs(x, ctx)
    acc, code, layer, ch = p.verify_fs_bound_batch_cuda(xi, c, _fe_tensor(out), _fe_tensor(tr), challenges=True)
    torch.cuda.synchronize()
    return acc.cpu().numpy(), code.cpu().numpy(), layer.cpu().numpy(), _fe_array(ch)


# ------------------------------------------------------------------ CPU
def test_cuda_batch_binding_rejects_bad_tensors_before_the_library(B, sha_circuit, monkeypatch):
    import gc

    import torch
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
    p.circuit, p.h, p.device = _Circuit(), None, 0
    called = []

    def no_lib():
        called.append(1)
        raise AssertionError("library called")

    gc.collect()   # (see test_batch_verify_binding_rejects_bad_shapes_before_the_library)
    monkeypatch.setattr(B, "lib", no_lib)
    x, c = torch.zeros((2, n_in), dtype=torch.int64), torch.zeros((2, 32), dtype=torch.uint8)
    out, tr = torch.zeros((2, n_out, 2), dtype=torch.int64), torch.zeros((2, n_tr, 2), dtype=torch.int64)
    prove_bad = [
        ((x.numpy(), c), "torch tensor"),                              # not a tensor
        ((x.to(torch.int32), c), "torch.int64"),                       # wrong dtype
        ((x, c.to(torch.int8)), "torch.uint8"),
        ((x[:, :-1], c), "shape"),                                     # short rows
        ((x.reshape(-1), c), "shape|statements"),                      # 1-D inputs
        ((torch.zeros((0, n_in), dtype=torch.int64), c[:0]), "statements"),   # B = 0
        ((x, c[:1]), "shape"),                                         # one context for two statements
        ((torch.zeros((n_in, 2), dtype=torch.int64).t(), c), "contiguous"),
        ((x, c), "cuda:0"),                                            # host memory
    ]
    verify_bad = [
        ((x, c, out[:, :-1], tr), "shape"),
        ((x, c, out, tr[:1]), "shape"),
        ((x, c, out.to(torch.float64), tr), "torch.int64"),
        ((x, c, out, tr.reshape(2, -1)), "shape"),
        ((x, c, out, torch.zeros((2, 2, n_tr), dtype=torch.int64).transpose(1, 2)), "contiguous"),
        ((x, c, out, tr), "cuda:0"),
    ]
    gc.disable()
    try:
        for k, (args, why) in enumerate(prove_bad):
            with pytest.raises(ValueError, match=why):
                p.prove_fs_bound_batch_cuda(*args)
            assert not called, f"prove case {k}"
        for k, (args, why) in enumerate(verify_bad):
            with pytest.raises(ValueError, match=why):
                p.verify_fs_bound_batch_cuda(*args)
            assert not called, f"verify case {k}"
    finally:
        gc.enable()


# ------------------------------------------------------------------ GPU
def _check_prove(B, p, circ, n, seed, name):
    x, ctx = _inputs(circ, n, seed), _contexts(n, seed)
    want = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    tr, ch, st, out, status = _prove_dev(p, x, ctx)
    assert not status.any(), f"{name} B={n}: statuses {status}"
    for what, a, b in zip(("transcripts", "challenges", "statements", "outputs"), (tr, ch, st, out), want):
        assert (a == b).all(), f"{name} B={n}: {what}"


@pytest.mark.gpu
def test_device_prove_is_bit_identical_to_the_host_batch(B, sha_circuit):
    cases = [("sha256_64", sha_circuit, (1, 3, 8)), ("sha256_64_x3", sha_circuit.replicate(3), (3,)),
             ("all_types", all_types_circuit(B, 41), (1, 5)), ("all_types_x5", all_types_circuit(B, 41).replicate(5), (3,))]
    cases += [(name, _golden_pws(B, name), (1, 4)) for name in ("small_allops", "small_chain", "small_notquirk", "small_random_a",
                                                               "small_random_b", "small_random_c")]
    for name, circ, sizes in cases:
        p = B.Prover(circ)
        for n in sizes:
            _check_prove(B, p, circ, n, 71 + n, name)
        p.close()


@pytest.mark.gpu
def test_device_prove_larger_than_the_phase_grid(B, sha_circuit):
    p = B.Prover(sha_circuit)
    _check_prove(B, p, sha_circuit, 600, 5, "sha256_64")
    p.close()


@pytest.mark.gpu
def test_device_prove_reports_every_failing_statement(B):
    import torch
    circ = _assert_circuit(B).replicate(2)
    n = 8
    rng = np.random.default_rng(4)
    xs = rng.integers(0, P, size=(n, circ.num_inputs), dtype=np.uint64)
    xs[:, 1::4] = xs[:, 0::4]   # every instance's assert holds ...
    ctx = _contexts(n, 2)
    broken = xs.copy()
    broken[5, 5] = (int(broken[5, 4]) + 1) % P   # ... except in instance 1 of statement 5
    broken[7, 1] = (int(broken[7, 0]) + 1) % P   # ... and statement 7
    p = B.Prover(circ)
    with pytest.raises(B.VpError) as e:   # the host-memory batch: one error, naming the first
        p.prove_fs_bound_batch(broken, ctx)
    assert "statement 5:" in str(e.value)
    bad = broken.copy()
    bad[2, 3] = P   # not < p
    xd, cd = _dev_inputs(bad, ctx)
    res = p.prove_fs_bound_batch_cuda(xd, cd, challenges=True, outputs=True)
    torch.cuda.synchronize()
    tr, ch, out = (_fe_array(res[k]) for k in (0, 1, 3))
    st, status = res[2].cpu().numpy(), res[4].cpu().numpy()
    assert int(xd[2, 3]) == P and (xd.cpu().numpy().view(np.uint64) == bad).all()   # the caller's inputs are not touched
    assert list(status) == [0, 0, 1, 0, 0, 3, 0, 3]   # 2 + layer 1 for the assert gate
    for b in (2, 5, 7):
        assert not (tr[b]["re"].any() or tr[b]["im"].any() or ch[b]["re"].any() or ch[b]["im"].any()), f"statement {b}"
        assert not (out[b]["re"].any() or out[b]["im"].any() or st[b].any()), f"statement {b}"
    good = [b for b in range(n) if b not in (2, 5, 7)]
    for b, (tr1, ch1, st1) in zip(good, _singles(B, circ, bad[good], [ctx[b] for b in good])):
        assert st[b].tobytes() == st1 and (tr[b] == tr1).all() and (ch[b] == ch1).all(), f"statement {b}"
    p.close()


def _check_verdicts(B, p, x, ctx, out, tr, name):
    acc, code, layer, ch = p.verify_fs_bound_batch(x, ctx, out, tr, return_challenges=True)
    dacc, dcode, dlayer, dch = _verify_dev(p, x, ctx, out, tr)
    assert (dacc == acc).all() and (dcode == code).all() and (dlayer == layer).all(), \
        f"{name}: device {list(zip(dacc, dcode, dlayer))} != host {list(zip(acc, code, layer))}"
    assert (dch == ch).all(), f"{name}: challenges"
    return set(int(c) for c in code)


@pytest.mark.gpu
def test_device_verdicts_equal_the_host_batch(B, sha_circuit):
    p = B.Prover(sha_circuit)
    x, ctx = _inputs(sha_circuit, 8, 3), _contexts(8, 3)
    tr, _, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    assert _check_verdicts(B, p, x, ctx, out, tr, "honest sha256_64") == {0}
    p.close()
    codes = set()
    for name, circ in _tamper_cases(B, sha_circuit):
        pos = _message_positions(circ)
        final, liu_final = _last_rounds(circ)
        tampers = [lambda s, k=k: s.update(tr=_bump(s["tr"], k)) for k in pos.values()]
        if final is not None:
            tampers.append(lambda s: s.update(tr=_keep_sum(s["tr"], final)))
        if liu_final is not None:
            tampers.append(lambda s: s.update(tr=_keep_sum(s["tr"], liu_final)))
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

        tampers += [lambda s: s.update(out=_bump(s["out"], n_out // 3, "im")), other_context, other_inputs, non_canonical]
        n = 2 * len(tampers) + 1
        p = B.Prover(circ)
        x, ctx = _inputs(circ, n, 61), _contexts(n, 61)
        tr, _, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
        x, tr, out, ctx = x.copy(), tr.copy(), out.copy(), list(ctx)
        for j, f in enumerate(tampers):
            b = 2 * j + 1
            s = dict(x=x[b], ctx=ctx[b], out=out[b], tr=tr[b])
            f(s)
            x[b], ctx[b], out[b], tr[b] = s["x"], s["ctx"], s["out"], s["tr"]
        codes |= _check_verdicts(B, p, x, ctx, out, tr, name)
        p.close()
    assert codes >= set(range(0, 9)), f"fail codes hit: {sorted(codes)}"


@pytest.mark.gpu
def test_device_verify_code_9_rejects_one_statement(B, sha_circuit):
    n = 6
    p = B.Prover(sha_circuit)
    x, ctx = _inputs(sha_circuit, n, 8), _contexts(n, 8)
    tr, ch, _, out = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    bx, bout = x.copy(), out.copy()
    bout[1, 7]["im"] = P       # a non-canonical claimed output
    bx[4, 2] = P + 5           # an input >= p
    with pytest.raises(B.VpError):   # the host-memory batch rejects the whole call
        p.verify_fs_bound_batch(bx, ctx, bout, tr)
    acc, code, layer, dch = _verify_dev(p, bx, ctx, bout, tr)
    assert list(acc) == [1, 0, 1, 1, 0, 1] and list(code) == [0, 9, 0, 0, 9, 0] and not layer.any()
    for b in range(n):
        if b in (1, 4):
            assert not (dch[b]["re"].any() or dch[b]["im"].any())
        else:
            assert (dch[b] == ch[b]).all()
    p.close()


@pytest.mark.gpu
def test_device_calls_queue_on_the_current_stream(B, sha_circuit):
    import torch
    n = 8
    p = B.Prover(sha_circuit)
    x, ctx = _inputs(sha_circuit, n, 21), _contexts(n, 21)
    want = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    xd, cd = _dev_inputs(x, ctx)
    src, out_d, tr_d = xd.clone(), _fe_tensor(want[3]), _fe_tensor(want[0])
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for _ in range(2):   # warm-up, on this stream
            p.prove_fs_bound_batch_cuda(xd, cd, challenges=True, outputs=True)
            p.verify_fs_bound_batch_cuda(xd, cd, out_d, tr_d)
        s.synchronize()

    def ordered_calls():
        """the right inputs exist only after a long kernel on s: calls that did not run behind it would prove zeros"""
        with torch.cuda.stream(s):
            xd.zero_()
            s.synchronize()
            t0 = time.perf_counter()
            torch.cuda._sleep(1 << 31)   # about a second
            xd.copy_(src)
            t1 = time.perf_counter()
            tr, ch, st, out, status = p.prove_fs_bound_batch_cuda(xd, cd, challenges=True, outputs=True)
            acc, code, layer, _ = p.verify_fs_bound_batch_cuda(xd, cd, out, tr)
            t2 = time.perf_counter()
            s.synchronize()
            t3 = time.perf_counter()
        assert t3 - t0 > 0.2, "the sleep was too short to tell"
        assert t2 - t1 < 0.5 * (t3 - t1), f"the calls waited for the stream: {t2 - t1:.3f} s of {t3 - t1:.3f} s"
        assert not status.cpu().any() and acc.cpu().all() and not code.cpu().any()
        for what, a, b in zip(("transcripts", "challenges", "statements", "outputs"),
                              (_fe_array(tr), _fe_array(ch), st.cpu().numpy(), _fe_array(out)), want):
            assert (a == b).all(), what
        assert p.last_prove_ms > 0

    ordered_calls()
    p.set_stream(None)   # the context back on a stream of its own: the next calls must move it to s again
    ordered_calls()
    p.close()


@pytest.mark.gpu
def test_device_calls_leave_the_context_untouched_and_do_not_grow_launches(B, sha_circuit):
    p = B.Prover(sha_circuit)
    fs0 = p.prove_fs_bound(CONTEXT)
    vals0 = p.values(sha_circuit.n_layers - 1)
    launches = {}
    for n in (1, 8, 1, 8):
        x, ctx = _inputs(sha_circuit, n, 1), _contexts(n, 1)
        tr, ch, st, out, status = _prove_dev(p, x, ctx)
        launches[("prove", n)] = p.last_prove_launches
        acc = _verify_dev(p, x, ctx, out, tr)[0]
        launches[("verify", n)] = p.last_prove_launches
        assert not status.any() and acc.all()
    assert launches[("prove", 1)] == launches[("prove", 8)] > 0
    assert launches[("verify", 1)] == launches[("verify", 8)] > 0
    assert (p.values(sha_circuit.n_layers - 1) == vals0).all()
    assert (p.transcript() == fs0[0]).all()
    assert p.verify(fs0[0]) == (True, 0, 0)   # the resident challenges are still those of the last single proof
    p.close()


@pytest.mark.gpu
def test_device_call_argument_errors_leave_the_context_usable(B, sha_circuit):
    import torch
    n = 3
    p = B.Prover(sha_circuit)
    x, ctx = _inputs(sha_circuit, n, 2), _contexts(n, 2)
    want = p.prove_fs_bound_batch(x, ctx, return_outputs=True)
    xd, cd = _dev_inputs(x, ctx)
    tr, ch, out = _fe_tensor(want[0]), _fe_tensor(want[1]), _fe_tensor(want[3])
    st = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    status = torch.empty(n, dtype=torch.int32, device="cuda")
    host_x = np.ascontiguousarray(x)
    L = B.lib()

    def prove(B_=n, x_=xd.data_ptr(), tr_=tr.data_ptr(), st_=st.data_ptr(), status_=status.data_ptr()):
        return L.vp_prove_fs_bound_batch_dev(p.h, B_, x_, cd.data_ptr(), tr_, None, None, st_, status_)

    acc = torch.empty(n, dtype=torch.int32, device="cuda")

    def verify(B_=n, out_=out.data_ptr(), acc_=acc.data_ptr()):
        return L.vp_verify_fs_bound_batch_dev(p.h, B_, xd.data_ptr(), cd.data_ptr(), out_, tr.data_ptr(), acc_, None, None, None)

    assert prove() == 0 and verify() == 0
    torch.cuda.synchronize()
    VP_ERR_ARG = prove(B_=0)
    assert VP_ERR_ARG != 0
    cases = [prove(B_=65536), prove(x_=B._ptr(host_x).value), prove(tr_=tr.data_ptr() + 8), prove(st_=st.data_ptr() + 4),
             prove(status_=status.data_ptr() + 4), verify(B_=0), verify(B_=65536), verify(out_=B._ptr(want[3]).value),
             verify(out_=out.data_ptr() + 8), verify(acc_=acc.data_ptr() + 4)]
    assert cases == [VP_ERR_ARG] * len(cases), cases
    tr2, _, st2, _, status2 = p.prove_fs_bound_batch_cuda(xd, cd)
    acc2 = p.verify_fs_bound_batch_cuda(xd, cd, out, tr2)[0]
    torch.cuda.synchronize()
    assert not status2.cpu().any() and acc2.cpu().all() and (_fe_array(tr2) == want[0]).all()
    p.close()
