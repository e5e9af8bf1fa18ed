"""The prover's size-dependent code paths, driven at sizes the oracle proves in seconds and compared with it bit for bit.

The engine chooses code from sizes and counts the circuit determines: how k_phase_dfs spreads a pass over its workers, how
long CSR rows are cut into items and summed back (k_combine_phase1/2), the item order inside a sort window, the phase-2
eq-product table (k_p2_hs), and the layer-count limits. Two knobs read at vp_create move those choices down to small
circuits: VP_DFS_GRID caps the pass-kernel grid (at least 2 blocks), VP_ITEM_SORT_WINDOW sets the sort window (1 turns
sorting off). VP_NO_HS turns the eq-product table off, which counts its launches. The knobs are set only around
B.Prover(...) (monkeypatch.context), so no other test's context sees them."""
import numpy as np
import pytest

from test_gpu_parity import _ADD, _INPUT, _MUL, _SUB, _all_types_circuit, _assert_same

# ------------------------------------------------------------------ the pass-work rule, restated
# engine.cu build_pass_plan (work per pass), launch_dfs_kernel (grid), kernels.cuh k_phase_dfs (share / active / alive)
DFS_SOLO, DFS_WCHUNK, WPB = 128, 128, 4          # VP_DFS_SOLO, items per warp chunk, warps per block (128 threads)
DFS_CHUNK = WPB * DFS_WCHUNK                     # items one block covers in one sweep


def _cdiv(a, b):
    return -(-a // b)


def ceil_log2(x):
    return (x - 1).bit_length() if x > 0 else -1


def pass_works(tabs, rounds):
    """work items of every pass of a phase: tabs = [(bits, live)] sorted by bits descending, two rounds per pass"""
    live = [t[1] for t in tabs]
    gone = [False] * len(tabs)
    works, j = [], 1
    while j <= rounds:
        nr = 2 if j + 1 <= rounds else 1
        work = 0
        for t, (bits, _) in enumerate(tabs):
            if gone[t]:
                continue
            rem = bits - (j - 1)
            if rem <= 0:
                gone[t] = True
                continue
            two = nr == 2 and rem >= 2
            work += (_cdiv(live[t], 4 if two else 2) + 31) & ~31
            live[t] = _cdiv(_cdiv(live[t], 2), 2) if two else _cdiv(live[t], 2)
            if not two and rem == 1 and nr == 2:
                gone[t] = True
        works.append(work)
        j += nr
    return works


def dfs_grid(max_work, grid_knob):
    """blocks of the launch under VP_DFS_GRID=grid_knob (the occupancy cap is far above every knob value used here)"""
    return 1 if max_work <= DFS_CHUNK else min(_cdiv(max_work, DFS_CHUNK) + 1, max(grid_knob, 2))


def pass_kind(work, n_workers):
    """('solo' | 'static' | 'chunked', active workers)"""
    if work <= DFS_SOLO or n_workers == 0:
        return "solo", 0
    share = min(DFS_WCHUNK, (_cdiv(work, n_workers * WPB) + 31) & ~31)
    active = min(n_workers, _cdiv(work, share * WPB))
    return ("static" if active * share * WPB >= work else "chunked"), active


def phase_plan(works, grid_knob):
    """[(kind, active, alive)] of every pass; alive = the largest `active` of this and all later passes"""
    n_workers = dfs_grid(max(works), grid_knob) - 1
    kinds = [pass_kind(w, n_workers) for w in works]
    alive, mx = [], 0
    for _, a in reversed(kinds):
        mx = max(mx, a)
        alive.append(mx)
    return [(k, a, al) for (k, a), al in zip(kinds, reversed(alive))]


def circuit_phases(circ):
    """(layer, phase, tables, rounds) of every sumcheck phase of a whole proof (engine.cu vp_create: phase 1 and Liu have
    one table over layer i-1, phase 2 one per non-empty dad subset, bits descending)"""
    K = circ.instances
    out = []
    for i in range(1, circ.n_layers):
        pb = circ.bit_length(i - 1)
        one = [(pb, circ.layer_size(i - 1) * K)]
        out.append((i, 1, one, pb))
        m = circ.max_dad_bit_length(i)
        if m != -1:
            tabs = [(ceil_log2(d * K), d * K) for d in (circ.dad_size(i, l) for l in range(i)) if d > 0]
            out.append((i, 2, sorted(tabs, key=lambda t: -t[0]), m))
        out.append((i, 3, one, pb))
    return [p for p in out if p[3] > 0]


def sweep_kinds(circ, grids):
    """{grid: set of pass kinds}, and whether some phase has a later pass with more active workers than an earlier one"""
    kinds, rising = {}, False
    for g in grids:
        ks = set()
        for _, _, tabs, rounds in circuit_phases(circ):
            plan = phase_plan(pass_works(tabs, rounds), g)
            ks |= {k for k, _, _ in plan}
            act = [a for k, a, _ in plan if k != "solo"]
            rising |= any(act[b] > act[a] for a in range(len(act)) for b in range(a + 1, len(act)))
        kinds[g] = ks
    return kinds, rising


def test_pass_rule_restatement():
    """the examples of k_phase_dfs's comment, the three modes, and the grid of launch_dfs_kernel"""
    assert pass_kind(2100, 8) == ("static", 6)
    assert pass_kind(2048, 8) == ("static", 8)
    assert pass_kind(128, 8) == ("solo", 0) and pass_kind(129, 8) == ("static", 2)
    assert pass_kind(5000, 0) == ("solo", 0)
    assert pass_kind(DFS_CHUNK * 8, 8) == ("static", 8) and pass_kind(DFS_CHUNK * 8 + 1, 8)[0] == "chunked"
    assert pass_kind(184 * DFS_CHUNK, 184)[0] == "static" and pass_kind(184 * DFS_CHUNK + 1, 184)[0] == "chunked"   # default grid: 185
    assert dfs_grid(512, 33) == 1 and dfs_grid(513, 33) == 3 and dfs_grid(513, 2) == 2 and dfs_grid(10 ** 6, 0) == 2
    # one table of 2^13 entries: 2048, 512, 128 and 32 items; the last one-round pass of 2^3 entries: 4 items in a warp
    assert pass_works([(13, 8192)], 13) == [2048, 512, 128, 32, 32, 32, 32]
    assert pass_works([(3, 8)], 3) == [32, 32]
    # a table that reaches one value in a pass's first round joins add_term in its second round and is gone after it
    assert pass_works([(5, 32), (1, 2)], 5) == [32 + 32, 32, 32]
    # 4000, 2100, then 2048 items on 8 workers: a later pass needs more workers than the one before it
    assert dfs_grid(4000, 9) == 9
    plan = phase_plan([4000, 2100, 2048], 9)
    assert [(a, al) for _, a, al in plan] == [(8, 8), (6, 8), (8, 8)]


# ------------------------------------------------------------------ shared checks
GRIDS = [2, 3, 4, 5, 7, 9, 16, 33, None]


def _oracle(O, circ):
    flat = circ.expand() if circ.instances > 1 else circ
    return O.OracleCircuit(flat.flat())


def _prover(B, monkeypatch, circ, **knobs):
    """B.Prover(circ) with the knobs set only while vp_create reads them"""
    with monkeypatch.context() as m:
        for k, v in knobs.items():
            if v is not None:
                m.setenv(k, str(v))
        return B.Prover(circ)


def _check_whole_proof(B, monkeypatch, circ, want, what, **knobs):
    """the whole proof on one and six lanes equals the oracle's; the device verifier accepts it"""
    p = _prover(B, monkeypatch, circ, **knobs)
    inp, ch = circ.inputs(), circ.draw_challenges()
    for lanes in (1, 6):
        p.set_lanes(lanes)
        _assert_same(p.prove(inputs=inp, challenges=ch), want, f"{what}, {lanes} lane(s)")
        launches = p.last_prove_launches
    assert p.verify(want) == (True, 0, 0), what
    p.close()
    return launches


def _check_interactive(B, monkeypatch, circ, want, what, **knobs):
    p = _prover(B, monkeypatch, circ, **knobs)
    _assert_same(B.prove_interactive(p, circ), want, f"{what}, method by method")
    p.close()


# ------------------------------------------------------------------ 1. worker-grid sweep
def _sweep_circuits(B, sha_circuit):
    zero = B.Circuit.random(6, 12, 31)
    zero.set_inputs(np.zeros(zero.num_inputs, np.uint64))
    cplx = _all_types_circuit(B, 41, n_layers=6, max_size=160, complex_consts=True, with_assert=True)
    assert any(int(c["im"]) for i in range(1, cplx.n_layers) for c in cplx.export_layer(i)["c"]), "no complex constant"
    top = _all_types_circuit(B, 43, n_layers=6, max_size=160, with_assert=True).replicate(24)
    top.set_inputs(np.full(top.num_inputs, B.P - 1, np.uint64))
    return [("random 6 x 2^13", B.Circuit.random(6, 13, 5)), ("SHA256_64 x 3", sha_circuit.replicate(3)),
            ("all types, complex constants, asserts x 64", cplx.replicate(64)), ("random 6 x 2^12, inputs 0", zero),
            ("all types, asserts x 24, inputs p-1", top), ("120 layers x 9", _deep_circuit(B, 120).replicate(9))]


@pytest.mark.gpu
def test_dfs_worker_grid_sweep(B, O, sha_circuit, monkeypatch):
    """every circuit at every grid against the oracle; the restatement shows that the sweep reaches all three pass modes
    and a phase in which a later pass has more active workers than an earlier one"""
    seen, rising = set(), False
    for name, circ in _sweep_circuits(B, sha_circuit):
        kinds, r = sweep_kinds(circ, [g for g in GRIDS if g])
        seen |= set().union(*kinds.values())
        rising |= r
        want, _, _ = _oracle(O, circ).prove()
        for g in GRIDS:
            _check_whole_proof(B, monkeypatch, circ, want, f"{name}, VP_DFS_GRID={g}", VP_DFS_GRID=g)
    assert seen == {"solo", "static", "chunked"} and rising


# ------------------------------------------------------------------ 2. long rows x sort window
ROW_LENGTHS = [1, 7, 8, 9, 16, 17, 63, 64, 65, 255, 256, 257, 2049]


def _hub_circuit(B, n_layers=5, size=4096, seed=7):
    """every non-input layer: phase-1 rows (gates by u) of ROW_LENGTHS plus rows of one; phase-2 rows (binary gates by
    (l, lv)) of ROW_LENGTHS spread over the earlier layers plus rows of one; Liu rows (later layers whose subset holds an
    entry) of 1 .. n_layers - 1 - i"""
    rng = np.random.default_rng(seed)
    hub = sum(ROW_LENGTHS)
    ty, l, u, v = [_INPUT] * size, [-1] * size, [int(x) for x in rng.integers(0, 1 << 31, size)], [0] * size
    for i in range(1, n_layers):
        # phase 1: hub row r reads u = 300 r + 1 (spread over the previous layer), the other gates distinct u's
        uu = [300 * r + 1 for r, n in enumerate(ROW_LENGTHS) for _ in range(n)]
        rest = [x for x in range(size) if x % 300 != 1][:size - hub]
        uu += rest
        # phase 2 (in another gate order): hub row r reads v = 5 r + 2 of layer r % i, the others distinct v's of layer i-1
        vv = [(r % i, 5 * r + 2) for r, n in enumerate(ROW_LENGTHS) for _ in range(n)]
        vv += [(i - 1, x) for x in range(size) if x % 5 != 2][:size - hub]
        perm = rng.permutation(size)
        for g in range(size):
            ll, vx = vv[perm[g]]
            ty.append((_ADD, _MUL, _SUB)[g % 3])
            l.append(ll)
            u.append(uu[g])
            v.append(vx)
    return B.Circuit.from_arrays([size] * n_layers, ty, l, u, v)


def test_hub_circuit_row_lengths(B):
    circ = _hub_circuit(B)
    for i in range(1, circ.n_layers):
        L = circ.export_layer(i)
        p1 = np.bincount(L["u"].astype(np.int64))
        assert set(ROW_LENGTHS) <= set(p1[p1 > 0].tolist()), i
        p2 = {}
        for ll, lv in zip(L["l"].tolist(), L["lv"].tolist()):
            p2[(ll, lv)] = p2.get((ll, lv), 0) + 1
        assert set(ROW_LENGTHS) <= set(p2.values()), i
        assert len({ll for (ll, _), n in p2.items() if n > 8}) == min(i, len(ROW_LENGTHS)), i   # long rows from every source
    liu = np.zeros(circ.layer_size(0), np.int64)
    for j in range(1, circ.n_layers):
        liu[circ.export_dad(j, 0)] += 1
    assert set(liu.tolist()) >= set(range(1, circ.n_layers)), "Liu rows of 1 .. n-1 entries"


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3, 8, 33])
def test_long_rows_and_sort_window(B, O, monkeypatch, K):
    circ = _hub_circuit(B)
    if K > 1:
        circ = circ.replicate(K)
    want, _, _ = _oracle(O, circ).prove()
    for w in (1, 2, 3, 32, 33, None):
        what = f"hub x {K}, VP_ITEM_SORT_WINDOW={w}"
        _check_whole_proof(B, monkeypatch, circ, want, what, VP_ITEM_SORT_WINDOW=w)
        _check_interactive(B, monkeypatch, circ, want, what, VP_ITEM_SORT_WINDOW=w)


# ------------------------------------------------------------------ 3. layer-count limits
SUBSET_SIZES = [1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33]


def _deep_circuit(B, n_layers, one_per_layer=False, seed=3):
    """every layer reads from every earlier layer: dad subset (i, l) has SUBSET_SIZES[(i + l) % 11] entries (top layer) or
    at most 5 (the others); with one_per_layer the top layer reads exactly one entry of each earlier layer"""
    rng = np.random.default_rng(seed)
    sizes = [64]
    ty, l, u, v = [_INPUT] * 64, [-1] * 64, [int(x) for x in rng.integers(0, 1 << 31, 64)], [0] * 64
    for i in range(1, n_layers):
        top = i == n_layers - 1
        if top and one_per_layer:
            subs = [1] * i
        else:
            subs = [SUBSET_SIZES[(i + s) % (11 if top else 5)] for s in range(i)]
        reads = [(s, x) for s in range(i) for x in range(subs[s])]
        S = max(64, len(reads))
        reads += [(i - 1, x % sizes[i - 1]) for x in range(S - len(reads))]
        sizes.append(S)
        for g, (s, x) in enumerate(reads):
            ty.append(_MUL if g % 2 else _ADD)
            l.append(s)
            u.append(int(rng.integers(0, sizes[i - 1])))
            v.append(x)
    return B.Circuit.from_arrays(sizes, ty, l, u, v)


def _claims_v_index(circ):
    """transcript index of claims_v[0] of the top layer (layout of helpers.transcript_text)"""
    top = circ.n_layers - 1
    return 1 + 3 * circ.bit_length(top - 1) + 1 + 3 * circ.max_dad_bit_length(top)


DEEP = [(64, False, 1), (64, False, 9), (65, False, 1), (65, False, 9), (120, False, 1), (120, False, 9), (120, True, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_layers,one_per_layer,K", DEEP)
def test_layer_count_limits(B, O, monkeypatch, n_layers, one_per_layer, K):
    circ = _deep_circuit(B, n_layers, one_per_layer)
    if K > 1:
        circ = circ.replicate(K)
    top = n_layers - 1
    assert all(circ.dad_size(top, s) > 0 for s in range(top))
    if one_per_layer:
        assert circ.max_dad_bit_length(top) == 0                      # phase 2 of the top layer has no round
    else:
        assert len({ceil_log2(circ.dad_size(top, s) * K) for s in range(top)}) >= 5
    oc = _oracle(O, circ)
    want, _, _ = oc.prove()
    what = f"{n_layers} layers x {K}"
    _check_whole_proof(B, monkeypatch, circ, want, what)
    _check_interactive(B, monkeypatch, circ, want, what)
    p = B.Prover(circ)
    p.prove(inputs=circ.inputs(), challenges=circ.draw_challenges())
    c0 = _claims_v_index(circ)
    for k in (0, 60, 118):
        if k >= top:
            continue
        bad = want.copy()
        bad[c0 + k]["re"] = (int(bad[c0 + k]["re"]) + 1) % B.P
        w = oc.verify(bad)
        assert not w[0] and p.verify(bad) == (bool(w[0]), w[1], w[2]), f"{what}: claims_v[{k}] tampered"
    # statement-bound proofs: one against the oracle, a batch of three against the single proofs
    ctx = [bytes([k + 1] * 32) for k in range(3)]
    rng = np.random.default_rng(n_layers + K)
    inputs = np.stack([circ.inputs()] + [rng.integers(0, B.P, circ.num_inputs, dtype=np.uint64) for _ in range(2)])
    singles = []
    for b in range(3):
        p.set_inputs(inputs[b])
        tr, ch, st = p.prove_fs_bound(ctx[b])
        singles.append(tr)
        if b == 0:
            want_tr, want_ch = oc.prove_fs(st)
            _assert_same(tr, want_tr, f"{what}: statement-bound transcript")
            _assert_same(ch, want_ch, f"{what}: statement-bound challenges")
    tr_b, _, _, out_b = p.prove_fs_bound_batch(inputs, ctx, return_outputs=True)
    for b in range(3):
        _assert_same(tr_b[b], singles[b], f"{what}: batch statement {b}")
    acc, code, layer = p.verify_fs_bound_batch(inputs, ctx, out_b, tr_b)
    assert acc.all(), (code, layer)
    p.close()


@pytest.mark.gpu
def test_121_layers_rejected(B):
    circ = _deep_circuit(B, 121)
    with pytest.raises(B.VpError):
        B.Prover(circ)


# ------------------------------------------------------------------ 4. phase-2 eq-product table (k_p2_hs)
def hs_layers(circ):
    """layers whose phase-2 init tabulates the eq products (engine.cu do_init_phase2): K >= 8 and ng * nu <= 64, with
    ng = (S_i >> fh_i) + 2, nu = (S_(i-1) >> fh_(i-1)) + 2 and fh = bit_length // 2 of the replicated layer"""
    K = circ.instances
    out = {}
    for i in range(1, circ.n_layers):
        if circ.max_dad_bit_length(i) == -1:
            continue
        ng = (circ.layer_size(i) >> (circ.bit_length(i) >> 1)) + 2
        nu = (circ.layer_size(i - 1) >> (circ.bit_length(i - 1) >> 1)) + 2
        out[i] = ng * nu
    return {i: x for i, x in out.items() if K >= 8}


def _hs_circuit(B, sizes, seed=9):
    rng = np.random.default_rng(seed)
    ty, l, u, v = [_INPUT] * sizes[0], [-1] * sizes[0], [int(x) for x in rng.integers(0, 1 << 31, sizes[0])], [0] * sizes[0]
    for i in range(1, len(sizes)):
        for g in range(sizes[i]):
            s = int(rng.integers(0, i))
            ty.append((_ADD, _MUL, _SUB)[g % 3])
            l.append(s)
            u.append(int(rng.integers(0, sizes[i - 1])))
            v.append(int(rng.integers(0, sizes[s])))
    return B.Circuit.from_arrays(sizes, ty, l, u, v)


HS_CASES = [((384, 384, 384, 504, 384, 64), 8), ((384, 384, 384, 504, 384, 64), 16), ((504, 504, 384, 384, 96, 200), 9)]


def test_hs_cases_straddle_the_bound(B):
    for sizes, K in HS_CASES:
        prods = hs_layers(_hs_circuit(B, sizes).replicate(K))
        assert any(x <= 64 for x in prods.values()) and any(x > 64 for x in prods.values()), (sizes, K, prods)
    assert any(x == 64 for sizes, K in HS_CASES for x in hs_layers(_hs_circuit(B, sizes).replicate(K)).values())


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,K", HS_CASES)
def test_phase2_eq_product_table_bound(B, O, monkeypatch, sizes, K):
    circ = _hs_circuit(B, sizes).replicate(K)
    want, _, _ = _oracle(O, circ).prove()
    n_hs = sum(x <= 64 for x in hs_layers(circ).values())
    with_hs = _check_whole_proof(B, monkeypatch, circ, want, f"{sizes} x {K}")
    without = _check_whole_proof(B, monkeypatch, circ, want, f"{sizes} x {K}, VP_NO_HS", VP_NO_HS=1)
    assert with_hs - without == n_hs
