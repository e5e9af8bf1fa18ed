"""The proof layout and the Fiat-Shamir order on the host, against the C oracle, on circuits whose layout has corner cases:
a layer without phase 2, two layers, a replicated circuit, 120 layers (the top one with a phase 2 of zero rounds) and
SHA256_64. Everything here is host code: the transcript and challenge counts, the host-side challenge replay, the GKRProof
container and the text dump."""
import numpy as np
import pytest

from helpers import transcript_text
from test_gpu_parity import _ADD, _COPY, _INPUT, _MUL, _NOT, _SUB
from test_kernel_paths import _deep_circuit


def _no_phase2_circuit(B):
    """layer 1 holds only unary gates (no dad subset: no phase 2); layer 2 reads layers 1 and 0"""
    rng = np.random.default_rng(11)
    sizes = [16, 8, 8]
    ty, l, u, v = [_INPUT] * 16, [-1] * 16, [int(x) for x in rng.integers(0, 1 << 31, 16)], [0] * 16
    for g in range(8):
        ty.append(_COPY if g % 2 else _NOT); l.append(-1); u.append(int(rng.integers(0, 16))); v.append(0)
    for g in range(8):
        ty.append((_ADD, _MUL, _SUB)[g % 3]); l.append(g % 2); u.append(int(rng.integers(0, 8))); v.append(int(rng.integers(0, 8)))
    return B.Circuit.from_arrays(sizes, ty, l, u, v)


def _two_layer_circuit(B):
    rng = np.random.default_rng(12)
    ty, l, u, v = [_INPUT] * 8, [-1] * 8, [int(x) for x in rng.integers(0, 1 << 31, 8)], [0] * 8
    for g in range(4):
        ty.append(_MUL if g % 2 else _ADD); l.append(0); u.append(int(rng.integers(0, 8))); v.append(int(rng.integers(0, 8)))
    return B.Circuit.from_arrays([8, 4], ty, l, u, v)


CIRCUITS = ["no_phase2", "two_layers", "replicated", "deep_120", "sha256_64"]


@pytest.fixture(scope="module")
def cases(B, sha_circuit):
    return {
        "no_phase2": _no_phase2_circuit(B),
        "two_layers": _two_layer_circuit(B),
        "replicated": B.Circuit.random(4, 5, 9).replicate(5),
        "deep_120": _deep_circuit(B, 120, one_per_layer=True),
        "sha256_64": sha_circuit,
    }


@pytest.mark.parametrize("name", CIRCUITS)
def test_layout_and_fiat_shamir_order_match_the_oracle(B, O, cases, name):
    circ = cases[name]
    n = circ.n_layers
    if name == "no_phase2":
        assert circ.max_dad_bit_length(1) == -1 and circ.max_dad_bit_length(2) != -1
    if name == "two_layers":
        assert n == 2
    if name == "deep_120":
        assert n == 120 and circ.max_dad_bit_length(n - 1) == 0
    oc = O.OracleCircuit((circ.expand() if circ.instances > 1 else circ).flat())
    assert circ.transcript_len == oc.transcript_len
    assert circ.challenge_count == len(circ.draw_challenges()) == oc.challenge_count
    seed = bytes(range(7, 39))
    tr, ch = oc.prove_fs(seed)
    got = circ.fs_challenges(seed, tr)
    assert (got["re"] == ch["re"]).all() and (got["im"] == ch["im"]).all()
    back = circ.from_gkrproof(circ.to_gkrproof(tr))
    assert (back["re"] == tr["re"]).all() and (back["im"] == tr["im"]).all()
    assert circ.transcript_text(tr, ch) == transcript_text(circ, tr, ch)
