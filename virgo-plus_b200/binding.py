"""ctypes binding of the C ABI in include/virgo_b200.h (libvirgo_b200.so).

Plumbing for tests/, bench.py and __graft_entry__.py only: every compute call goes straight into
the shared library; there is no Python or CPU fallback. Loading fails loudly if the library has
not been built (run `python -c "import __graft_entry__ as g; g.build()"` or `make -C virgo-plus_b200`).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VP_LIB") or os.path.join(HERE, "libvirgo_b200.so")  # VP_LIB: development variants

F_DTYPE = np.dtype([("re", "<u8"), ("im", "<u8")])  # == vp_F == virgo::fieldElement
P = (1 << 61) - 1


class VpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"virgo_b200 error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it first (there is no fallback path)")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def _declare(L):
    vp = C.c_void_p
    u64p = C.POINTER(C.c_uint64)
    L.vp_last_error.restype = C.c_char_p
    L.vp_version.restype = C.c_char_p
    L.vp_circuit_load_pws.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.vp_circuit_load_pws_text.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp)]
    L.vp_circuit_random.argtypes = [C.c_int, C.c_int, C.c_uint64, C.POINTER(vp)]
    L.vp_circuit_from_arrays.argtypes = [C.c_int] + [vp] * 10 + [C.POINTER(vp)]
    L.vp_circuit_replicate.argtypes = [vp, C.c_uint64, C.POINTER(vp)]
    L.vp_circuit_expand.argtypes = [vp, C.POINTER(vp)]
    L.vp_circuit_free.argtypes = [vp]
    L.vp_circuit_free.restype = None
    L.vp_circuit_num_layers.argtypes = [vp]
    L.vp_circuit_instances.argtypes = [vp]
    L.vp_circuit_instances.restype = C.c_uint64
    L.vp_circuit_layer_size.argtypes = [vp, C.c_int]
    L.vp_circuit_layer_size.restype = C.c_uint64
    L.vp_circuit_bit_length.argtypes = [vp, C.c_int]
    L.vp_circuit_dad_size.argtypes = [vp, C.c_int, C.c_int]
    L.vp_circuit_dad_size.restype = C.c_uint64
    L.vp_circuit_max_dad_bit_length.argtypes = [vp, C.c_int]
    L.vp_circuit_total_gates.argtypes = [vp]
    L.vp_circuit_total_gates.restype = C.c_uint64
    L.vp_circuit_num_inputs.argtypes = [vp]
    L.vp_circuit_num_inputs.restype = C.c_uint64
    L.vp_circuit_export_layer.argtypes = [vp, C.c_int] + [vp] * 7
    L.vp_circuit_export_dad.argtypes = [vp, C.c_int, C.c_int, vp]
    L.vp_circuit_get_inputs.argtypes = [vp, vp]
    L.vp_circuit_set_inputs.argtypes = [vp, vp]
    L.vp_challenge_count.argtypes = [vp]
    L.vp_challenge_count.restype = C.c_size_t
    L.vp_draw_challenges.argtypes = [vp, C.c_uint, vp]
    L.vp_draw_field.argtypes = [C.c_uint, C.c_size_t, vp]
    L.vp_transcript_len.argtypes = [vp]
    L.vp_transcript_len.restype = C.c_size_t
    L.vp_transcript_to_gkrproof.argtypes = [vp, vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.vp_gkrproof_to_transcript.argtypes = [vp, vp, C.c_size_t, vp]
    L.vp_transcript_text.argtypes = [vp, vp, vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.vp_create.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.vp_nccl_unique_id.argtypes = [vp]
    L.vp_create_sharded.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, C.POINTER(vp)]
    L.vp_destroy.argtypes = [vp]
    L.vp_shard_describe.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.vp_shard_map_index.argtypes = [C.c_uint32] * 3 + [C.POINTER(C.c_uint32)]
    L.vp_destroy.restype = None
    L.vp_set_inputs.argtypes = [vp, vp, C.c_size_t]
    L.vp_evaluate.argtypes = [vp]
    L.vp_get_values.argtypes = [vp, C.c_int, vp, C.c_size_t]
    L.vp_vres.argtypes = [vp, vp, C.c_int, vp]
    L.vp_sumcheck_init_all.argtypes = [vp, vp, C.c_int]
    L.vp_sumcheck_init.argtypes = [vp]
    L.vp_init_phase1.argtypes = [vp, vp]
    L.vp_init_phase2.argtypes = [vp]
    L.vp_init_liu.argtypes = [vp, vp, C.c_int]
    L.vp_round.argtypes = [vp, C.c_int, vp, vp]
    L.vp_finalize1.argtypes = [vp, vp, vp]
    L.vp_finalize2.argtypes = [vp, vp, vp, C.c_int]
    L.vp_finalize_liu.argtypes = [vp, vp, vp]
    L.vp_inner_prod.argtypes = [vp, vp, C.c_size_t, vp]
    L.vp_input_mle.argtypes = [vp, vp, C.c_int, vp]
    L.vp_dot_host.argtypes = [vp, vp, vp, C.c_size_t, vp]
    L.vp_proof_size_bytes.argtypes = [vp]
    L.vp_proof_size_bytes.restype = C.c_uint64
    L.vp_prove_seconds.argtypes = [vp]
    L.vp_prove_seconds.restype = C.c_double
    L.vp_set_challenges.argtypes = [vp, vp, C.c_size_t]
    L.vp_prove.argtypes = [vp, C.c_int, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t]
    L.vp_input_range.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.vp_prove_local.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t]
    L.vp_commit_private.argtypes = [vp, vp, C.c_size_t, vp]
    L.vp_commit_export.argtypes = [vp, vp, vp, vp]
    L.vp_commit_slice_size.argtypes = [vp]
    L.vp_commit_slice_size.restype = C.c_uint64
    L.vp_last_commit_ms.argtypes = [vp]
    L.vp_last_commit_ms.restype = C.c_float
    L.vp_pc_commit.argtypes = [C.c_int, vp, C.c_size_t, C.c_int, vp, vp, vp, vp, C.POINTER(C.c_float)]
    L.vp_pc_commit_public.argtypes = [C.c_int, vp, C.c_size_t, vp, C.c_size_t, C.c_int, vp, vp, vp, vp, vp, C.POINTER(C.c_float)]
    L.vp_commit_public.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, vp, vp]
    L.vp_commit_public_export.argtypes = [vp, vp, vp, vp, vp]
    L.vp_commit_export_interleaved.argtypes = [vp, C.c_int, vp]
    L.vp_fri_commit_steps.argtypes = [vp, vp, C.c_int, vp]
    L.vp_fri_steps.argtypes = [vp]
    L.vp_fri_restart.argtypes = [vp]
    L.vp_fri_export_level.argtypes = [vp, C.c_int, vp, vp]
    L.vp_fft_gkr_rnd_count.argtypes = [C.c_int]
    L.vp_fft_gkr_rnd_count.restype = C.c_size_t
    L.vp_fft_gkr_poly_count.argtypes = [C.c_int]
    L.vp_fft_gkr_poly_count.restype = C.c_size_t
    L.vp_fft_gkr.argtypes = [C.c_int, C.c_int, vp, C.c_size_t, vp, vp, C.c_size_t, vp, C.POINTER(C.c_int), C.POINTER(C.c_int),
                             C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_float)]
    L.vp_pc_fri.argtypes = [C.c_int, vp, C.c_size_t, vp, C.c_size_t, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, C.POINTER(C.c_float)]
    L.vp_prove_fs.argtypes = [vp, C.c_char_p, vp, C.c_size_t, vp, C.c_size_t]
    L.vp_fs_challenges.argtypes = [vp, C.c_char_p, vp, C.c_size_t, vp, C.c_size_t]
    L.vp_verify_fs.argtypes = [vp, C.c_char_p, vp, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.vp_statement_digest.argtypes = [vp, C.c_char_p, vp, vp, vp, vp]
    L.vp_prove_fs_bound.argtypes = [vp, C.c_char_p, vp, C.c_size_t, vp, C.c_size_t, vp]
    L.vp_verify_fs_bound.argtypes = [vp, C.c_char_p, vp, C.c_size_t, vp, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int)]
    L.vp_fs_round_stamps.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.vp_prove_fs_bound_batch.argtypes = [vp, C.c_size_t, vp, C.c_size_t, vp, vp, C.c_size_t, vp, C.c_size_t, vp]
    L.vp_last_batch_outputs.argtypes = [vp, vp, C.c_size_t]
    L.vp_verify_fs_bound_batch.argtypes = [vp, C.c_size_t, vp, C.c_size_t, vp, vp, C.c_size_t, vp, C.c_size_t, vp, vp, vp, vp,
                                           C.c_size_t]
    L.vp_prove_fs_bound_batch_dev.argtypes = [vp, C.c_size_t] + [vp] * 7
    L.vp_verify_fs_bound_batch_dev.argtypes = [vp, C.c_size_t] + [vp] * 8
    L.vp_aggregate_digest.argtypes = [vp, C.c_size_t, vp, vp, vp]
    L.vp_prove_fs_aggregate.argtypes = [vp, C.c_size_t, vp, vp, C.c_size_t, vp, C.c_size_t, vp, vp]
    L.vp_verify_fs_aggregate.argtypes = [vp, C.c_size_t, vp, vp, C.c_size_t, vp, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                         C.POINTER(C.c_int)]
    L.vp_get_transcript.argtypes = [vp, vp, C.c_size_t]
    L.vp_last_prove_ms.argtypes = [vp]
    L.vp_last_prove_ms.restype = C.c_float
    L.vp_last_prove_launches.argtypes = [vp]
    L.vp_last_prove_launches.restype = C.c_uint64
    L.vp_stream.argtypes = [vp]
    L.vp_set_stream.argtypes = [vp, vp]
    L.vp_set_profiling.argtypes = [vp, C.c_int]
    L.vp_shard_eval_ranges.argtypes = [vp, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.vp_selftest_field.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.vp_verify.argtypes = [vp, C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.vp_set_lanes.argtypes = [vp, C.c_int]
    L.vp_set_lanes.restype = C.c_int
    L.vp_get_profile.argtypes = [vp, vp, vp, vp, C.c_int]
    L.vp_stream.restype = C.c_void_p
    L.vp_sumcheck_create.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
    L.vp_sumcheck_load.argtypes = [vp, vp, vp, vp]
    L.vp_sumcheck_fill_random.argtypes = [vp, C.c_uint64]
    L.vp_sumcheck_export.argtypes = [vp, vp, vp, vp]
    L.vp_sumcheck_run.argtypes = [vp, vp, vp, C.POINTER(C.c_float)]
    L.vp_sumcheck_run_fused.argtypes = [vp, vp, vp, C.POINTER(C.c_float)]
    L.vp_sumcheck_round_ms.argtypes = [vp, vp]
    L.vp_sumcheck_pass_stamps.argtypes = [vp, vp, C.c_int]
    L.vp_sumcheck_destroy.argtypes = [vp]
    L.vp_sumcheck_destroy.restype = None


EXPORTED_SYMBOLS = None  # filled by tests from the header


def _ck(rc):
    if rc != 0:
        raise VpError(rc, lib().vp_last_error().decode())


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _context(context):
    context = bytes(context)
    if len(context) != 32:
        raise ValueError("a Fiat-Shamir context is 32 bytes")
    return context


def _contexts(B, contexts):
    """B contexts (B `bytes` of 32 or a [B, 32] uint8 array) as one contiguous [B, 32] uint8 array"""
    if isinstance(contexts, np.ndarray):
        if contexts.dtype != np.uint8 or contexts.shape != (B, 32):
            raise ValueError(f"contexts must be a [{B}, 32] uint8 array, got {contexts.dtype} {contexts.shape}")
        return np.ascontiguousarray(contexts)
    contexts = list(contexts)
    if len(contexts) != B:
        raise ValueError(f"{B} statements need {B} contexts, got {len(contexts)}")
    return np.frombuffer(b"".join(_context(c) for c in contexts), np.uint8).reshape(B, 32)


def _verdict(call):
    """call(accept, fail_code, fail_layer) with the three int out-parameters -> (accept, fail_code, fail_layer)"""
    a, c, l = C.c_int(0), C.c_int(0), C.c_int(0)
    _ck(call(C.byref(a), C.byref(c), C.byref(l)))
    return bool(a.value), c.value, l.value


def fe(re, im=0):
    """one field element as a 0-d structured array"""
    a = np.zeros((), dtype=F_DTYPE)
    a["re"] = re
    a["im"] = im
    return a


def fe_array(pairs):
    a = np.zeros(len(pairs), dtype=F_DTYPE)
    for i, (re, im) in enumerate(pairs):
        a[i] = (re, im)
    return a


class Circuit:
    """Host-side layered circuit (vp_circuit)."""

    def __init__(self, handle):
        self.h = C.c_void_p(handle)

    @staticmethod
    def _new(fn, *args):
        h = C.c_void_p()
        _ck(fn(*args, C.byref(h)))
        return Circuit(h.value)

    @classmethod
    def load_pws(cls, path):
        return cls._new(lib().vp_circuit_load_pws, os.fsencode(path))

    @classmethod
    def from_pws_text(cls, text):
        if isinstance(text, str):
            text = text.encode()
        return cls._new(lib().vp_circuit_load_pws_text, text, len(text))

    @classmethod
    def random(cls, n_layers, log_size, seed):
        return cls._new(lib().vp_circuit_random, n_layers, log_size, seed)

    @classmethod
    def from_arrays(cls, layer_size, ty, l, u, v, lv=None, c=None, is_assert=None, dad_size=None, dad_id=None):
        layer_size = np.ascontiguousarray(layer_size, dtype=np.uint64)
        ty = np.ascontiguousarray(ty, dtype=np.uint8)
        l = np.ascontiguousarray(l, dtype=np.int32)
        u = np.ascontiguousarray(u, dtype=np.uint64)
        v = np.ascontiguousarray(v, dtype=np.uint64)
        lv = None if lv is None else np.ascontiguousarray(lv, dtype=np.uint64)
        c = None if c is None else np.ascontiguousarray(c, dtype=F_DTYPE)
        is_assert = None if is_assert is None else np.ascontiguousarray(is_assert, dtype=np.uint8)
        dad_size = None if dad_size is None else np.ascontiguousarray(dad_size, dtype=np.uint64)
        dad_id = None if dad_id is None else np.ascontiguousarray(dad_id, dtype=np.uint64)
        keep = (layer_size, ty, l, u, v, lv, c, is_assert, dad_size, dad_id)
        return cls._new(lib().vp_circuit_from_arrays, len(layer_size), *[_ptr(a) for a in keep])

    def replicate(self, k):
        return Circuit._new(lib().vp_circuit_replicate, self.h, k)

    def expand(self):
        return Circuit._new(lib().vp_circuit_expand, self.h)

    def __del__(self):
        try:
            if self.h:
                lib().vp_circuit_free(self.h)
                self.h = None
        except Exception:
            pass

    # ---- metadata
    @property
    def n_layers(self):
        return lib().vp_circuit_num_layers(self.h)

    @property
    def instances(self):
        return lib().vp_circuit_instances(self.h)

    def layer_size(self, i):
        return lib().vp_circuit_layer_size(self.h, i)

    def bit_length(self, i):
        return lib().vp_circuit_bit_length(self.h, i)

    def dad_size(self, i, l):
        return lib().vp_circuit_dad_size(self.h, i, l)

    def max_dad_bit_length(self, i):
        return lib().vp_circuit_max_dad_bit_length(self.h, i)

    @property
    def total_gates(self):
        return lib().vp_circuit_total_gates(self.h)

    @property
    def num_inputs(self):
        return lib().vp_circuit_num_inputs(self.h)

    @property
    def challenge_count(self):
        return lib().vp_challenge_count(self.h)

    @property
    def transcript_len(self):
        return lib().vp_transcript_len(self.h)

    def export_layer(self, i):
        n = self.layer_size(i)
        out = dict(
            ty=np.zeros(n, np.uint8), l=np.zeros(n, np.int32), u=np.zeros(n, np.uint32), v=np.zeros(n, np.uint32),
            lv=np.zeros(n, np.uint32), c=np.zeros(n, F_DTYPE), is_assert=np.zeros(n, np.uint8),
        )
        _ck(lib().vp_circuit_export_layer(self.h, i, *[_ptr(out[k]) for k in ("ty", "l", "u", "v", "lv", "c", "is_assert")]))
        return out

    def export_dad(self, i, l):
        out = np.zeros(self.dad_size(i, l), np.uint32)
        if len(out):
            _ck(lib().vp_circuit_export_dad(self.h, i, l, _ptr(out)))
        return out

    def inputs(self):
        out = np.zeros(self.num_inputs, np.uint64)
        _ck(lib().vp_circuit_get_inputs(self.h, _ptr(out)))
        return out

    def set_inputs(self, a):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        assert len(a) == self.num_inputs
        _ck(lib().vp_circuit_set_inputs(self.h, _ptr(a)))

    def draw_challenges(self, seed=3396):
        out = np.zeros(self.challenge_count, F_DTYPE)
        _ck(lib().vp_draw_challenges(self.h, seed, _ptr(out)))
        return out

    def to_gkrproof(self, transcript):
        """bytes in the layout of GKRProof::write (src/GKRProof.hpp:23-58) + {Vres, input MLE} trailer"""
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        assert len(tr) == self.transcript_len
        n = C.c_size_t()
        _ck(lib().vp_transcript_to_gkrproof(self.h, _ptr(tr), None, 0, C.byref(n)))
        buf = np.zeros(n.value, np.uint8)
        _ck(lib().vp_transcript_to_gkrproof(self.h, _ptr(tr), _ptr(buf), len(buf), C.byref(n)))
        return buf.tobytes()

    def from_gkrproof(self, data):
        buf = np.frombuffer(data, dtype=np.uint8).copy()
        tr = np.zeros(self.transcript_len, F_DTYPE)
        _ck(lib().vp_gkrproof_to_transcript(self.h, _ptr(buf), len(buf), _ptr(tr)))
        return tr

    def transcript_text(self, transcript, challenges=None):
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        ch = np.ascontiguousarray(self.draw_challenges() if challenges is None else challenges, dtype=F_DTYPE)
        n = C.c_size_t()
        _ck(lib().vp_transcript_text(self.h, _ptr(tr), _ptr(ch), None, 0, C.byref(n)))
        buf = np.zeros(n.value, np.uint8)
        _ck(lib().vp_transcript_text(self.h, _ptr(tr), _ptr(ch), _ptr(buf), len(buf), C.byref(n)))
        return buf.tobytes().decode()

    def fs_challenges(self, seed32, transcript):
        """the challenges of a Fiat-Shamir transcript, recomputed from the messages (host only)"""
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        ch = np.zeros(self.challenge_count, F_DTYPE)
        _ck(lib().vp_fs_challenges(self.h, bytes(seed32), _ptr(tr), len(tr), _ptr(ch), len(ch)))
        return ch

    def flat(self):
        """Flat arrays of this circuit (instances must be 1), concatenated over layers (used by tests)."""
        assert self.instances == 1
        n = self.n_layers
        layers = [self.export_layer(i) for i in range(n)]
        sizes = np.array([self.layer_size(i) for i in range(n)], np.uint64)
        gate_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        cat = lambda k, dt: np.ascontiguousarray(np.concatenate([L[k] for L in layers]).astype(dt))
        dad_size = np.zeros((n, n), np.uint64)
        dad_off = np.zeros(n * n + 1, np.uint64)
        ids = []
        o = 0
        for i in range(n):
            for l in range(n):
                dad_off[i * n + l] = o
                if l < i:
                    d = self.export_dad(i, l)
                    dad_size[i, l] = len(d)
                    ids.append(d)
                    o += len(d)
        dad_off[n * n] = o
        dad_id = np.ascontiguousarray(np.concatenate(ids) if ids else np.zeros(0, np.uint32), dtype=np.uint32)
        return dict(
            n_layers=n, layer_size=sizes, gate_off=gate_off, ty=cat("ty", np.uint8), l=cat("l", np.int32),
            u=cat("u", np.uint32), v=cat("v", np.uint32), lv=cat("lv", np.uint32), c=cat("c", F_DTYPE),
            is_assert=cat("is_assert", np.uint8), dad_size=np.ascontiguousarray(dad_size.reshape(-1)),
            dad_off=dad_off, dad_id=dad_id if len(dad_id) else np.zeros(1, np.uint32), inputs=self.inputs(),
        )


def nccl_unique_id():
    out = np.zeros(128, np.uint8)
    _ck(lib().vp_nccl_unique_id(_ptr(out)))
    return out


def selftest_field(op, a, b, c, device=0):
    a, b, c = (np.ascontiguousarray(x, dtype=F_DTYPE) for x in (a, b, c))
    out = np.zeros(len(a), F_DTYPE)
    _ck(lib().vp_selftest_field(device, op, _ptr(a), _ptr(b), _ptr(c), _ptr(out), len(a)))
    return out


def pc_commit(array, log_len, device=0, want_arrays=True, want_l_eval=True):
    """commit phase of the polynomial commitment on a host array (vp_pc_commit) -> dict(root, l_eval, leaf_hash, tree, ms)"""
    a = np.ascontiguousarray(array, dtype=F_DTYPE)
    ss = 1 << (log_len - 1)
    root = np.zeros(32, np.uint8)
    l_eval = np.zeros(65 * ss, F_DTYPE) if want_arrays and want_l_eval else None
    leaf = np.zeros(ss // 2 * 32, np.uint8) if want_arrays else None
    tree = np.zeros(ss * 32, np.uint8) if want_arrays else None
    ms = C.c_float()
    _ck(lib().vp_pc_commit(device, _ptr(a), len(a), log_len, _ptr(root), _ptr(l_eval), _ptr(leaf), _ptr(tree), C.byref(ms)))
    return dict(root=root.tobytes(), l_eval=l_eval, leaf_hash=leaf, tree=tree, slice_size=ss, ms=ms.value)


def pc_commit_public(array, pub, log_len, device=0, want_arrays=True):
    """commit_private_array + commit_public_array on host arrays -> dict(root_l, root_h, all_sum, h_eval, vow, ms)"""
    a = np.ascontiguousarray(array, dtype=F_DTYPE)
    q = np.ascontiguousarray(pub, dtype=F_DTYPE)
    N = 1 << (log_len - 1)
    root_l, root_h = np.zeros(32, np.uint8), np.zeros(32, np.uint8)
    all_sum = np.zeros(65, F_DTYPE)
    h_eval = np.zeros(65 * N, F_DTYPE) if want_arrays else None
    vow = np.zeros(64 * N, F_DTYPE) if want_arrays else None
    ms = C.c_float()
    _ck(lib().vp_pc_commit_public(device, _ptr(a), len(a), _ptr(q), len(q), log_len, _ptr(root_l), _ptr(root_h), _ptr(all_sum), _ptr(h_eval),
                                  _ptr(vow), C.byref(ms)))
    return dict(root_l=root_l.tobytes(), root_h=root_h.tobytes(), all_sum=all_sum, h_eval=h_eval, vow=vow, slice_size=N, ms=ms.value)


def pc_fri(array, pub, log_len, randomness, device=0, want_arrays=True):
    """both commitments of host arrays, then one FRI commit step per fold challenge (fri::commit_phase_step)
    -> dict(root_l, root_h, roots [steps], codes [per level], trees [per level], ms = device time of the steps)"""
    a = np.ascontiguousarray(array, dtype=F_DTYPE)
    q = np.ascontiguousarray(pub, dtype=F_DTYPE)
    r = np.ascontiguousarray(randomness, dtype=F_DTYPE)
    N, steps = 1 << (log_len - 1), len(r)
    sizes = [N >> (l + 1) for l in range(steps)]
    root_l, root_h, roots = np.zeros(32, np.uint8), np.zeros(32, np.uint8), np.zeros(32 * max(steps, 1), np.uint8)
    codes = np.zeros(64 * sum(sizes), F_DTYPE) if want_arrays else None
    trees = np.zeros(32 * sum(sizes), np.uint8) if want_arrays else None
    ms = C.c_float()
    _ck(lib().vp_pc_fri(device, _ptr(a), len(a), _ptr(q), len(q), log_len, _ptr(r), steps, _ptr(root_l), _ptr(root_h), _ptr(roots), _ptr(codes),
                        _ptr(trees), C.byref(ms)))
    out = dict(root_l=root_l.tobytes(), root_h=root_h.tobytes(), roots=[roots[32 * l:32 * l + 32].tobytes() for l in range(steps)], codes=[],
               trees=[], ms=ms.value)
    o = 0
    for m in sizes if want_arrays else []:
        out["codes"].append(codes[64 * o:64 * (o + m)])
        out["trees"].append(trees[32 * o:32 * (o + m)].tobytes())
        o += m
    return out


def draw_field(n, seed=3396):
    """the first n values of fieldElement::random() after srand(seed)"""
    out = np.zeros(n, F_DTYPE)
    _ck(lib().vp_draw_field(seed, n, _ptr(out)))
    return out


def fft_gkr_release():
    lib().vp_fft_gkr_release()


def fft_gkr_rnd_count(lg):
    return int(lib().vp_fft_gkr_rnd_count(lg))


def fft_gkr(lg, rnd, device=0, want_layers=True):
    """the polynomial commitment's inner GKR (fft_circuit_gkr::fft_gkr) with the randomness handed in
    -> dict(layers, polys [rounds, 3], claims, proof_size, ok, verifier_seconds, prover_seconds, device_ms)"""
    r = np.ascontiguousarray(rnd, dtype=F_DTYPE)
    n, npoly = 1 << lg, int(lib().vp_fft_gkr_poly_count(lg))
    layers = np.zeros((lg + 2) * n + 64 * n + 64, F_DTYPE) if want_layers else None
    polys, claims = np.zeros(3 * npoly, F_DTYPE), np.zeros(4 + lg + 2, F_DTYPE)
    ps, ok, vt, pt, ms = C.c_int(), C.c_int(), C.c_double(), C.c_double(), C.c_float()
    _ck(lib().vp_fft_gkr(device, lg, _ptr(r), len(r), _ptr(layers), _ptr(polys), npoly, _ptr(claims), C.byref(ps), C.byref(ok), C.byref(vt),
                         C.byref(pt), C.byref(ms)))
    return dict(layers=layers, polys=polys.reshape(npoly, 3), claims=claims, proof_size=ps.value, ok=bool(ok.value),
                verifier_seconds=vt.value, prover_seconds=pt.value, device_ms=ms.value)


def shard_describe(circuit, world, rank, layer, phase):
    out = np.zeros(10 * 256, np.uint32)
    n = C.c_size_t()
    _ck(lib().vp_shard_describe(circuit.h, world, rank, layer, phase, _ptr(out), len(out), C.byref(n)))
    keys = ("bits", "live", "sharded", "m", "row_lo", "row_hi", "local_len", "present", "n_blocks", "reversed")
    return [dict(zip(keys, (int(x) for x in out[10 * t:10 * t + 10]))) for t in range(n.value)]


def shard_eval_ranges(circuit, world, rank):
    n = circuit.n_layers
    lo, hi = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    _ck(lib().vp_shard_eval_ranges(circuit.h, world, rank, _ptr(lo), _ptr(hi)))
    return lo, hi


def shard_map_index(lo, hi, idx):
    loc = C.c_uint32()
    rc = lib().vp_shard_map_index(lo, hi, idx, C.byref(loc))
    assert rc >= 0, "shard_global(shard_local(idx)) != idx"
    return (rc == 1), loc.value


class Prover:
    """vp_ctx: the GPU prover (mirrors the method names of the reference's `prover`, src/prover.h:12-42).
    world > 1: this process is `rank` of a sharded context (one process per GPU, whole-proof mode only)."""

    def __init__(self, circuit, device=0, rank=0, world=1, nccl_id=None):
        self.circuit = circuit
        self.device = device
        h = C.c_void_p()
        if world == 1:
            _ck(lib().vp_create(circuit.h, device, C.byref(h)))
        else:
            nccl_id = np.ascontiguousarray(nccl_id, dtype=np.uint8)
            assert len(nccl_id) == 128
            _ck(lib().vp_create_sharded(circuit.h, device, rank, world, _ptr(nccl_id), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            lib().vp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_inputs(self, a):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        _ck(lib().vp_set_inputs(self.h, _ptr(a), len(a)))

    def evaluate(self):
        _ck(lib().vp_evaluate(self.h))

    def values(self, layer):
        n = self.circuit.layer_size(layer) * self.circuit.instances
        out = np.zeros(n, F_DTYPE)
        _ck(lib().vp_get_values(self.h, layer, _ptr(out), n))
        return out

    def Vres(self, r):
        r = np.ascontiguousarray(r, dtype=F_DTYPE)
        out = np.zeros(1, F_DTYPE)
        _ck(lib().vp_vres(self.h, _ptr(r), len(r), _ptr(out)))
        return out[0]

    def sumcheckInitAll(self, r):
        r = np.ascontiguousarray(r, dtype=F_DTYPE)
        _ck(lib().vp_sumcheck_init_all(self.h, _ptr(r), len(r)))

    def sumcheckInit(self):
        _ck(lib().vp_sumcheck_init(self.h))

    def sumcheckInitPhase1(self, assert_random):
        a = np.ascontiguousarray(assert_random, dtype=F_DTYPE).reshape(1)
        _ck(lib().vp_init_phase1(self.h, _ptr(a)))

    def sumcheckInitPhase2(self):
        _ck(lib().vp_init_phase2(self.h))

    def sumcheckInitLiu(self, sig):
        s = np.ascontiguousarray(sig, dtype=F_DTYPE)
        _ck(lib().vp_init_liu(self.h, _ptr(s), len(s)))

    def _round(self, phase, prev):
        p = np.ascontiguousarray(prev, dtype=F_DTYPE).reshape(1)
        out = np.zeros(3, F_DTYPE)
        _ck(lib().vp_round(self.h, phase, _ptr(p), _ptr(out)))
        return out

    def sumcheckUpdatePhase1(self, prev):
        return self._round(1, prev)

    def sumcheckUpdatePhase2(self, prev):
        return self._round(2, prev)

    def sumcheckLiuUpdate(self, prev):
        return self._round(3, prev)

    def sumcheckFinalize1(self, prev):
        p = np.ascontiguousarray(prev, dtype=F_DTYPE).reshape(1)
        out = np.zeros(1, F_DTYPE)
        _ck(lib().vp_finalize1(self.h, _ptr(p), _ptr(out)))
        return out[0]

    def sumcheckFinalize2(self, prev, n):
        p = np.ascontiguousarray(prev, dtype=F_DTYPE).reshape(1)
        out = np.zeros(n, F_DTYPE)
        _ck(lib().vp_finalize2(self.h, _ptr(p), _ptr(out), n))
        return out

    def sumcheckLiuFinalize(self, prev):
        p = np.ascontiguousarray(prev, dtype=F_DTYPE).reshape(1)
        out = np.zeros(1, F_DTYPE)
        _ck(lib().vp_finalize_liu(self.h, _ptr(p), _ptr(out)))
        return out[0]

    def inner_prod(self, pub):
        pub = np.ascontiguousarray(pub, dtype=F_DTYPE)
        out = np.zeros(1, F_DTYPE)
        _ck(lib().vp_inner_prod(self.h, _ptr(pub), len(pub), _ptr(out)))
        return out[0]

    def input_mle(self, r):
        r = np.ascontiguousarray(r, dtype=F_DTYPE)
        out = np.zeros(1, F_DTYPE)
        _ck(lib().vp_input_mle(self.h, _ptr(r), len(r), _ptr(out)))
        return out[0]

    def proofSize(self):
        return lib().vp_proof_size_bytes(self.h) / 1024.0

    def proveTime(self):
        return lib().vp_prove_seconds(self.h)

    # ---- whole proof
    def set_challenges(self, ch):
        ch = np.ascontiguousarray(ch, dtype=F_DTYPE)
        _ck(lib().vp_set_challenges(self.h, _ptr(ch), len(ch)))

    def prove(self, inputs=None, challenges=None, transcript=None):
        """host_io proof when inputs/challenges are given (host numpy buffers), else device-resident."""
        if inputs is not None:
            inputs = np.ascontiguousarray(inputs, dtype=np.uint64)
            challenges = np.ascontiguousarray(challenges, dtype=F_DTYPE)
            if transcript is None:
                transcript = np.zeros(self.circuit.transcript_len, F_DTYPE)
            _ck(lib().vp_prove(self.h, 1, _ptr(inputs), len(inputs), _ptr(challenges), len(challenges),
                               _ptr(transcript), len(transcript)))
            return transcript
        _ck(lib().vp_prove(self.h, 0, None, 0, None, 0, None, 0))
        return None

    def commit_private(self, mask=None):
        """prover::commit_private (prover.cpp:524-530) on the device: the Merkle root of the input layer's commitment"""
        m = np.zeros(1, F_DTYPE) if mask is None else np.ascontiguousarray(mask, dtype=F_DTYPE)
        root = np.zeros(32, np.uint8)
        _ck(lib().vp_commit_private(self.h, _ptr(m), len(m), _ptr(root)))
        return root.tobytes()

    def commit_public(self, pub, mask=None):
        """prover::commit_public's commitment part on the device -> (root_h, all_sum[65])"""
        q = np.ascontiguousarray(pub, dtype=F_DTYPE)
        m = np.zeros(1, F_DTYPE) if mask is None else np.ascontiguousarray(mask, dtype=F_DTYPE)
        root, all_sum = np.zeros(32, np.uint8), np.zeros(65, F_DTYPE)
        _ck(lib().vp_commit_public(self.h, _ptr(q), len(q), _ptr(m), len(m), _ptr(root), _ptr(all_sum)))
        return root.tobytes(), all_sum

    def fri_commit_steps(self, randomness):
        """fri::commit_phase_step per fold challenge on the virtual oracle commit_public left on the device -> [root]"""
        r = np.ascontiguousarray(randomness, dtype=F_DTYPE)
        roots = np.zeros(32 * max(len(r), 1), np.uint8)
        _ck(lib().vp_fri_commit_steps(self.h, _ptr(r), len(r), _ptr(roots)))
        return [roots[32 * l:32 * l + 32].tobytes() for l in range(len(r))]

    @property
    def fri_steps(self):
        return int(lib().vp_fri_steps(self.h))

    def fri_restart(self):
        _ck(lib().vp_fri_restart(self.h))

    def fri_export_level(self, lvl):
        m = int(lib().vp_commit_slice_size(self.h)) >> (lvl + 1)
        code, tree = np.zeros(64 * m, F_DTYPE), np.zeros(32 * m, np.uint8)
        _ck(lib().vp_fri_export_level(self.h, lvl, _ptr(code), _ptr(tree)))
        return code, tree.tobytes()

    def commit_export_interleaved(self, which):
        out = np.zeros(64 * int(lib().vp_commit_slice_size(self.h)), F_DTYPE)
        _ck(lib().vp_commit_export_interleaved(self.h, which, _ptr(out)))
        return out

    def commit_export(self):
        ss = int(lib().vp_commit_slice_size(self.h))
        l_eval, leaf, tree = np.zeros(65 * ss, F_DTYPE), np.zeros(ss // 2 * 32, np.uint8), np.zeros(ss * 32, np.uint8)
        _ck(lib().vp_commit_export(self.h, _ptr(l_eval), _ptr(leaf), _ptr(tree)))
        return dict(l_eval=l_eval, leaf_hash=leaf, tree=tree, slice_size=ss)

    @property
    def last_commit_ms(self):
        return float(lib().vp_last_commit_ms(self.h))

    def _proof_arrays(self, *B):
        """zeroed transcript and challenge arrays of one proof, or of B proofs ([B, n]) when B is given"""
        return np.zeros(B + (self.circuit.transcript_len,), F_DTYPE), np.zeros(B + (self.circuit.challenge_count,), F_DTYPE)

    def prove_fs(self, seed32):
        """Fiat-Shamir mode: (transcript, challenges) with every challenge hashed from the messages before it"""
        tr, ch = self._proof_arrays()
        _ck(lib().vp_prove_fs(self.h, bytes(seed32), _ptr(tr), len(tr), _ptr(ch), len(ch)))
        return tr, ch

    def verify_fs(self, seed32, transcript):
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        return _verdict(lambda *v: lib().vp_verify_fs(self.h, bytes(seed32), _ptr(tr), len(tr), *v))

    def statement_digest(self, context=bytes(32)):
        """the statement of the resident inputs (include/virgo_b200.h) -> dict(circuit, inputs, outputs, statement), 32 bytes each"""
        out = [np.zeros(32, np.uint8) for _ in range(4)]
        _ck(lib().vp_statement_digest(self.h, _context(context), *[_ptr(x) for x in out]))
        return dict(zip(("circuit", "inputs", "outputs", "statement"), (x.tobytes() for x in out)))

    def prove_fs_bound(self, context=bytes(32)):
        """statement-bound Fiat-Shamir proof -> (transcript, challenges, statement); == prove_fs(statement)"""
        tr, ch = self._proof_arrays()
        st = np.zeros(32, np.uint8)
        _ck(lib().vp_prove_fs_bound(self.h, _context(context), _ptr(tr), len(tr), _ptr(ch), len(ch), _ptr(st)))
        return tr, ch, st.tobytes()

    def _batch_statements(self, inputs, contexts):
        """checked (inputs [B, n_inputs] uint64, contexts [B, 32] uint8) of a batch call"""
        n_in = self.circuit.layer_size(0) * self.circuit.instances
        inputs = np.asarray(inputs)
        if inputs.ndim != 2 or inputs.shape[1] != n_in or inputs.shape[0] < 1:
            raise ValueError(f"inputs must be a [B, {n_in}] array with B >= 1, got shape {inputs.shape}")
        if inputs.dtype.kind not in "ui":
            raise ValueError(f"inputs must be integers, got {inputs.dtype}")
        return np.ascontiguousarray(inputs, dtype=np.uint64), _contexts(inputs.shape[0], contexts)

    def _n_outputs(self):
        return self.circuit.layer_size(self.circuit.n_layers - 1) * self.circuit.instances

    def prove_fs_bound_batch(self, inputs, contexts, return_outputs=False):
        """B independent statement-bound proofs of this circuit in one pass: inputs [B, n_inputs], contexts B `bytes` of 32
        or a [B, 32] uint8 array -> (transcripts [B, n_tr], challenges [B, n_chal], statements [B, 32] uint8), and with
        return_outputs the statements' output layers [B, n_outputs] as well; proof b == prove_fs_bound(contexts[b]) after
        set_inputs(inputs[b]). The resident inputs and values are not changed."""
        inputs, ctx = self._batch_statements(inputs, contexts)
        B = inputs.shape[0]
        tr, ch = self._proof_arrays(B)
        st = np.zeros((B, 32), np.uint8)
        _ck(lib().vp_prove_fs_bound_batch(self.h, B, _ptr(inputs), inputs.size, _ptr(ctx), _ptr(tr), tr.size, _ptr(ch), ch.size,
                                          _ptr(st)))
        if not return_outputs:
            return tr, ch, st
        out = np.zeros((B, self._n_outputs()), F_DTYPE)
        _ck(lib().vp_last_batch_outputs(self.h, _ptr(out), out.size))
        return tr, ch, st, out

    def verify_fs_bound_batch(self, inputs, contexts, outputs, transcripts, return_challenges=False):
        """B statement-bound proofs checked in one pass: inputs and contexts as prove_fs_bound_batch, the claimed outputs
        [B, n_outputs] and the transcripts [B, n_tr] (F_DTYPE) -> (accept bool[B], fail_code int32[B], fail_layer int32[B]),
        and with return_challenges the challenges [B, n_chal]; verdict b == verify_fs_bound(contexts[b], outputs[b],
        transcripts[b]) after set_inputs(inputs[b]). The resident inputs, values and challenges are not changed."""
        inputs, ctx = self._batch_statements(inputs, contexts)
        B = inputs.shape[0]
        for name, a, n in (("outputs", outputs, self._n_outputs()), ("transcripts", transcripts, self.circuit.transcript_len)):
            if not isinstance(a, np.ndarray) or a.dtype != F_DTYPE or a.shape != (B, n):
                raise ValueError(f"{name} must be a [{B}, {n}] field-element array, got "
                                 f"{getattr(a, 'dtype', type(a))} {getattr(a, 'shape', None)}")
        out, tr = np.ascontiguousarray(outputs), np.ascontiguousarray(transcripts)
        acc, code, layer = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
        ch = np.zeros((B, self.circuit.challenge_count), F_DTYPE) if return_challenges else None
        _ck(lib().vp_verify_fs_bound_batch(self.h, B, _ptr(inputs), inputs.size, _ptr(ctx), _ptr(out), out.size, _ptr(tr), tr.size,
                                           _ptr(acc), _ptr(code), _ptr(layer), _ptr(ch), 0 if ch is None else ch.size))
        res = (acc.astype(bool), code, layer)
        return res + (ch,) if return_challenges else res

    # ---- batches in device memory (torch CUDA tensors)
    def _cuda_batch(self, arrays):
        """checks (name, tensor, dtype, shape) of a device-memory batch call: a contiguous CUDA tensor on this context's
        device with that dtype and shape (B taken from the first) -> B; then runs the next call on the current torch stream"""
        import torch
        dev = getattr(self, "device", 0)
        B = None
        for name, t, dtype, shape in arrays:
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"{name} must be a torch tensor, got {type(t)}")
            if t.dtype != dtype:
                raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
            if B is None:
                B = t.shape[0] if t.dim() >= 1 else 0
                if not 1 <= B <= 65535:
                    raise ValueError(f"{name} must hold 1 to 65535 statements, got shape {tuple(t.shape)}")
            want = (B,) + shape
            if tuple(t.shape) != want:
                raise ValueError(f"{name} must have shape {list(want)}, got {list(t.shape)}")
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
        for name, t, _, _ in arrays:
            if t.device.type != "cuda" or (t.device.index or 0) != dev:
                raise ValueError(f"{name} must be on cuda:{dev}, got {t.device}")
        # the context runs on the current stream; vp_set_stream waits for the context's previous stream, so it is called only
        # when the context's actual stream (vp_stream) is another one. torch's default stream is the legacy NULL stream,
        # cudaStreamLegacy (1) to the runtime.
        s = torch.cuda.current_stream(dev).cuda_stream or 1
        if (self.stream or 0) != s:
            self.set_stream(s)
        return B

    def _field_tensors(self, B, *counts):
        import torch
        return [torch.empty((B, n, 2), dtype=torch.int64, device=f"cuda:{self.device}") for n in counts]

    def prove_fs_bound_batch_cuda(self, inputs, contexts, challenges=False, outputs=False):
        """prove_fs_bound_batch on CUDA tensors, queued on torch.cuda.current_stream() without waiting for it. The context
        moves onto that stream, so later calls of this Prover (host-memory ones too) run there until the next set_stream;
        a change of the current stream costs one host synchronisation (of the context's previous stream). inputs int64
        [B, n_inputs], contexts uint8 [B, 32] -> (transcripts int64 [B, n_tr, 2] as (re, im), challenges [B, n_chal, 2] or
        None, statements uint8 [B, 32], outputs [B, n_outputs, 2] or None, status int32 [B]). status b: 0 proved, 1 an input
        >= p, 2 + l an assert gate of layer l is non-zero; the rows of a failed statement are zero."""
        import torch
        n_in = self.circuit.layer_size(0) * self.circuit.instances
        B = self._cuda_batch([("inputs", inputs, torch.int64, (n_in,)), ("contexts", contexts, torch.uint8, (32,))])
        tr, ch, out = self._field_tensors(B, self.circuit.transcript_len, self.circuit.challenge_count if challenges else 0,
                                          self._n_outputs() if outputs else 0)
        st = torch.empty((B, 32), dtype=torch.uint8, device=tr.device)
        status = torch.empty(B, dtype=torch.int32, device=tr.device)
        ch, out = (ch if challenges else None), (out if outputs else None)
        _ck(lib().vp_prove_fs_bound_batch_dev(self.h, B, inputs.data_ptr(), contexts.data_ptr(), tr.data_ptr(),
                                              None if ch is None else ch.data_ptr(), None if out is None else out.data_ptr(),
                                              st.data_ptr(), status.data_ptr()))
        return tr, ch, st, out, status

    def verify_fs_bound_batch_cuda(self, inputs, contexts, outputs, transcripts, challenges=False):
        """verify_fs_bound_batch on CUDA tensors, queued on torch.cuda.current_stream() without waiting for it (the context
        moves onto that stream, as in prove_fs_bound_batch_cuda): inputs int64
        [B, n_inputs], contexts uint8 [B, 32], outputs int64 [B, n_outputs, 2], transcripts int64 [B, n_tr, 2] -> (accept,
        fail_code, fail_layer int32 [B], challenges [B, n_chal, 2] or None). fail_code 9: an input or output of the statement
        is not canonical."""
        import torch
        n_in = self.circuit.layer_size(0) * self.circuit.instances
        B = self._cuda_batch([("inputs", inputs, torch.int64, (n_in,)), ("contexts", contexts, torch.uint8, (32,)),
                              ("outputs", outputs, torch.int64, (self._n_outputs(), 2)),
                              ("transcripts", transcripts, torch.int64, (self.circuit.transcript_len, 2))])
        acc, code, layer = (torch.empty(B, dtype=torch.int32, device=inputs.device) for _ in range(3))
        ch = self._field_tensors(B, self.circuit.challenge_count)[0] if challenges else None
        _ck(lib().vp_verify_fs_bound_batch_dev(self.h, B, inputs.data_ptr(), contexts.data_ptr(), outputs.data_ptr(),
                                               transcripts.data_ptr(), acc.data_ptr(), code.data_ptr(), layer.data_ptr(),
                                               None if ch is None else ch.data_ptr()))
        return acc, code, layer, ch

    def verify_fs_bound(self, context, outputs, transcript):
        """(accept, fail_code, fail_layer) of a statement-bound proof for the claimed outputs and this context's inputs"""
        out = np.ascontiguousarray(outputs, dtype=F_DTYPE)
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        return _verdict(lambda *v: lib().vp_verify_fs_bound(self.h, _context(context), _ptr(out), len(out), _ptr(tr), len(tr), *v))

    def _aggregate_contexts(self, B, contexts):
        """checked contexts [B, 32] uint8 of an aggregate call: 1 <= B <= 65535 statements dividing the instances"""
        N = self.circuit.instances
        if not isinstance(B, (int, np.integer)) or isinstance(B, bool) or not 1 <= B <= 65535:
            raise ValueError(f"B must be an integer in [1, 65535], got {B!r}")
        if N % B:
            raise ValueError(f"{B} statements do not divide the {N} instances")
        return _contexts(B, contexts)

    def aggregate_digest(self, B, contexts):
        """the B statements of the resident inputs (statement b: instances [b K, (b + 1) K), K = instances / B) and their
        aggregate (include/virgo_b200.h) -> (statements [B, 32] uint8, aggregate 32 bytes)"""
        ctx = self._aggregate_contexts(B, contexts)
        st, agg = np.zeros((B, 32), np.uint8), np.zeros(32, np.uint8)
        _ck(lib().vp_aggregate_digest(self.h, B, _ptr(ctx), _ptr(st), _ptr(agg)))
        return st, agg.tobytes()

    def prove_fs_aggregate(self, B, contexts):
        """one Fiat-Shamir proof of B statements with their own contexts -> (transcript, challenges, statements [B, 32] uint8,
        aggregate); == prove_fs(aggregate)"""
        ctx = self._aggregate_contexts(B, contexts)
        tr, ch = self._proof_arrays()
        st, agg = np.zeros((B, 32), np.uint8), np.zeros(32, np.uint8)
        _ck(lib().vp_prove_fs_aggregate(self.h, B, _ptr(ctx), _ptr(tr), len(tr), _ptr(ch), len(ch), _ptr(st), _ptr(agg)))
        return tr, ch, st, agg.tobytes()

    def verify_fs_aggregate(self, B, contexts, outputs, transcript):
        """(accept, fail_code, fail_layer) of an aggregate proof for the claimed outputs [instances * S_out] (statement-major,
        as the output layer) and this context's inputs"""
        ctx = self._aggregate_contexts(B, contexts)
        for name, a, n in (("outputs", outputs, self._n_outputs()), ("transcript", transcript, self.circuit.transcript_len)):
            if not isinstance(a, np.ndarray) or a.dtype != F_DTYPE or a.shape != (n,):
                raise ValueError(f"{name} must be a [{n}] field-element array, got "
                                 f"{getattr(a, 'dtype', type(a))} {getattr(a, 'shape', None)}")
        out, tr = np.ascontiguousarray(outputs), np.ascontiguousarray(transcript)
        return _verdict(lambda *v: lib().vp_verify_fs_aggregate(self.h, B, _ptr(ctx), _ptr(out), out.size, _ptr(tr), tr.size, *v))

    def fs_round_stamps(self):
        """block 0's %globaltimer stamps (ns) per round of the last device Fiat-Shamir proof: [rounds, 4] = round start, own
        fold work done, polynomial reduced, challenge drawn"""
        n = C.c_size_t()
        _ck(lib().vp_fs_round_stamps(self.h, None, 0, C.byref(n)))
        out = np.zeros(4 * max(n.value, 1), np.uint64)
        _ck(lib().vp_fs_round_stamps(self.h, _ptr(out), len(out), C.byref(n)))
        return out[:4 * n.value].reshape(n.value, 4)

    def input_range(self):
        """instances [first, end) whose witness this rank uploads (everything on an unsharded context)"""
        a, b = C.c_uint64(), C.c_uint64()
        _ck(lib().vp_input_range(self.h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def prove_local(self, local_inputs, challenges, transcript=None):
        """vp_prove(host_io=1) for a caller that only holds the inputs of input_range()"""
        local_inputs = np.ascontiguousarray(local_inputs, dtype=np.uint64)
        challenges = np.ascontiguousarray(challenges, dtype=F_DTYPE)
        if transcript is None:
            transcript = np.zeros(self.circuit.transcript_len, F_DTYPE)
        _ck(lib().vp_prove_local(self.h, _ptr(local_inputs), len(local_inputs), _ptr(challenges), len(challenges),
                                 _ptr(transcript), len(transcript)))
        return transcript

    def transcript(self):
        out = np.zeros(self.circuit.transcript_len, F_DTYPE)
        _ck(lib().vp_get_transcript(self.h, _ptr(out), len(out)))
        return out

    @property
    def last_prove_ms(self):
        return float(lib().vp_last_prove_ms(self.h))

    @property
    def last_prove_launches(self):
        return int(lib().vp_last_prove_launches(self.h))

    @property
    def stream(self):
        return lib().vp_stream(self.h)

    def set_stream(self, cuda_stream):
        _ck(lib().vp_set_stream(self.h, C.c_void_p(cuda_stream)))

    KERNEL_CLASSES = ("round_fold", "round_first", "init_phase1", "init_phase2", "init_liu", "evaluate", "other")

    def set_profiling(self, on):
        _ck(lib().vp_set_profiling(self.h, 1 if on else 0))

    def verify(self, transcript):
        """(accept, fail_code, fail_layer) of the device-side verifier on a transcript (inputs + challenges resident)"""
        tr = np.ascontiguousarray(transcript, dtype=F_DTYPE)
        return _verdict(lambda *v: lib().vp_verify(self.h, _ptr(tr), len(tr), *v))

    def set_lanes(self, lanes):
        return int(lib().vp_set_lanes(self.h, int(lanes)))

    def profile(self):
        n = len(self.KERNEL_CLASSES)
        ms, by, la = np.zeros(n), np.zeros(n), np.zeros(n, np.uint64)
        _ck(lib().vp_get_profile(self.h, _ptr(ms), _ptr(by), _ptr(la), n))
        return {k: dict(ms=float(ms[i]), bytes=float(by[i]), launches=int(la[i])) for i, k in enumerate(self.KERNEL_CLASSES)}


def prove_interactive(prover, circuit, seed=3396):
    """Drive the prover method-by-method in the order of verifier::verify (src/verifier.cpp:134-337),
    feeding it the verifier's challenge stream; returns the transcript in vp_transcript_len layout."""
    ch = circuit.draw_challenges(seed)
    n = circuit.n_layers
    K = circuit.instances
    max_bl = max(circuit.bit_length(i) for i in range(n))
    tr = []
    zero = fe(0, 0)
    ci = 0
    out_bl = circuit.bit_length(n - 1)
    r_out = ch[ci:ci + out_bl]
    ci += out_bl
    prover.evaluate()
    tr.append(prover.Vres(r_out))
    prover.sumcheckInitAll(r_out)
    r_liu = None
    for i in range(n - 1, 0, -1):
        pb = circuit.bit_length(i - 1)
        m = circuit.max_dad_bit_length(i)
        prover.sumcheckInit()
        r_u = ch[ci:ci + max_bl]
        ci += max_bl
        assert_r = ch[ci]
        ci += 1
        prover.sumcheckInitPhase1(assert_r)
        prev = zero
        for j in range(pb):
            tr.extend(prover.sumcheckUpdatePhase1(prev))
            prev = r_u[j]
        tr.append(prover.sumcheckFinalize1(prev))
        if m != -1:
            r_v = ch[ci:ci + m]
            ci += m
            prover.sumcheckInitPhase2()
            prev = zero
            for j in range(m):
                tr.extend(prover.sumcheckUpdatePhase2(prev))
                prev = r_v[j]
            tr.extend(prover.sumcheckFinalize2(prev, i))
        sig = ch[ci:ci + n]
        ci += n
        r_liu = ch[ci:ci + max_bl]
        ci += max_bl
        prover.sumcheckInitLiu(sig)
        prev = zero
        for j in range(pb):
            tr.extend(prover.sumcheckLiuUpdate(prev))
            prev = r_liu[j]
        tr.append(prover.sumcheckLiuFinalize(prev))
    tr.append(prover.input_mle(r_liu[:circuit.bit_length(0)]))
    assert ci == len(ch)
    out = np.zeros(len(tr), F_DTYPE)
    for k, x in enumerate(tr):
        out[k] = x
    return out


class Sumcheck:
    """Stand-alone multilinear sumcheck over three 2^log_n tables (config C2)."""

    def __init__(self, log_n, device=0):
        self.log_n = log_n
        h = C.c_void_p()
        _ck(lib().vp_sumcheck_create(log_n, device, C.byref(h)))
        self.h = h

    def load(self, V, add, mult):
        a = [np.ascontiguousarray(x, dtype=F_DTYPE) for x in (V, add, mult)]
        assert all(len(x) == 1 << self.log_n for x in a)
        _ck(lib().vp_sumcheck_load(self.h, *[_ptr(x) for x in a]))

    def fill_random(self, seed):
        _ck(lib().vp_sumcheck_fill_random(self.h, seed))

    def export(self):
        n = 1 << self.log_n
        a = [np.zeros(n, F_DTYPE) for _ in range(3)]
        _ck(lib().vp_sumcheck_export(self.h, *[_ptr(x) for x in a]))
        return a

    def run(self, r, fused=False):
        """fused=False: one round per launch (what the interactive prover does); fused=True: one cooperative
        launch, two rounds per pass (what vp_prove does)."""
        r = np.ascontiguousarray(r, dtype=F_DTYPE)
        assert len(r) == self.log_n
        out = np.zeros(3 * self.log_n + 3, F_DTYPE)
        ms = C.c_float()
        fn = lib().vp_sumcheck_run_fused if fused else lib().vp_sumcheck_run
        _ck(fn(self.h, _ptr(r), _ptr(out), C.byref(ms)))
        return out, ms.value

    def pass_stamps(self):
        out = np.zeros(256 + 2048, np.uint64)
        _ck(lib().vp_sumcheck_pass_stamps(self.h, _ptr(out), len(out)))
        n = (self.log_n + 1) // 2
        self.block_stamps = out[256:].reshape(1024, 2)
        return out[:4 * n].reshape(n, 4)

    def round_ms(self):
        out = np.zeros(self.log_n, np.float32)
        _ck(lib().vp_sumcheck_round_ms(self.h, _ptr(out)))
        return out

    def close(self):
        if getattr(self, "h", None):
            lib().vp_sumcheck_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
