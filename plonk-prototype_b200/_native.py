"""ctypes binding of libpb200.so (the C ABI in include/pb200.h).

There is no fallback of any kind: if the shared library is missing, or no sm_100 GPU is present,
creating a Context raises.  Nothing in this package imports oracle/.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpb200.so")
_lib = None

EXPORTS = [
    "pb200_init", "pb200_destroy", "pb200_last_error", "pb200_stream", "pb200_sync",
    "pb200_malloc", "pb200_free", "pb200_h2d", "pb200_d2h",
    "pb200_domain_log_size", "pb200_ntt", "pb200_ntt_dev", "pb200_ntt_batch_dev", "pb200_ntt_columns_dev", "pb200_ntt_columns_scatter_dev",
    "pb200_ipc_export", "pb200_ipc_open", "pb200_ipc_close", "pb200_block_transpose_dev",
    "pb200_srs_upload", "pb200_srs_wrap_dev", "pb200_srs_precompute", "pb200_srs_lagrange", "pb200_srs_free", "pb200_srs_len",
    "pb200_msm_g1", "pb200_msm_g1_dev", "pb200_msm_g1_batch_dev", "pb200_pippenger_g1", "pb200_g1_sum", "pb200_msm_window_bits",
    "pb200_srs_generate", "pb200_srs_generate_range", "pb200_srs_dev_ptr", "pb200_kzg_witness_dev", "pb200_fr_horner_step_dev",
    "pb200_srs_from_compressed", "pb200_srs_to_compressed",
    "pb200_preprocess", "pb200_preprocess_sharded", "pb200_prover_key_free", "pb200_prover_key_size", "pb200_prover_key_bytes", "pb200_prove", "pb200_prove_dev",
    "pb200_transcript_selftest", "pb200_synthetic_circuit", "pb200_verify", "pb200_verify_batch", "pb200_opening_key_from_tau",
    "pb200_pairing_selftest",
    "pb200_synthetic_bases_dev", "pb200_profile_enable", "pb200_profile_ms", "pb200_profile_reset", "pb200_profile_sum_ms",
    "pb200_launch_count",
    "pb200_imad_peak",
    "pb200_comm_unique_id", "pb200_comm_init", "pb200_comm_destroy", "pb200_comm_info", "pb200_allgather_dev", "pb200_alltoall_dev",
    "pb200_msm_g1_sharded_dev", "pb200_ntt_sharded_dev", "pb200_preprocess_comm",
]


class Pb200Error(RuntimeError):
    pass


# per-point status of pb200_srs_from_compressed (PB200_G1_* in include/pb200.h)
G1_OK, G1_BAD_FLAGS, G1_X_RANGE, G1_NOT_ON_CURVE, G1_NOT_IN_SUBGROUP, G1_IDENTITY = range(6)


ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)
DEV_COLLECTIVE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)


class Shard(ctypes.Structure):
    """`pb200_shard` (include/pb200.h)."""
    _fields_ = [("rank", ctypes.c_uint32), ("world", ctypes.c_uint32), ("allgather", ALLGATHER_FN), ("user", ctypes.c_void_p),
                ("alltoall_dev", DEV_COLLECTIVE_FN), ("allgather_dev", DEV_COLLECTIVE_FN), ("flags", ctypes.c_uint32)]


class Circuit(ctypes.Structure):
    """`pb200_circuit` (include/pb200.h)."""
    _fields_ = [("n_gates", ctypes.c_size_t), ("n_vars", ctypes.c_size_t), ("selectors", ctypes.c_void_p * 11),
                ("wires", ctypes.c_void_p * 4)]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Pb200Error("libpb200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                             "there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        vp, u64p = ctypes.c_void_p, ctypes.c_void_p
        L.pb200_init.argtypes = [ctypes.POINTER(vp), ctypes.c_int]
        L.pb200_destroy.argtypes = [vp]
        L.pb200_destroy.restype = None
        L.pb200_last_error.argtypes = [vp]
        L.pb200_last_error.restype = ctypes.c_char_p
        L.pb200_stream.argtypes = [vp]
        L.pb200_stream.restype = vp
        L.pb200_sync.argtypes = [vp]
        L.pb200_malloc.argtypes = [vp, ctypes.POINTER(vp), ctypes.c_size_t]
        L.pb200_free.argtypes = [vp, vp]
        L.pb200_h2d.argtypes = [vp, vp, vp, ctypes.c_size_t]
        L.pb200_d2h.argtypes = [vp, vp, vp, ctypes.c_size_t]
        L.pb200_domain_log_size.argtypes = [ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint32)]
        L.pb200_ntt.argtypes = [vp, u64p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]
        L.pb200_ntt_dev.argtypes = [vp, u64p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]
        L.pb200_ntt_batch_dev.argtypes = [vp, u64p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]
        L.pb200_ntt_columns_dev.argtypes = [vp, u64p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int]
        L.pb200_ntt_columns_scatter_dev.argtypes = [vp, u64p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                                                    ctypes.c_uint32, ctypes.POINTER(vp)]
        L.pb200_ipc_export.argtypes = [vp, vp, ctypes.c_char_p]
        L.pb200_ipc_open.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(vp)]
        L.pb200_ipc_close.argtypes = [vp, vp]
        L.pb200_block_transpose_dev.argtypes = [vp, u64p, u64p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]
        L.pb200_srs_upload.argtypes = [vp, u64p, ctypes.c_size_t, ctypes.POINTER(vp)]
        L.pb200_srs_wrap_dev.argtypes = [vp, u64p, ctypes.c_size_t, ctypes.POINTER(vp)]
        L.pb200_srs_precompute.argtypes = [vp, vp]
        L.pb200_srs_lagrange.argtypes = [vp, vp, ctypes.c_uint32, ctypes.POINTER(vp)]
        L.pb200_srs_free.argtypes = [vp, vp]
        L.pb200_srs_free.restype = None
        L.pb200_srs_len.argtypes = [vp]
        L.pb200_srs_len.restype = ctypes.c_size_t
        L.pb200_msm_g1.argtypes = [vp, vp, ctypes.c_size_t, u64p, ctypes.c_size_t, u64p]
        L.pb200_msm_g1_dev.argtypes = [vp, vp, ctypes.c_size_t, u64p, ctypes.c_size_t, u64p]
        L.pb200_msm_g1_batch_dev.argtypes = [vp, vp, ctypes.c_size_t, u64p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_size_t, u64p]
        L.pb200_g1_sum.argtypes = [vp, u64p, ctypes.c_size_t, u64p]
        L.pb200_pippenger_g1.argtypes = [vp, u64p, u64p, ctypes.c_size_t, u64p]
        L.pb200_msm_window_bits.argtypes = [ctypes.c_size_t]
        L.pb200_msm_window_bits.restype = ctypes.c_uint32
        L.pb200_srs_generate.argtypes = [vp, u64p, ctypes.c_size_t, ctypes.POINTER(vp)]
        L.pb200_srs_dev_ptr.argtypes = [vp]
        L.pb200_srs_dev_ptr.restype = vp
        L.pb200_kzg_witness_dev.argtypes = [vp, u64p, ctypes.c_size_t, u64p, u64p, u64p]
        L.pb200_fr_horner_step_dev.argtypes = [vp, u64p, ctypes.c_size_t, u64p, ctypes.c_size_t, u64p]
        L.pb200_preprocess.argtypes = [vp, vp, ctypes.POINTER(Circuit), ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(vp), vp]
        L.pb200_preprocess_sharded.argtypes = [vp, vp, ctypes.POINTER(Circuit), ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(Shard),
                                               ctypes.POINTER(vp), vp]
        L.pb200_srs_generate_range.argtypes = [vp, u64p, ctypes.c_size_t, ctypes.c_size_t, ctypes.POINTER(vp)]
        L.pb200_srs_from_compressed.argtypes = [vp, vp, ctypes.c_size_t, vp, ctypes.POINTER(vp)]
        L.pb200_srs_to_compressed.argtypes = [vp, vp, ctypes.c_size_t, ctypes.c_size_t, vp]
        L.pb200_prover_key_free.argtypes = [vp, vp]
        L.pb200_prover_key_free.restype = None
        L.pb200_prover_key_size.argtypes = [vp]
        L.pb200_prover_key_size.restype = ctypes.c_size_t
        L.pb200_prover_key_bytes.argtypes = [vp]
        L.pb200_prover_key_bytes.restype = ctypes.c_size_t
        L.pb200_prove.argtypes = [vp, vp, vp, u64p, vp, u64p, ctypes.c_size_t, vp]
        L.pb200_prove_dev.argtypes = [vp, vp, vp, u64p, vp, u64p, ctypes.c_size_t, vp]
        L.pb200_transcript_selftest.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p,
                                                ctypes.c_char_p, ctypes.c_size_t]
        L.pb200_verify.argtypes = [vp, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, vp, vp, u64p, ctypes.c_size_t, u64p,
                                   ctypes.POINTER(ctypes.c_int)]
        L.pb200_verify_batch.argtypes = [vp, vp, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, vp, ctypes.c_size_t, vp, u64p,
                                         ctypes.c_size_t, u64p, vp, vp, ctypes.POINTER(ctypes.c_int)]
        L.pb200_opening_key_from_tau.argtypes = [u64p, u64p]
        L.pb200_pairing_selftest.argtypes = [u64p, u64p, ctypes.POINTER(ctypes.c_int)]
        L.pb200_synthetic_circuit.argtypes = [ctypes.c_size_t, ctypes.c_uint64, ctypes.c_uint32, ctypes.POINTER(vp), ctypes.POINTER(vp), u64p,
                                              ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), vp, u64p]
        L.pb200_synthetic_bases_dev.argtypes = [vp, u64p, ctypes.c_size_t, ctypes.c_uint64, ctypes.c_uint64]
        L.pb200_profile_enable.argtypes = [vp, ctypes.c_int]
        L.pb200_profile_ms.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_float)]
        L.pb200_profile_reset.argtypes = [vp]
        L.pb200_profile_sum_ms.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint32)]
        L.pb200_launch_count.argtypes = [vp]
        L.pb200_launch_count.restype = ctypes.c_uint64
        L.pb200_imad_peak.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        L.pb200_comm_unique_id.argtypes = [ctypes.c_char_p]
        L.pb200_comm_init.argtypes = [vp, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint32]
        L.pb200_comm_destroy.argtypes = [vp]
        L.pb200_comm_info.argtypes = [vp, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
        L.pb200_allgather_dev.argtypes = [vp, vp, vp, ctypes.c_size_t]
        L.pb200_alltoall_dev.argtypes = [vp, vp, vp, ctypes.c_size_t]
        L.pb200_msm_g1_sharded_dev.argtypes = [vp, vp, ctypes.c_size_t, u64p, ctypes.c_size_t, u64p]
        L.pb200_ntt_sharded_dev.argtypes = [vp, u64p, u64p, ctypes.c_uint32, ctypes.c_int]
        L.pb200_preprocess_comm.argtypes = [vp, vp, ctypes.POINTER(Circuit), ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(vp), vp]
        _lib = L
    return _lib


def _ptr(a):
    """Address of a numpy array (host) or an int device pointer."""
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return ctypes.c_void_p(a.ctypes.data)
    return ctypes.c_void_p(int(a))


def opening_key_from_tau(tau_mont):
    """β·H ∈ G2 (24 u64) for a trapdoor-generated SRS — host only, no GPU."""
    tau = np.ascontiguousarray(tau_mont, dtype=np.uint64).reshape(4)
    out = np.zeros(24, np.uint64)
    if lib().pb200_opening_key_from_tau(_ptr(tau), _ptr(out)) != 0:
        raise Pb200Error("pb200_opening_key_from_tau failed")
    return out


def verify(vk_bytes, n, label, proof, pi_gate, pi_mont, beta_h):
    """`Proof::verify` on the host CPU (csrc/verify.cu).  Returns True / False."""
    vk = np.frombuffer(bytes(vk_bytes), dtype=np.uint8).copy()
    pr = np.frombuffer(bytes(proof), dtype=np.uint8).copy()
    assert vk.size == 720 and pr.size == 1040
    pos = np.ascontiguousarray(pi_gate, dtype=np.uint32)
    piv = np.ascontiguousarray(pi_mont, dtype=np.uint64).reshape(-1, 4)
    bh = np.ascontiguousarray(beta_h, dtype=np.uint64).reshape(24)
    ok = ctypes.c_int(0)
    rc = lib().pb200_verify(_ptr(vk), n, bytes(label), len(label), _ptr(pr), _ptr(pos) if pos.size else None,
                            _ptr(piv) if pos.size else None, pos.shape[0], _ptr(bh), ctypes.byref(ok))
    if rc != 0:
        raise Pb200Error("pb200_verify: bad argument (%d)" % rc)
    return bool(ok.value)


def verify_batch(ctx, vk_bytes, n, label, proofs, pi_gate, pi_mont, beta_h, seed=None):
    """Many proofs of one circuit in one batched check on the GPU (pb200_verify_batch).  proofs: a sequence of 1040-byte
    proofs (or their concatenation); pi_gate: the n_pi gates every proof's public inputs sit at; pi_mont: (K, n_pi, 4)
    uint64 Montgomery values; seed: 32 bytes, drawn from os.urandom when None.  Returns a numpy bool array, entry k being
    what `verify` returns for proof k."""
    h = ctx._h if isinstance(ctx, Context) else ctx
    vk = np.frombuffer(bytes(vk_bytes), dtype=np.uint8).copy()
    pr = np.frombuffer(b"".join(bytes(p) for p in proofs) if not isinstance(proofs, (bytes, bytearray)) else bytes(proofs),
                       dtype=np.uint8).copy()
    assert vk.size == 720 and pr.size % 1040 == 0
    K = pr.size // 1040
    pos = np.ascontiguousarray(pi_gate, dtype=np.uint32).reshape(-1)
    piv = np.ascontiguousarray(pi_mont, dtype=np.uint64).reshape(K, pos.size, 4) if pos.size else np.zeros((K, 0, 4), np.uint64)
    bh = np.ascontiguousarray(beta_h, dtype=np.uint64).reshape(24)
    sd = np.frombuffer(os.urandom(32) if seed is None else bytes(seed), dtype=np.uint8).copy()
    assert sd.size == 32
    acc = np.zeros(max(K, 1), np.uint8)
    all_ok = ctypes.c_int(0)
    rc = lib().pb200_verify_batch(h, _ptr(vk), n, bytes(label), len(label), _ptr(pr) if K else None, K, _ptr(pos) if pos.size else None,
                                  _ptr(piv) if pos.size else None, pos.size, _ptr(bh), _ptr(sd), _ptr(acc), ctypes.byref(all_ok))
    if rc != 0:
        raise Pb200Error("pb200_verify_batch failed (%d): %s" % (rc, lib().pb200_last_error(h).decode()))
    return acc[:K].astype(bool)


class Context:
    """One CUDA device + stream (pb200_ctx)."""

    def __init__(self, device=0):
        self._h = ctypes.c_void_p()
        rc = lib().pb200_init(ctypes.byref(self._h), int(device))
        if rc != 0:
            msg = lib().pb200_last_error(self._h).decode() if self._h else "no usable sm_100 GPU"
            if self._h:
                lib().pb200_destroy(self._h)
                self._h = ctypes.c_void_p()
            raise Pb200Error("pb200_init failed (%d): %s — there is no CPU fallback" % (rc, msg))
        self.device = device

    def close(self):
        if self._h:
            lib().pb200_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise Pb200Error("pb200 error %d: %s" % (rc, lib().pb200_last_error(self._h).decode()))

    # -- plumbing
    @property
    def stream(self):
        return lib().pb200_stream(self._h)

    def sync(self):
        self._check(lib().pb200_sync(self._h))

    def malloc(self, nbytes):
        p = ctypes.c_void_p()
        self._check(lib().pb200_malloc(self._h, ctypes.byref(p), nbytes))
        return p.value

    def free(self, dev):
        self._check(lib().pb200_free(self._h, ctypes.c_void_p(dev)))

    def h2d(self, dev, host):
        self._check(lib().pb200_h2d(self._h, ctypes.c_void_p(dev), _ptr(host), host.nbytes))

    def d2h(self, host, dev):
        self._check(lib().pb200_d2h(self._h, _ptr(host), ctypes.c_void_p(dev), host.nbytes))

    # -- NTT
    def ntt(self, data_host, log_n, inverse=False, coset=False):
        assert data_host.dtype == np.uint64 and data_host.size == 4 << log_n
        self._check(lib().pb200_ntt(self._h, _ptr(data_host), log_n, int(inverse), int(coset)))

    def ntt_dev(self, dev, log_n, inverse=False, coset=False):
        self._check(lib().pb200_ntt_dev(self._h, ctypes.c_void_p(dev), log_n, int(inverse), int(coset)))

    def ntt_batch_dev(self, dev, log_n, batch, inverse=False, coset=False):
        self._check(lib().pb200_ntt_batch_dev(self._h, ctypes.c_void_p(dev), log_n, batch, int(inverse), int(coset)))

    def ntt_columns_dev(self, dev, log_n, log_n1, log_cols, col_offset, inverse=False):
        self._check(lib().pb200_ntt_columns_dev(self._h, ctypes.c_void_p(dev), log_n, log_n1, log_cols, col_offset, int(inverse)))

    def ntt_columns_scatter_dev(self, dev, log_n, log_n1, log_cols, col_offset, peer_row_bufs):
        arr = (ctypes.c_void_p * len(peer_row_bufs))(*[int(p) for p in peer_row_bufs])
        self._check(lib().pb200_ntt_columns_scatter_dev(self._h, ctypes.c_void_p(dev), log_n, log_n1, log_cols, col_offset,
                                                        len(peer_row_bufs), arr))

    def ipc_export(self, dev):
        buf = ctypes.create_string_buffer(64)
        self._check(lib().pb200_ipc_export(self._h, ctypes.c_void_p(dev), buf))
        return buf.raw

    def ipc_open(self, handle):
        p = ctypes.c_void_p()
        self._check(lib().pb200_ipc_open(self._h, handle, ctypes.byref(p)))
        return p.value

    def ipc_close(self, dev):
        self._check(lib().pb200_ipc_close(self._h, ctypes.c_void_p(dev)))

    def block_transpose_dev(self, dst, src, blocks, rows, cols):
        self._check(lib().pb200_block_transpose_dev(self._h, ctypes.c_void_p(dst), ctypes.c_void_p(src), blocks, rows, cols))

    # -- MSM
    def srs_upload(self, xy_host):
        assert xy_host.dtype == np.uint64 and xy_host.size % 12 == 0
        h = ctypes.c_void_p()
        self._check(lib().pb200_srs_upload(self._h, _ptr(xy_host), xy_host.size // 12, ctypes.byref(h)))
        return h

    def srs_wrap_dev(self, dev, n):
        h = ctypes.c_void_p()
        self._check(lib().pb200_srs_wrap_dev(self._h, ctypes.c_void_p(dev), n, ctypes.byref(h)))
        return h

    def srs_precompute(self, srs):
        self._check(lib().pb200_srs_precompute(self._h, srs))

    def srs_lagrange(self, srs, log_n):
        """New commit key [L_i(τ)]G, i < 2^log_n, in the Lagrange basis of the domain of size 2^log_n (pb200_srs_lagrange)."""
        h = ctypes.c_void_p()
        self._check(lib().pb200_srs_lagrange(self._h, srs, log_n, ctypes.byref(h)))
        return h

    def srs_free(self, srs):
        lib().pb200_srs_free(self._h, srs)

    def msm(self, srs, scalars_host, offset=0):
        n = scalars_host.size // 4
        out = np.zeros(18, np.uint64)
        self._check(lib().pb200_msm_g1(self._h, srs, offset, _ptr(scalars_host), n, _ptr(out)))
        return out

    def msm_dev(self, srs, scalars_dev, n, offset=0):
        out = np.zeros(18, np.uint64)
        self._check(lib().pb200_msm_g1_dev(self._h, srs, offset, ctypes.c_void_p(scalars_dev), n, _ptr(out)))
        return out

    def msm_batch_dev(self, srs, scalars_dev, n, batch, stride, offset=0):
        out = np.zeros((batch, 18), np.uint64)
        self._check(lib().pb200_msm_g1_batch_dev(self._h, srs, offset, ctypes.c_void_p(scalars_dev), n, batch, stride, _ptr(out)))
        return out

    def pippenger(self, points_xyz_host, scalars_host):
        """`multiscalar_mul::pippenger`: bases in projective coordinates (n, 18) u64, scalars (n, 4) u64, both Montgomery."""
        pts = np.ascontiguousarray(points_xyz_host, dtype=np.uint64).reshape(-1, 18)
        sc = np.ascontiguousarray(scalars_host, dtype=np.uint64).reshape(-1, 4)
        assert pts.shape[0] == sc.shape[0]
        out = np.zeros(18, np.uint64)
        self._check(lib().pb200_pippenger_g1(self._h, _ptr(pts) if pts.size else None, _ptr(sc) if sc.size else None, pts.shape[0], _ptr(out)))
        return out

    def g1_sum(self, points_xyz_host):
        pts = np.ascontiguousarray(points_xyz_host, dtype=np.uint64).reshape(-1, 18)
        out = np.zeros(18, np.uint64)
        self._check(lib().pb200_g1_sum(self._h, _ptr(pts), pts.shape[0], _ptr(out)))
        return out

    # -- KZG layer
    def srs_generate(self, tau_mont, n):
        tau = np.ascontiguousarray(tau_mont, dtype=np.uint64).reshape(4)
        h = ctypes.c_void_p()
        self._check(lib().pb200_srs_generate(self._h, _ptr(tau), n, ctypes.byref(h)))
        return h

    def srs_generate_range(self, tau_mont, first, n):
        tau = np.ascontiguousarray(tau_mont, dtype=np.uint64).reshape(4)
        h = ctypes.c_void_p()
        self._check(lib().pb200_srs_generate_range(self._h, _ptr(tau), first, n, ctypes.byref(h)))
        return h

    def srs_dev_ptr(self, srs):
        return lib().pb200_srs_dev_ptr(srs)

    def srs_from_compressed(self, data, status_out=None):
        """`CommitKey::from_slice` on the device: 48-byte compressed points (bytes-like, length a positive multiple of 48) →
        an SRS handle.  Every point is checked (flags, x < p, on the curve, prime-order subgroup); an invalid one raises
        ValueError with the library's message, which names the first invalid index and the reason.  status_out (optional
        uint8 array of one byte per point) receives G1_* per point, also when the call fails."""
        buf = np.frombuffer(data, dtype=np.uint8)
        if buf.size == 0 or buf.size % 48:
            raise ValueError("compressed commit key: %d bytes is not a positive multiple of 48" % buf.size)
        n = buf.size // 48
        if status_out is not None:
            assert status_out.dtype == np.uint8 and status_out.size == n and status_out.flags["C_CONTIGUOUS"]
        h = ctypes.c_void_p()
        rc = lib().pb200_srs_from_compressed(self._h, _ptr(buf), n, _ptr(status_out) if status_out is not None else None,
                                             ctypes.byref(h))
        if rc == 1:   # PB200_ERR_ARG: an invalid point (or argument) — a property of the input, not of the device
            raise ValueError(lib().pb200_last_error(self._h).decode())
        self._check(rc)
        return h

    def srs_to_compressed(self, srs, offset=0, n=None):
        """`CommitKey::to_var_bytes` of points [offset, offset + n) (default: to the end): 48·n bytes."""
        if n is None:
            n = lib().pb200_srs_len(srs) - offset
        out = np.empty(48 * n, np.uint8)
        self._check(lib().pb200_srs_to_compressed(self._h, srs, offset, n, _ptr(out)))
        return out.tobytes()

    def kzg_witness_dev(self, poly_dev, n, z_mont, quotient_dev):
        z = np.ascontiguousarray(z_mont, dtype=np.uint64).reshape(4)
        ev = np.zeros(4, np.uint64)
        self._check(lib().pb200_kzg_witness_dev(self._h, ctypes.c_void_p(poly_dev), n, _ptr(z), ctypes.c_void_p(quotient_dev), _ptr(ev)))
        return ev

    def fr_horner_step_dev(self, acc_dev, n_acc, poly_dev, n_poly, c_mont):
        c = np.ascontiguousarray(c_mont, dtype=np.uint64).reshape(4)
        self._check(lib().pb200_fr_horner_step_dev(self._h, ctypes.c_void_p(acc_dev), n_acc, ctypes.c_void_p(poly_dev), n_poly, _ptr(c)))

    # -- PLONK prover rounds
    def preprocess(self, srs, selectors, wires, n_vars, label, shard=None):
        """selectors: 11 (n_gates, 4) uint64 arrays or None; wires: 4 uint32 arrays.  Returns (key handle, 15×48 vk bytes).
        shard = (rank, world, allgather[, alltoall_dev, allgather_dev]) makes the key point-range-sharded: `srs` is this
        rank's slice and allgather(send: bytes) -> bytes of world × len(send), rank-major, is the host's collective; the
        two optional device collectives (send_ptr, recv_ptr, nbytes) -> None additionally shard round 3."""
        keep = []
        c = Circuit()
        c.n_gates = len(wires[0])
        c.n_vars = n_vars
        for k in range(11):
            if selectors[k] is None:
                c.selectors[k] = None
            else:
                a = np.ascontiguousarray(selectors[k], dtype=np.uint64).reshape(-1, 4)
                assert a.shape[0] == c.n_gates
                keep.append(a)
                c.selectors[k] = a.ctypes.data
        for k in range(4):
            a = np.ascontiguousarray(wires[k], dtype=np.uint32)
            assert a.shape[0] == c.n_gates
            keep.append(a)
            c.wires[k] = a.ctypes.data
        h = ctypes.c_void_p()
        vk = np.zeros(15 * 48, np.uint8)
        if shard is None:
            self._check(lib().pb200_preprocess(self._h, srs, ctypes.byref(c), bytes(label), len(label), ctypes.byref(h), _ptr(vk)))
            return h, vk.tobytes()
        rank, world, gather = shard[:3]
        dev_fns = list(shard[3:5]) if len(shard) >= 5 else [None, None]

        def dev_trampoline(fn):
            def call(_user, send, recv, nbytes):
                try:
                    fn(send, recv, nbytes)
                    return 0
                except Exception:
                    import traceback
                    traceback.print_exc()
                    return 2
            return DEV_COLLECTIVE_FN(call)

        def trampoline(_user, send, recv, nbytes):
            try:
                out = gather(ctypes.string_at(send, nbytes))
                if len(out) != world * nbytes:
                    return 1
                ctypes.memmove(recv, out, len(out))
                return 0
            except Exception:  # never let an exception cross the C ABI
                import traceback
                traceback.print_exc()
                return 2

        cb = ALLGATHER_FN(trampoline)
        dev_cbs = [dev_trampoline(f) if f is not None else DEV_COLLECTIVE_FN() for f in dev_fns]
        sh = Shard(rank, world, cb, None, dev_cbs[0], dev_cbs[1], 0)
        self._check(lib().pb200_preprocess_sharded(self._h, srs, ctypes.byref(c), bytes(label), len(label), ctypes.byref(sh),
                                                   ctypes.byref(h), _ptr(vk)))
        if not hasattr(self, "_keepalive"):
            self._keepalive = {}
        self._keepalive[h.value] = (cb, dev_cbs)  # the key holds the function pointers for every later pb200_prove
        return h, vk.tobytes()

    # -- multi-GPU communicator inside the library (NCCL; csrc/comm.cu)
    @staticmethod
    def comm_unique_id():
        buf = ctypes.create_string_buffer(128)
        rc = lib().pb200_comm_unique_id(buf)
        if rc != 0:
            raise Pb200Error("pb200_comm_unique_id failed (%d): NCCL (libnccl.so.2) is not loadable in this process" % rc)
        return buf.raw

    def comm_init(self, unique_id, rank, world):
        self._check(lib().pb200_comm_init(self._h, bytes(unique_id), rank, world))

    def comm_init_from_torch(self, dist):
        """Bind the library's own NCCL communicator using torch.distributed only to broadcast the 128-byte id."""
        rank, world = dist.get_rank(), dist.get_world_size()
        box = [self.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        self.comm_init(box[0], rank, world)

    def comm_destroy(self):
        self._check(lib().pb200_comm_destroy(self._h))

    def allgather_dev(self, send_dev, recv_dev, nbytes):
        self._check(lib().pb200_allgather_dev(self._h, ctypes.c_void_p(send_dev), ctypes.c_void_p(recv_dev), nbytes))

    def alltoall_dev(self, send_dev, recv_dev, bytes_per_peer):
        self._check(lib().pb200_alltoall_dev(self._h, ctypes.c_void_p(send_dev), ctypes.c_void_p(recv_dev), bytes_per_peer))

    def msm_sharded_dev(self, srs_slice, scalars_dev, n, offset=0):
        out = np.zeros(18, np.uint64)
        self._check(lib().pb200_msm_g1_sharded_dev(self._h, srs_slice, offset, ctypes.c_void_p(scalars_dev), n, _ptr(out)))
        return out

    def ntt_sharded_dev(self, data_dev, tmp_dev, log_n, inverse=False):
        self._check(lib().pb200_ntt_sharded_dev(self._h, ctypes.c_void_p(data_dev), ctypes.c_void_p(tmp_dev), log_n, int(inverse)))

    def preprocess_comm(self, srs_slice, selectors, wires, n_vars, label):
        """`pb200_preprocess_comm`: a sharded prover key whose collectives are the library's own NCCL calls."""
        keep = []
        c = Circuit()
        c.n_gates = len(wires[0])
        c.n_vars = n_vars
        for k in range(11):
            if selectors[k] is None:
                c.selectors[k] = None
            else:
                a = np.ascontiguousarray(selectors[k], dtype=np.uint64).reshape(-1, 4)
                keep.append(a)
                c.selectors[k] = a.ctypes.data
        for k in range(4):
            a = np.ascontiguousarray(wires[k], dtype=np.uint32)
            keep.append(a)
            c.wires[k] = a.ctypes.data
        h = ctypes.c_void_p()
        vk = np.zeros(15 * 48, np.uint8)
        self._check(lib().pb200_preprocess_comm(self._h, srs_slice, ctypes.byref(c), bytes(label), len(label), ctypes.byref(h), _ptr(vk)))
        return h, vk.tobytes()

    def prover_key_free(self, pk):
        lib().pb200_prover_key_free(self._h, pk)
        getattr(self, "_keepalive", {}).pop(getattr(pk, "value", None), None)

    def prover_key_size(self, pk):
        return lib().pb200_prover_key_size(pk)

    def prover_key_bytes(self, pk):
        return lib().pb200_prover_key_bytes(pk)

    def prove(self, srs, pk, values_mont, pi_gate, pi_mont):
        vals = np.ascontiguousarray(values_mont, dtype=np.uint64).reshape(-1, 4)
        pos = np.ascontiguousarray(pi_gate, dtype=np.uint32)
        piv = np.ascontiguousarray(pi_mont, dtype=np.uint64).reshape(-1, 4)
        assert pos.shape[0] == piv.shape[0]
        out = np.zeros(1040, np.uint8)
        self._check(lib().pb200_prove(self._h, srs, pk, _ptr(vals), _ptr(pos) if pos.size else None, _ptr(piv) if pos.size else None,
                                      pos.shape[0], _ptr(out)))
        return out.tobytes()

    def prove_dev(self, srs, pk, values_dev, pi_gate, pi_mont):
        """`pb200_prove_dev`: the witness (n_vars × 32 B) is already in device memory."""
        pos = np.ascontiguousarray(pi_gate, dtype=np.uint32)
        piv = np.ascontiguousarray(pi_mont, dtype=np.uint64).reshape(-1, 4)
        assert pos.shape[0] == piv.shape[0]
        out = np.zeros(1040, np.uint8)
        self._check(lib().pb200_prove_dev(self._h, srs, pk, ctypes.c_void_p(int(values_dev)), _ptr(pos) if pos.size else None,
                                          _ptr(piv) if pos.size else None, pos.shape[0], _ptr(out)))
        return out.tobytes()

    def synthetic_bases_dev(self, dev, n, a=0xB2000001, d=0x9E3779B1):
        self._check(lib().pb200_synthetic_bases_dev(self._h, ctypes.c_void_p(dev), n, a, d))

    # -- batched verification
    def verify_batch(self, vk_bytes, n, label, proofs, pi_gate, pi_mont, beta_h, seed=None):
        """`verify_batch` on this context."""
        return verify_batch(self, vk_bytes, n, label, proofs, pi_gate, pi_mont, beta_h, seed)

    # -- measurement
    def profile_enable(self, on=True):
        self._check(lib().pb200_profile_enable(self._h, int(on)))

    def profile_ms(self, name):
        v = ctypes.c_float()
        self._check(lib().pb200_profile_ms(self._h, name.encode(), ctypes.byref(v)))
        return v.value

    def profile_reset(self):
        self._check(lib().pb200_profile_reset(self._h))

    def profile_sum_ms(self, name):
        """(Σ ms, samples) of timer `name` since the last profile_reset."""
        v, c = ctypes.c_float(), ctypes.c_uint32()
        self._check(lib().pb200_profile_sum_ms(self._h, name.encode(), ctypes.byref(v), ctypes.byref(c)))
        return v.value, c.value

    def launch_count(self):
        return int(lib().pb200_launch_count(self._h))

    def imad_peak(self):
        ops, mhz = ctypes.c_double(), ctypes.c_double()
        self._check(lib().pb200_imad_peak(self._h, ctypes.byref(ops), ctypes.byref(mhz)))
        return ops.value, mhz.value
