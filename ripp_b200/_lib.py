"""ctypes binding of libripp_b200.so (include/ripp_b200.h).  No CPU fallback: importing works
without a GPU (so the symbol table can be checked), but creating a context without one raises."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RIPP_B200_LIB") or os.path.join(HERE, "libripp_b200.so")

RIPP_OK = 0
RIPP_ERR_LEN_MISMATCH = -1
RIPP_ERR_NOT_POW2 = -2
RIPP_ERR_CUDA = -3
RIPP_ERR_ARG = -4
RIPP_ERR_INNER_PRODUCT = -5
RIPP_ERR_NO_DEVICE = -6
RIPP_ERR_NCCL = -7

TEST_OPS = [
    "FQ_MUL", "FQ_ADD", "FQ_SUB", "FQ_INV", "FQ_HALF",
    "FR_MUL", "FR_ADD", "FR_SUB", "FR_INV",
    "FQ2_MUL", "FQ2_SQR", "FQ2_INV",
    "FQ12_MUL", "FQ12_SQR", "FQ12_INV", "FQ12_CYC_SQR", "FQ12_FROB1",
    "FINAL_EXP", "MILLER",
    "G1_ADD", "G1_DBL", "G2_ADD", "G2_DBL",
]
TEST_OP_ID = {n: i for i, n in enumerate(TEST_OPS)}


class RippError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("ripp_b200 status %d: %s" % (status, msg))
        self.status = status


GIPA_PAIRING, GIPA_MULTIEXP_PEDERSEN, GIPA_MULTIEXP_SSM = 0, 1, 2
GIPA_SCALAR_PEDERSEN_G2_G2, GIPA_SCALAR_PEDERSEN_G2_G1, GIPA_SCALAR_SSM, GIPA_SCALAR_SSM_G1 = 3, 4, 5, 6


class LengthMismatch(RippError):
    """InnerProductError::MessageLengthInvalid (inner_products/src/lib.rs:18-38)."""


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libripp_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                "ripp_b200 has no CPU fallback"
            )
        L = ctypes.CDLL(LIB_PATH)
        L.ripp_last_error_string.restype = ctypes.c_char_p
        L.ripp_ctx_stream.restype = ctypes.c_void_p
        L.ripp_ctx_launch_count.restype = ctypes.c_uint64
        _lib = L
    return _lib


def check(status):
    if status != RIPP_OK:
        msg = lib().ripp_last_error_string().decode()
        if status == RIPP_ERR_LEN_MISMATCH:
            raise LengthMismatch(status, msg)
        raise RippError(status, msg)


def _p(a):
    """void* of a host numpy array / device pointer int / None."""
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return ctypes.c_void_p(a.ctypes.data)
    if isinstance(a, DeviceBuffer):
        return ctypes.c_void_p(a.ptr)
    return ctypes.c_void_p(int(a))


class DeviceBuffer:
    """RAII handle on device memory owned by a Context (`ripp_vec_*` of SURVEY.md §8b)."""

    def __init__(self, ctx, nbytes):
        self.ctx, self.nbytes = ctx, nbytes
        p = ctypes.c_void_p()
        check(lib().ripp_dev_alloc(ctx.handle, ctypes.c_size_t(nbytes), ctypes.byref(p)))
        self.ptr = p.value

    def upload(self, host):
        host = np.ascontiguousarray(host)
        assert host.nbytes <= self.nbytes
        check(lib().ripp_dev_upload(self.ctx.handle, _p(self.ptr), _p(host), ctypes.c_size_t(host.nbytes)))
        return self

    def download(self, shape, dtype=np.uint32, offset=0):
        out = np.empty(shape, dtype=dtype)
        assert offset + out.nbytes <= self.nbytes
        check(lib().ripp_dev_download(self.ctx.handle, _p(out), _p(self.ptr + offset), ctypes.c_size_t(out.nbytes)))
        return out

    def free(self):
        # a buffer that outlives its context (interpreter shutdown, a traceback holding a reference) has nothing left to
        # free: ripp_ctx_destroy released the device and ripp_dev_free on a destroyed context would read freed memory
        if self.ptr and self.ctx.handle:
            check(lib().ripp_dev_free(self.ctx.handle, _p(self.ptr)))
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    def __init__(self, device=0):
        h = ctypes.c_void_p()
        check(lib().ripp_ctx_create(int(device), ctypes.byref(h)))
        self.handle = h
        self.device = device

    def close(self):
        if self.handle:
            lib().ripp_ctx_destroy(self.handle)
            self.handle = None

    def sync(self):
        check(lib().ripp_ctx_sync(self.handle))

    @property
    def stream(self):
        return lib().ripp_ctx_stream(self.handle)

    def set_stream(self, cuda_stream):
        check(lib().ripp_ctx_set_stream(self.handle, ctypes.c_void_p(int(cuda_stream) if cuda_stream else 0)))

    TIMING_CATS = ("miller", "final_exp", "msm", "fold", "scale", "other", "msm_sort", "msm_reduce")

    def set_timing(self, on):
        check(lib().ripp_ctx_set_timing(self.handle, int(on)))

    def timing(self):
        """-> {category: (ms, scopes)} since the last call (synchronises)."""
        ms = (ctypes.c_double * 8)()
        cnt = (ctypes.c_uint64 * 8)()
        check(lib().ripp_ctx_timing(self.handle, ms, cnt))
        return {c: (ms[i], int(cnt[i])) for i, c in enumerate(self.TIMING_CATS)}

    @property
    def launches(self):
        return int(lib().ripp_ctx_launch_count(self.handle))

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, host):
        host = np.ascontiguousarray(host)
        return DeviceBuffer(self, host.nbytes).upload(host)

    # ---- L1 -------------------------------------------------------------------------------
    def pairing_ip(self, g1_jac, g2_jac):
        """Host Jacobian arrays (n, 36) / (n, 72) uint32 -> GT (144,) uint32."""
        out = np.empty(144, dtype=np.uint32)
        check(lib().ripp_pairing_ip(self.handle, _p(g1_jac), ctypes.c_size_t(len(g1_jac)), _p(g2_jac),
                                    ctypes.c_size_t(len(g2_jac)), _p(out)))
        return out

    def pairing_ip_affine(self, g1, g2):
        out = np.empty(144, dtype=np.uint32)
        check(lib().ripp_pairing_ip_affine(self.handle, _p(g1), ctypes.c_size_t(len(g1)), _p(g2),
                                           ctypes.c_size_t(len(g2)), _p(out)))
        return out

    def pairing_ip_dev(self, g1_dev, g2_dev, n, out_dev):
        check(lib().ripp_pairing_ip_dev(self.handle, _p(g1_dev), _p(g2_dev), ctypes.c_size_t(n), _p(out_dev)))

    def miller_partial_dev(self, g1_dev, g2_dev, n, out_dev):
        check(lib().ripp_miller_partial_dev(self.handle, _p(g1_dev), _p(g2_dev), ctypes.c_size_t(n), _p(out_dev)))

    def gt_combine_dev(self, partials_dev, count, out_dev):
        check(lib().ripp_gt_combine_dev(self.handle, _p(partials_dev), ctypes.c_size_t(count), _p(out_dev)))

    def g1_scale_dev(self, pts_dev, fr_dev, n, out_dev):
        check(lib().ripp_g1_scale_dev(self.handle, _p(pts_dev), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    def g2_scale_dev(self, pts_dev, fr_dev, n, out_dev):
        check(lib().ripp_g2_scale_dev(self.handle, _p(pts_dev), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    def msm_g1(self, g1_jac, fr):
        out = np.empty(36, dtype=np.uint32)
        check(lib().ripp_msm_g1(self.handle, _p(g1_jac), ctypes.c_size_t(len(g1_jac)), _p(fr), ctypes.c_size_t(len(fr)), _p(out)))
        return out

    def msm_g2(self, g2_jac, fr):
        out = np.empty(72, dtype=np.uint32)
        check(lib().ripp_msm_g2(self.handle, _p(g2_jac), ctypes.c_size_t(len(g2_jac)), _p(fr), ctypes.c_size_t(len(fr)), _p(out)))
        return out

    def msm_g1_dev(self, bases_dev, fr_dev, n, out_dev):
        check(lib().ripp_msm_g1_dev(self.handle, _p(bases_dev), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    def msm_g2_dev(self, bases_dev, fr_dev, n, out_dev):
        check(lib().ripp_msm_g2_dev(self.handle, _p(bases_dev), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    def scalar_ip(self, a, b):
        out = np.empty(8, dtype=np.uint32)
        check(lib().ripp_scalar_ip(self.handle, _p(a), ctypes.c_size_t(len(a)), _p(b), ctypes.c_size_t(len(b)), _p(out)))
        return out

    def g1_fold_dev(self, hi, lo, c_host, n, out):
        check(lib().ripp_g1_fold_dev(self.handle, _p(hi), _p(lo), _p(c_host), ctypes.c_size_t(n), _p(out)))

    def g2_fold_dev(self, hi, lo, c_host, n, out):
        check(lib().ripp_g2_fold_dev(self.handle, _p(hi), _p(lo), _p(c_host), ctypes.c_size_t(n), _p(out)))

    def fr_fold_dev(self, hi, lo, c_host, n, out):
        check(lib().ripp_fr_fold_dev(self.handle, _p(hi), _p(lo), _p(c_host), ctypes.c_size_t(n), _p(out)))

    # ---- L3 / L4 ------------------------------------------------------------------------------
    def gipa_prove_dev(self, kind, a, b, v, w, n):
        """-> (GIPAProof bytes, r_transcript (k, 8) uint32, ck_base bytes)."""
        k = max(n.bit_length() - 1, 0)
        cap = 64 + k * 6 * 600 + 2 * 600
        proof = np.empty(cap, dtype=np.uint8)
        plen, cklen = ctypes.c_size_t(), ctypes.c_size_t()
        tr = np.zeros((k, 8), dtype=np.uint32)
        ck = np.empty(1024, dtype=np.uint8)
        check(lib().ripp_gipa_prove_dev(self.handle, int(kind), _p(a), _p(b), _p(v), _p(w), ctypes.c_size_t(n), _p(proof),
                                        ctypes.c_size_t(cap), ctypes.byref(plen), _p(tr), _p(ck), ctypes.c_size_t(1024),
                                        ctypes.byref(cklen)))
        return proof[: plen.value].tobytes(), tr, ck[: cklen.value].tobytes()

    def gipa_prove_checked_dev(self, kind, a, b, v, w, n, com):
        """GIPA::prove (gipa.rs:108-133): the statement `com` (bytes) is checked against the vectors first.  -> proof bytes"""
        k = max(n.bit_length() - 1, 0)
        cap = 64 + k * 6 * 600 + 2 * 600
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        cb = self._bytes(com)
        check(lib().ripp_gipa_prove_checked_dev(self.handle, int(kind), _p(a), _p(b), _p(v), _p(w), ctypes.c_size_t(n), _p(cb),
                                                ctypes.c_size_t(len(cb)), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    # ---- multi-GPU: NCCL inside the library (comm.cu, sharded.cuh) ---------------------------------
    @staticmethod
    def comm_unique_id():
        """128 bytes to hand to every rank (rank 0 calls this)."""
        buf = np.zeros(128, dtype=np.uint8)
        check(lib().ripp_comm_unique_id(_p(buf)))
        return buf.tobytes()

    def comm_init(self, unique_id, rank, world):
        check(lib().ripp_comm_init(self.handle, _p(self._bytes(unique_id)), int(rank), int(world)))

    def comm_info(self):
        r, w = ctypes.c_int(), ctypes.c_int()
        check(lib().ripp_comm_info(self.handle, ctypes.byref(r), ctypes.byref(w)))
        return r.value, w.value

    def comm_destroy(self):
        check(lib().ripp_comm_destroy(self.handle))

    def all_gather_dev(self, send_dev, nbytes, recv_dev):
        check(lib().ripp_all_gather_dev(self.handle, _p(send_dev), ctypes.c_size_t(nbytes), _p(recv_dev)))

    def pairing_ip_sharded_dev(self, g1_slice, g2_slice, n_local, out_dev):
        check(lib().ripp_pairing_ip_sharded_dev(self.handle, _p(g1_slice), _p(g2_slice), ctypes.c_size_t(n_local), _p(out_dev)))

    def msm_sharded_dev(self, group, bases_slice, fr_slice, n_local, out_dev):
        fn = lib().ripp_msm_g1_sharded_dev if group == 1 else lib().ripp_msm_g2_sharded_dev
        check(fn(self.handle, _p(bases_slice), _p(fr_slice), ctypes.c_size_t(n_local), _p(out_dev)))

    def gipa_prove_sharded_dev(self, kind, a, b, v, w, n_local, world, tail_len=0):
        """GIPA::prove_with_aux over cyclic shares.  -> (proof bytes, r_transcript (k, 8) uint32, ck_base bytes)."""
        k = max((n_local * world).bit_length() - 1, 0)
        cap = 64 + k * 6 * 600 + 2 * 600
        proof = np.empty(cap, dtype=np.uint8)
        plen, cklen = ctypes.c_size_t(), ctypes.c_size_t()
        tr = np.zeros((k, 8), dtype=np.uint32)
        ck = np.empty(1024, dtype=np.uint8)
        check(lib().ripp_gipa_prove_sharded_dev(self.handle, int(kind), _p(a), _p(b), _p(v), _p(w), ctypes.c_size_t(n_local),
                                                ctypes.c_size_t(tail_len), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen), _p(tr),
                                                _p(ck), ctypes.c_size_t(1024), ctypes.byref(cklen)))
        return proof[: plen.value].tobytes(), tr, ck[: cklen.value].tobytes()

    def tipp_aggregate_sharded_dev(self, srs_g1, srs_g2, a, b, c, n_total, tail_len=0):
        k = max(n_total.bit_length() - 1, 0)
        cap = 8192 + 2 * (64 + k * 6 * 600 + 8 * 600)
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp_tipp_aggregate_sharded_dev(self.handle, _p(srs_g1), _p(srs_g2), _p(a), _p(b), _p(c), ctypes.c_size_t(n_total),
                                                    ctypes.c_size_t(tail_len), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    # ---- setup --------------------------------------------------------------------------------
    def fixed_base_msm_dev(self, group, base, fr_dev, n, out_dev):
        """out[i] = s[i] * base (base: packed affine words or None = generator)."""
        fn = lib().ripp_fixed_base_msm_g1_dev if group == 1 else lib().ripp_fixed_base_msm_g2_dev
        check(fn(self.handle, _p(base), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    def structured_generators_dev(self, group, base, s, num, out_dev):
        """structured_generators_scalar_power (tipa/mod.rs:372-391): out[i] = s^i * base."""
        fn = lib().ripp_structured_generators_g1_dev if group == 1 else lib().ripp_structured_generators_g2_dev
        check(fn(self.handle, _p(base), _p(s), ctypes.c_size_t(num), _p(out_dev)))

    def tipa_setup_dev(self, alpha, beta, size):
        """TIPA::setup (tipa/mod.rs:150-164) for given trapdoors ((8,) uint32 Montgomery each).
        -> (srs_g1 DeviceBuffer, srs_g2 DeviceBuffer, g_beta words, h_alpha words)"""
        m = 2 * size - 1
        s1, s2 = self.alloc(m * 96), self.alloc(m * 192)
        gb, ha = np.zeros(24, dtype=np.uint32), np.zeros(48, dtype=np.uint32)
        check(lib().ripp_tipa_setup_dev(self.handle, _p(alpha), _p(beta), ctypes.c_size_t(size), _p(s1), _p(s2), _p(gb), _p(ha)))
        return s1, s2, gb, ha

    def gipa_prove_resume_dev(self, kind, a, b, v, w, n, prev_challenge):
        """As gipa_prove_dev, continuing a transcript whose last challenge is prev_challenge ((8,) uint32 Montgomery)."""
        k = max(n.bit_length() - 1, 0)
        cap = 64 + k * 6 * 600 + 2 * 600
        proof = np.empty(cap, dtype=np.uint8)
        plen, cklen = ctypes.c_size_t(), ctypes.c_size_t()
        tr = np.zeros((k, 8), dtype=np.uint32)
        ck = np.empty(1024, dtype=np.uint8)
        check(lib().ripp_gipa_prove_resume_dev(self.handle, int(kind), _p(a), _p(b), _p(v), _p(w), ctypes.c_size_t(n),
                                               _p(prev_challenge), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen), _p(tr),
                                               _p(ck), ctypes.c_size_t(1024), ctypes.byref(cklen)))
        return proof[: plen.value].tobytes(), tr, ck[: cklen.value].tobytes()

    def tipa_prove_dev(self, kind, srs_g1, srs_g2, a, b, v, w, n, r_shift=None):
        k = max(n.bit_length() - 1, 0)
        cap = 64 + k * 6 * 600 + 8 * 600
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp_tipa_prove_dev(self.handle, int(kind), _p(srs_g1), _p(srs_g2), _p(a), _p(b), _p(v), _p(w),
                                        ctypes.c_size_t(n), _p(r_shift), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    def kzg_open_dev(self, group, srs, n_srs, transcript, r_shift, z):
        k = len(transcript)
        out = np.zeros(24 if group == 1 else 48, dtype=np.uint32)
        fn = lib().ripp_kzg_open_g1_dev if group == 1 else lib().ripp_kzg_open_g2_dev
        check(fn(self.handle, _p(srs), ctypes.c_size_t(n_srs), _p(np.ascontiguousarray(transcript)), ctypes.c_size_t(k),
                 _p(r_shift), _p(z), _p(out)))
        return out

    def tipp_aggregate_dev(self, srs_g1, srs_g2, a, b, c, n):
        k = max(n.bit_length() - 1, 0)
        cap = 8 * 600 + 2 * (64 + k * 6 * 600 + 8 * 600)
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp_tipp_aggregate_dev(self.handle, _p(srs_g1), _p(srs_g2), _p(a), _p(b), _p(c), ctypes.c_size_t(n),
                                            _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    def tipp_aggregate(self, srs_g1, srs_g2, a_host, b_host, c_host):
        n = len(a_host)
        k = max(n.bit_length() - 1, 0)
        cap = 8 * 600 + 2 * (64 + k * 6 * 600 + 8 * 600)
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp_tipp_aggregate(self.handle, _p(srs_g1), _p(srs_g2), _p(a_host), _p(b_host), _p(c_host),
                                        ctypes.c_size_t(n), _p(proof), ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    # ---- deserialisation (csrc/deserialize.cu) ------------------------------------------------------
    def g1_deserialize_dev(self, bytes_dev, n, stride, compressed, out_dev, status_dev):
        """Decode and validate n ark-serialize G1 points at `stride` bytes (device) into affine words + status bytes."""
        check(lib().ripp_g1_deserialize_dev(self.handle, _p(bytes_dev), ctypes.c_size_t(n), ctypes.c_size_t(stride),
                                            int(bool(compressed)), _p(out_dev), _p(status_dev)))

    def g2_deserialize_dev(self, bytes_dev, n, stride, compressed, out_dev, status_dev):
        check(lib().ripp_g2_deserialize_dev(self.handle, _p(bytes_dev), ctypes.c_size_t(n), ctypes.c_size_t(stride),
                                            int(bool(compressed)), _p(out_dev), _p(status_dev)))

    def tipp_aggregate_serialized(self, srs_g1, srs_g2, data, n, compressed):
        """aggregate_proofs from n ark-groth16 Proof records (bytes, 192 B compressed / 384 B uncompressed each)."""
        k = max(n.bit_length() - 1, 0)
        cap = 8 * 600 + 2 * (64 + k * 6 * 600 + 8 * 600)
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        buf = self._bytes(data)
        check(lib().ripp_tipp_aggregate_serialized(self.handle, _p(srs_g1), _p(srs_g2), _p(buf), ctypes.c_size_t(len(data)),
                                                   ctypes.c_size_t(n), int(bool(compressed)), _p(proof), ctypes.c_size_t(cap),
                                                   ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    def sipp_product_with_coeffs(self, a, b, r):
        out = np.empty(144, dtype=np.uint32)
        check(lib().ripp_sipp_product_with_coeffs(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(len(a)), _p(out)))
        return out

    def sipp_prove(self, a, b, r, value):
        n = len(a)
        cap = max(n.bit_length() - 1, 0) * 1152 + 16
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp_sipp_prove(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(n), _p(value), _p(proof),
                                    ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    # ---- batch primitives of the sharded provers (parallel.py) ---------------------------------------
    def miller_partial_batch_dev(self, g1_ptrs, g2_ptrs, n, out_dev):
        k = len(g1_ptrs)
        a1 = (ctypes.c_void_p * k)(*[int(_p(x).value or 0) for x in g1_ptrs])
        a2 = (ctypes.c_void_p * k)(*[int(_p(x).value or 0) for x in g2_ptrs])
        check(lib().ripp_miller_partial_batch_dev(self.handle, k, a1, a2, ctypes.c_size_t(n), _p(out_dev)))

    def gt_combine_batch_dev(self, partials_dev, count, nseg, out_dev):
        check(lib().ripp_gt_combine_batch_dev(self.handle, _p(partials_dev), ctypes.c_size_t(count), int(nseg), _p(out_dev)))

    def seg_sum_dev(self, type_id, in_dev, count, nseg, out_dev):
        """type_id: 1 = G1 affine, 2 = G2 affine, 3 = Fr."""
        check(lib().ripp_seg_sum_dev(self.handle, int(type_id), _p(in_dev), ctypes.c_size_t(count), int(nseg), _p(out_dev)))

    def scalar_ip_dev(self, a_dev, b_dev, n, out_dev):
        check(lib().ripp_scalar_ip_dev(self.handle, _p(a_dev), _p(b_dev), ctypes.c_size_t(n), _p(out_dev)))

    def kzg_quotient(self, transcript, r_shift, z, n_srs):
        """-> (n_srs, 8) uint32 Montgomery Fr: coefficients of (f - f(z)) / (X - z), zero padded (tipa/mod.rs:313-332)."""
        transcript = np.ascontiguousarray(transcript, dtype=np.uint32)
        out = np.zeros((n_srs, 8), dtype=np.uint32)
        check(lib().ripp_kzg_quotient(_p(transcript), ctypes.c_size_t(len(transcript)), _p(r_shift), _p(z),
                                      ctypes.c_size_t(n_srs), _p(out)))
        return out

    # ---- verifiers --------------------------------------------------------------------------------
    def gt_multiexp_dev(self, gt_dev, fr_dev, n, out_dev):
        check(lib().ripp_gt_multiexp_dev(self.handle, _p(gt_dev), _p(fr_dev), ctypes.c_size_t(n), _p(out_dev)))

    @staticmethod
    def _bytes(b):
        return np.frombuffer(bytes(b), dtype=np.uint8).copy() if len(b) else np.zeros(1, dtype=np.uint8)

    def gipa_verify_dev(self, kind, v, w, n, com, proof, scalar_b=None):
        """-> bool.  com / proof: serialize_uncompressed bytes."""
        acc = ctypes.c_int(0)
        cb, pb = self._bytes(com), self._bytes(proof)
        check(lib().ripp_gipa_verify_dev(self.handle, int(kind), _p(v), _p(w), ctypes.c_size_t(n), _p(cb),
                                         ctypes.c_size_t(len(com)), _p(scalar_b), _p(pb), ctypes.c_size_t(len(proof)),
                                         ctypes.byref(acc)))
        return bool(acc.value)

    def tipa_verify(self, kind, vsrs, com, proof, shift=None):
        acc = ctypes.c_int(0)
        cb, pb = self._bytes(com), self._bytes(proof)
        check(lib().ripp_tipa_verify(self.handle, int(kind), _p(vsrs), _p(cb), ctypes.c_size_t(len(com)), _p(shift), _p(pb),
                                     ctypes.c_size_t(len(proof)), ctypes.byref(acc)))
        return bool(acc.value)

    def tipp_verify_aggregate(self, vsrs, vk, public_inputs, proof):
        """public_inputs: (n, m, 8) uint32 Montgomery Fr."""
        acc = ctypes.c_int(0)
        pb = self._bytes(proof)
        n, m = public_inputs.shape[0], public_inputs.shape[1]
        check(lib().ripp_tipp_verify_aggregate(self.handle, _p(vsrs), _p(vk), ctypes.c_size_t(m), _p(public_inputs),
                                               ctypes.c_size_t(n), _p(pb), ctypes.c_size_t(len(proof)), ctypes.byref(acc)))
        return bool(acc.value)

    def sipp_verify(self, a, b, r, value, proof):
        acc = ctypes.c_int(0)
        pb = self._bytes(proof)
        check(lib().ripp_sipp_verify(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(len(a)), _p(value), _p(pb),
                                     ctypes.c_size_t(len(proof)), ctypes.byref(acc)))
        return bool(acc.value)

    # ---- BLS12-377 (csrc/sipp377.cu): SIPP on the reference's own curve ----------------------------
    def pairing_ip_affine_377(self, g1, g2):
        out = np.empty(144, dtype=np.uint32)
        check(lib().ripp377_pairing_ip_affine(self.handle, _p(g1), ctypes.c_size_t(len(g1)), _p(g2), ctypes.c_size_t(len(g2)), _p(out)))
        return out

    def sipp_product_with_coeffs_377(self, a, b, r):
        out = np.empty(144, dtype=np.uint32)
        check(lib().ripp377_sipp_product_with_coeffs(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(len(a)), _p(out)))
        return out

    def sipp_prove_377(self, a, b, r, value):
        n = len(a)
        cap = max(n.bit_length() - 1, 0) * 1152 + 16
        proof = np.empty(cap, dtype=np.uint8)
        plen = ctypes.c_size_t()
        check(lib().ripp377_sipp_prove(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(n), _p(value), _p(proof),
                                       ctypes.c_size_t(cap), ctypes.byref(plen)))
        return proof[: plen.value].tobytes()

    def sipp_verify_377(self, a, b, r, value, proof):
        acc = ctypes.c_int(0)
        pb = self._bytes(proof)
        check(lib().ripp377_sipp_verify(self.handle, _p(a), _p(b), _p(r), ctypes.c_size_t(len(a)), _p(value), _p(pb),
                                        ctypes.c_size_t(len(proof)), ctypes.byref(acc)))
        return bool(acc.value)

    # ---- diagnostics ----------------------------------------------------------------------
    def test_elementwise(self, op, a, b, out_words):
        a = np.ascontiguousarray(a, dtype=np.uint32)
        n = a.shape[0]
        b = None if b is None else np.ascontiguousarray(b, dtype=np.uint32)
        r = np.empty((n, out_words), dtype=np.uint32)
        check(lib().ripp_test_elementwise(self.handle, TEST_OP_ID[op], _p(a), _p(b), _p(r), ctypes.c_size_t(n)))
        return r

    def bench_imad(self, kind, iters=2048):
        macs, ms = ctypes.c_double(), ctypes.c_double()
        check(lib().ripp_bench_imad(self.handle, int(kind), int(iters), ctypes.byref(macs), ctypes.byref(ms)))
        return macs.value, ms.value
