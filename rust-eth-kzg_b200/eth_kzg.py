"""ctypes binding of libc_eth_kzg_b200.so -- the same stub a maintainer of any of the reference's
language bindings would write against `c_eth_kzg.h` (see INTEGRATION.md).  Method names, argument
meaning and error behaviour follow the reference's Rust API:
  crates/eip7594/src/prover.rs:100-171, crates/eip7594/src/verifier.rs:72, crates/eip7594/src/eip4844_methods.rs:13-77.
There is no CPU fallback: if the library is missing or no B200 is visible, construction raises."""
import ctypes as C
import os
import subprocess

BYTES_PER_BLOB = 131072
BYTES_PER_CELL = 2048
BYTES_PER_COMMITMENT = 48
BYTES_PER_PROOF = 48
CELLS_PER_EXT_BLOB = 128

_HERE = os.path.dirname(os.path.abspath(__file__))


class KzgError(Exception):
    """The reference returns Err(...) (CResult.status == Err on the C ABI)."""


class _CResult(C.Structure):
    _fields_ = [("status", C.c_int), ("error_msg", C.c_void_p)]


def library_path():
    # EKZG_LIB: an A/B build of the same library (tools/*.sh compare kernel variants this way); the product path is the default
    return os.environ.get("EKZG_LIB") or os.path.join(_HERE, "lib", "libc_eth_kzg_b200.so")


def build_library():
    subprocess.check_call(["make", "-s", "-C", _HERE, "-j4"])
    return library_path()


_lib = None
_u8p = C.POINTER(C.c_uint8)


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise KzgError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)" % path)
    lib = C.CDLL(path)
    lib.eth_kzg_das_context_new.restype = C.c_void_p
    lib.eth_kzg_das_context_new.argtypes = [C.c_bool]
    lib.eth_kzg_das_context_free.argtypes = [C.c_void_p]
    lib.eth_kzg_free_error_message.argtypes = [C.c_void_p]
    for name in ("eth_kzg_constant_bytes_per_cell", "eth_kzg_constant_bytes_per_proof", "eth_kzg_constant_cells_per_ext_blob",
                 "eth_kzg_b200_context_table_bytes", "eth_kzg_b200_kernel_launch_count"):
        getattr(lib, name).restype = C.c_uint64
    lib.eth_kzg_b200_context_table_bytes.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_context_device.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_context_window.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_probe_imad_wide.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_probe_imad_wide.restype = C.c_double
    lib.eth_kzg_b200_context_srs_window.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_context_device_count.argtypes = [C.c_void_p]
    lib.eth_kzg_b200_context_device_at.argtypes = [C.c_void_p, C.c_int]
    for name in ("eth_kzg_blob_to_kzg_commitment", "eth_kzg_compute_cells_and_kzg_proofs", "eth_kzg_compute_cells",
                 "eth_kzg_verify_cell_kzg_proof_batch", "eth_kzg_recover_cells_and_proofs", "eth_kzg_compute_kzg_proof",
                 "eth_kzg_compute_blob_kzg_proof", "eth_kzg_verify_kzg_proof", "eth_kzg_verify_blob_kzg_proof",
                 "eth_kzg_verify_blob_kzg_proof_batch", "eth_kzg_b200_compute_cells_and_kzg_proofs_batch",
                 "eth_kzg_b200_compute_cells_and_kzg_proofs_device", "eth_kzg_b200_debug_fk20_stages", "eth_kzg_b200_debug_g1_ntt_prefix",
                 "eth_kzg_b200_recover_cells_and_kzg_proofs_batch", "eth_kzg_b200_blob_to_kzg_commitment_batch", "eth_kzg_b200_compute_blob_kzg_proof_batch",
                 "eth_kzg_b200_das_context_new_from_json", "eth_kzg_b200_debug_parse_trusted_setup_json", "eth_kzg_b200_debug_g2_keys"):
        getattr(lib, name).restype = _CResult
    for name in ("eth_kzg_b200_verify_cell_kzg_proof_batch_groups", "eth_kzg_b200_verify_blob_kzg_proof_batch_items"):
        if hasattr(lib, name):   # (an EKZG_LIB build from before these entry points lacks them)
            getattr(lib, name).restype = _CResult
    _lib = lib
    return lib


def _check(lib, res):
    if res.status != 0:
        msg = C.cast(res.error_msg, C.c_char_p).value.decode("utf-8", "replace") if res.error_msg else "error"
        lib.eth_kzg_free_error_message(res.error_msg)
        raise KzgError(msg)


def _batch_status(lib, res, status, n):
    """the status list of a batch call; raises KzgError when the call failed and no item is flagged (an infrastructure error)"""
    st = list(status.raw[:n])
    if res.status != 0:
        msg = C.string_at(res.error_msg).decode("utf-8", "replace") if res.error_msg else ""
        lib.eth_kzg_free_error_message(res.error_msg)
        if not any(st):
            raise KzgError("batch failed: " + msg)
    return st


def _exact(b, n, what):
    """the reference's API takes fixed-size array references; a wrong length cannot cross its FFI either"""
    if len(b) != n:
        raise KzgError("%s must be exactly %d bytes, got %d" % (what, n, len(b)))
    return bytes(b)


def _ptr_array(items):
    """array of pointers to individual byte strings (bindings/c/src/pointer_utils.rs:25-44)"""
    bufs = [C.create_string_buffer(bytes(x), len(x)) for x in items]
    arr = (C.c_void_p * max(len(bufs), 1))(*[C.addressof(b) for b in bufs])
    return arr, bufs


def _out_array(n, size):
    bufs = [C.create_string_buffer(size) for _ in range(n)]
    arr = (C.c_void_p * n)(*[C.addressof(b) for b in bufs])
    return arr, bufs


class DASContext:
    """Mirror of rust_eth_kzg::DASContext (crates/eip7594/src/lib.rs:41).  `use_precomp` is the only
    runtime knob of the C ABI (bindings/c/src/lib.rs:79)."""

    def __init__(self, use_precomp=False, _handle=None):
        self._lib = load_library()
        if _handle is not None:
            self._ctx = _handle
            return
        self._ctx = self._lib.eth_kzg_das_context_new(bool(use_precomp))
        if not self._ctx:
            raise KzgError("eth_kzg_das_context_new failed (no usable CUDA device? there is no CPU fallback)")

    @classmethod
    def from_json(cls, json_text, use_precomp=False, subgroup_check=True):
        """DASContext::new(&TrustedSetup::from_json(json), use_precomp) -- or from_json_unchecked with subgroup_check=False
        (crates/trusted_setup/src/lib.rs:112-127).  Raises KzgError where the reference panics."""
        lib = load_library()
        data = json_text.encode() if isinstance(json_text, str) else bytes(json_text)
        out = C.c_void_p()
        _check(lib, lib.eth_kzg_b200_das_context_new_from_json(data, C.c_uint64(len(data)), C.c_bool(subgroup_check), C.c_bool(use_precomp),
                                                               C.byref(out)))
        return cls(_handle=out.value)

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.eth_kzg_das_context_free(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- info -------------------------------------------------------------------------------
    @property
    def handle(self):
        return self._ctx

    @property
    def device(self):
        return self._lib.eth_kzg_b200_context_device(self._ctx)

    @property
    def window(self):
        return self._lib.eth_kzg_b200_context_window(self._ctx)

    @property
    def table_bytes(self):
        return self._lib.eth_kzg_b200_context_table_bytes(self._ctx)

    def probe_imad_wide(self):
        """measured carry-chained IMAD.WIDE multiply-adds per second on this context's device"""
        return float(self._lib.eth_kzg_b200_probe_imad_wide(C.c_void_p(self._ctx)))

    @property
    def srs_window(self):
        return self._lib.eth_kzg_b200_context_srs_window(self._ctx)

    @property
    def devices(self):
        """CUDA ordinals this context spans (EKZG_DEVICES; one entry unless that is set)"""
        n = self._lib.eth_kzg_b200_context_device_count(self._ctx)
        return [self._lib.eth_kzg_b200_context_device_at(self._ctx, i) for i in range(n)]

    # ---- EIP-7594 prover (crates/eip7594/src/prover.rs:100-171) ------------------------------
    def blob_to_kzg_commitment(self, blob):
        out = C.create_string_buffer(48)
        _check(self._lib, self._lib.eth_kzg_blob_to_kzg_commitment(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), out))
        return out.raw

    def compute_cells_and_kzg_proofs(self, blob):
        cells, cb = _out_array(CELLS_PER_EXT_BLOB, BYTES_PER_CELL)
        proofs, pb = _out_array(CELLS_PER_EXT_BLOB, BYTES_PER_PROOF)
        _check(self._lib, self._lib.eth_kzg_compute_cells_and_kzg_proofs(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), cells, proofs))
        return [b.raw for b in cb], [b.raw for b in pb]

    def compute_cells(self, blob):
        cells, cb = _out_array(CELLS_PER_EXT_BLOB, BYTES_PER_CELL)
        _check(self._lib, self._lib.eth_kzg_compute_cells(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), cells))
        return [b.raw for b in cb]

    def recover_cells_and_kzg_proofs(self, cell_indices, cells):
        cells = [_exact(c, BYTES_PER_CELL, "cell") for c in cells]
        arr, keep = _ptr_array(cells)
        idx = (C.c_uint64 * max(len(cell_indices), 1))(*cell_indices)
        oc, cb = _out_array(CELLS_PER_EXT_BLOB, BYTES_PER_CELL)
        op, pb = _out_array(CELLS_PER_EXT_BLOB, BYTES_PER_PROOF)
        _check(self._lib, self._lib.eth_kzg_recover_cells_and_proofs(C.c_void_p(self._ctx), C.c_uint64(len(cells)), arr,
                                                                     C.c_uint64(len(cell_indices)), idx, oc, op))
        del keep
        return [b.raw for b in cb], [b.raw for b in pb]

    # ---- EIP-7594 verifier (crates/eip7594/src/verifier.rs:72) --------------------------------
    def verify_cell_kzg_proof_batch(self, commitments, cell_indices, cells, proofs):
        commitments = [_exact(c, 48, "commitment") for c in commitments]
        cells = [_exact(c, BYTES_PER_CELL, "cell") for c in cells]
        proofs = [_exact(p, 48, "proof") for p in proofs]
        ca, k1 = _ptr_array(commitments)
        cl, k2 = _ptr_array(cells)
        pa, k3 = _ptr_array(proofs)
        idx = (C.c_uint64 * max(len(cell_indices), 1))(*cell_indices)
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_verify_cell_kzg_proof_batch(
            C.c_void_p(self._ctx), C.c_uint64(len(commitments)), ca, C.c_uint64(len(cell_indices)), idx,
            C.c_uint64(len(cells)), cl, C.c_uint64(len(proofs)), pa, C.byref(ok)))
        del k1, k2, k3
        return bool(ok.value)

    def verify_cell_kzg_proof_batch_groups(self, commitments, cell_indices, cells, proofs, groups, n_groups=None):
        """verify_cell_kzg_proof_batch with a verdict per caller-defined group: opening k belongs to group groups[k]
        (< n_groups, default max(groups) + 1).  -> (all_ok, [status per group]): 0 verifies (also an empty group), 1 does not,
        2 holds a malformed item (invalid commitment / proof, non-canonical cell, cell index >= 128).  Raises KzgError only
        for structural faults: lengths that differ, a group id >= n_groups, n_groups above 2^20."""
        n = len(commitments)
        if not (n == len(cell_indices) == len(cells) == len(proofs) == len(groups)):
            raise KzgError("Verifier(BatchVerificationInputsMustHaveSameLength)")
        if n_groups is None:
            n_groups = max(groups) + 1 if n else 0
        if min(groups, default=0) < 0 or max(groups, default=0) >= 1 << 32:
            raise KzgError("group id out of range")
        commitments = [_exact(c, 48, "commitment") for c in commitments]
        cells = [_exact(c, BYTES_PER_CELL, "cell") for c in cells]
        proofs = [_exact(p, 48, "proof") for p in proofs]
        ca, k1 = _ptr_array(commitments)
        cl, k2 = _ptr_array(cells)
        pa, k3 = _ptr_array(proofs)
        idx = (C.c_uint64 * max(n, 1))(*cell_indices)
        grp = (C.c_uint32 * max(n, 1))(*groups)
        status = C.create_string_buffer(max(n_groups, 1)) if n_groups <= 1 << 20 else None
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_b200_verify_cell_kzg_proof_batch_groups(
            C.c_void_p(self._ctx), C.c_uint64(n), ca, idx, cl, pa, C.c_uint64(n_groups), grp, status, C.byref(ok)))
        del k1, k2, k3
        return bool(ok.value), list(status.raw[:n_groups])

    # ---- EIP-4844 methods re-exported on DASContext (crates/eip7594/src/eip4844_methods.rs:13-77) ----
    def compute_kzg_proof(self, blob, z):
        proof, y = C.create_string_buffer(48), C.create_string_buffer(32)
        _check(self._lib, self._lib.eth_kzg_compute_kzg_proof(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), _exact(z, 32, "z"), proof, y))
        return proof.raw, y.raw

    def compute_blob_kzg_proof(self, blob, commitment):
        proof = C.create_string_buffer(48)
        _check(self._lib, self._lib.eth_kzg_compute_blob_kzg_proof(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"),
                                                                   _exact(commitment, 48, "commitment"), proof))
        return proof.raw

    def verify_kzg_proof(self, commitment, z, y, proof):
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_verify_kzg_proof(C.c_void_p(self._ctx), _exact(commitment, 48, "commitment"), _exact(z, 32, "z"),
                                                             _exact(y, 32, "y"), _exact(proof, 48, "proof"), C.byref(ok)))
        return bool(ok.value)

    def verify_blob_kzg_proof(self, blob, commitment, proof):
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_verify_blob_kzg_proof(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"),
                                                                  _exact(commitment, 48, "commitment"), _exact(proof, 48, "proof"), C.byref(ok)))
        return bool(ok.value)

    def verify_blob_kzg_proof_batch(self, blobs, commitments, proofs):
        blobs = [_exact(b, BYTES_PER_BLOB, "blob") for b in blobs]
        commitments = [_exact(c, 48, "commitment") for c in commitments]
        proofs = [_exact(p, 48, "proof") for p in proofs]
        ba, k1 = _ptr_array(blobs)
        ca, k2 = _ptr_array(commitments)
        pa, k3 = _ptr_array(proofs)
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_verify_blob_kzg_proof_batch(
            C.c_void_p(self._ctx), C.c_uint64(len(blobs)), ba, C.c_uint64(len(commitments)), ca, C.c_uint64(len(proofs)), pa, C.byref(ok)))
        del k1, k2, k3
        return bool(ok.value)

    def verify_blob_kzg_proof_batch_items(self, blobs, commitments, proofs):
        """verify_blob_kzg_proof_batch with a verdict per blob -> (all_ok, [status]): 0 verifies, 1 does not, 2 malformed
        (non-canonical blob, invalid commitment or proof).  Raises KzgError only when the lengths differ."""
        n = len(blobs)
        if not (n == len(commitments) == len(proofs)):
            raise KzgError("Verifier(BatchVerificationInputsMustHaveSameLength)")
        blobs = [_exact(b, BYTES_PER_BLOB, "blob") for b in blobs]
        commitments = [_exact(c, 48, "commitment") for c in commitments]
        proofs = [_exact(p, 48, "proof") for p in proofs]
        ba, k1 = _ptr_array(blobs)
        ca, k2 = _ptr_array(commitments)
        pa, k3 = _ptr_array(proofs)
        status = C.create_string_buffer(max(n, 1))
        ok = C.c_bool(False)
        _check(self._lib, self._lib.eth_kzg_b200_verify_blob_kzg_proof_batch_items(C.c_void_p(self._ctx), C.c_uint64(n), ba, ca, pa, status,
                                                                                   C.byref(ok)))
        del k1, k2, k3
        return bool(ok.value), list(status.raw[:n])

    # ---- additive batch / device entry points --------------------------------------------------
    def compute_cells_and_kzg_proofs_batch(self, blobs_flat, n, want_proofs=True):
        """n blobs, contiguous host bytes -> (cells_flat, proofs_flat, status list).  Raises KzgError if any blob is invalid."""
        blobs_flat = _exact(blobs_flat, n * BYTES_PER_BLOB, "blobs")
        cells = C.create_string_buffer(n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL)
        proofs = C.create_string_buffer(n * CELLS_PER_EXT_BLOB * 48) if want_proofs else None
        status = C.create_string_buffer(max(n, 1))
        res = self._lib.eth_kzg_b200_compute_cells_and_kzg_proofs_batch(C.c_void_p(self._ctx), C.c_uint64(n), blobs_flat, cells, proofs, status)
        st = _batch_status(self._lib, res, status, n)
        return cells.raw, (proofs.raw if want_proofs else None), st

    def blob_to_kzg_commitment_batch(self, blobs_flat, n):
        """-> (commitments_flat (n*48 B), status list); raises only on infrastructure errors"""
        out = C.create_string_buffer(max(n, 1) * 48)
        status = C.create_string_buffer(max(n, 1))
        res = self._lib.eth_kzg_b200_blob_to_kzg_commitment_batch(C.c_void_p(self._ctx), C.c_uint64(n), _exact(blobs_flat, n * BYTES_PER_BLOB, "blobs"), out, status)
        st = _batch_status(self._lib, res, status, n)
        return out.raw[:n * 48], st

    def compute_blob_kzg_proof_batch(self, blobs_flat, commitments_flat, n):
        out = C.create_string_buffer(max(n, 1) * 48)
        status = C.create_string_buffer(max(n, 1))
        res = self._lib.eth_kzg_b200_compute_blob_kzg_proof_batch(C.c_void_p(self._ctx), C.c_uint64(n), _exact(blobs_flat, n * BYTES_PER_BLOB, "blobs"),
                                                                  _exact(commitments_flat, n * 48, "commitments"), out, status)
        st = _batch_status(self._lib, res, status, n)
        return out.raw[:n * 48], st

    def recover_cells_and_kzg_proofs_batch(self, indices_per_blob, cells_per_blob):
        """lists (one entry per blob) of cell index lists and of lists of 2048-byte cells -> (cells_flat, proofs_flat, status)"""
        n = len(indices_per_blob)
        counts = (C.c_uint64 * max(n, 1))(*[len(x) for x in indices_per_blob])
        flat_idx = [i for x in indices_per_blob for i in x]
        idx = (C.c_uint64 * max(len(flat_idx), 1))(*flat_idx)
        cells = b"".join(_exact(c, BYTES_PER_CELL, "cell") for x in cells_per_blob for c in x)
        oc = C.create_string_buffer(max(n, 1) * CELLS_PER_EXT_BLOB * BYTES_PER_CELL)
        op = C.create_string_buffer(max(n, 1) * CELLS_PER_EXT_BLOB * 48)
        status = C.create_string_buffer(max(n, 1))
        res = self._lib.eth_kzg_b200_recover_cells_and_kzg_proofs_batch(C.c_void_p(self._ctx), C.c_uint64(n), counts, idx, cells, oc, op, status)
        st = _batch_status(self._lib, res, status, n)
        return oc.raw, op.raw, st

    def compute_cells_and_kzg_proofs_device(self, n, d_blobs, d_cells, d_proofs, d_status, stream=0):
        """device pointers (ints), asynchronous on `stream`"""
        _check(self._lib, self._lib.eth_kzg_b200_compute_cells_and_kzg_proofs_device(
            C.c_void_p(self._ctx), C.c_uint64(n), C.c_void_p(d_blobs), C.c_void_p(d_cells), C.c_void_p(d_proofs), C.c_void_p(d_status), C.c_void_p(stream)))

    def set_profiling(self, on):
        self._lib.eth_kzg_b200_set_profiling(C.c_void_p(self._ctx), C.c_bool(bool(on)))

    def collect_stage_times(self):
        """-> (batches, [ms per stage: K1 coeffs/cells, K2 scalars, K4 MSM, K5 G1 NTT, K6 compress])"""
        ms = (C.c_double * 5)()
        n = self._lib.eth_kzg_b200_collect_stage_times(C.c_void_p(self._ctx), ms)
        return n, list(ms)

    def debug_g1_ntt_prefix(self, blob, phases):
        out = C.create_string_buffer(128 * 48)
        _check(self._lib, self._lib.eth_kzg_b200_debug_g1_ntt_prefix(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), C.c_int(phases), out))
        return [out.raw[48 * i:48 * i + 48] for i in range(128)]

    def debug_fk20_stages(self, blob):
        sc = (C.c_uint32 * (128 * 64 * 8))()
        msm = C.create_string_buffer(128 * 48)
        h = C.create_string_buffer(64 * 48)
        _check(self._lib, self._lib.eth_kzg_b200_debug_fk20_stages(C.c_void_p(self._ctx), _exact(blob, BYTES_PER_BLOB, "blob"), sc, msm, h))
        scalars = [[sum(int(sc[(j * 64 + k) * 8 + l]) << (32 * l) for l in range(8)) for k in range(64)] for j in range(128)]
        return scalars, [msm.raw[48 * j:48 * j + 48] for j in range(128)], [h.raw[48 * i:48 * i + 48] for i in range(64)]
