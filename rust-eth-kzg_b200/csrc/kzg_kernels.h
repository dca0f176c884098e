// Host-visible launch wrappers for the kernels in kzg_kernels.cu / kzg_kernels_*.cu.
#pragma once
#include <atomic>
#include "kzg_device.cuh"

namespace ekzg {

// every kernel launch of the library goes through this check; the counter feeds bench.py's gpu_launches
extern std::atomic<unsigned long long> g_kernel_launches;
#define EKZG_LAUNCH_CHECK()                                                  \
    do {                                                                     \
        ::ekzg::g_kernel_launches.fetch_add(1, std::memory_order_relaxed);   \
        cudaError_t e_ = cudaGetLastError();                                 \
        if (e_ != cudaSuccess) return e_;                                    \
    } while (0)

cudaError_t kernels_init();
cudaError_t launch_powers(Fr* out, const uint32_t* base_mont, int n, cudaStream_t st, const uint32_t* scale_mont = nullptr);
cudaError_t launch_blob_to_coeffs_cells(const uint8_t* blobs, Fr* coeffs, uint8_t* cells, uint32_t* status, const DevTables& T,
                                        int B, bool want_cells, cudaStream_t st);
cudaError_t launch_coeffs_to_cells(const Fr* coeffs, uint8_t* cells, const DevTables& T, int B, cudaStream_t st);
cudaError_t launch_coeffs_to_blob(const Fr* coeffs, uint8_t* blobs, const DevTables& T, int B, cudaStream_t st);   // cells 0..63 only
// blobs [b0, b0 + cnt) of a batch of B (cnt < 0: to the end)
cudaError_t launch_toeplitz_scalars(const Fr* coeffs, uint32_t* scalars, const DevTables& T, int B, cudaStream_t st, int b0 = 0, int cnt = -1);
// scratch: fixed_msm_scratch_bytes(T) bytes for the batched-affine kernel (nullptr: the XYZZ kernels are used)
cudaError_t launch_fixed_msm(const uint32_t* scalars, G1Jac* pts, const MsmTable& T, int ngroups, int B, cudaStream_t st, int b0 = 0, int cnt = -1,
                             void* scratch = nullptr);
size_t fixed_msm_scratch_bytes(const MsmTable& T);
size_t g1_ntt_queue_words(int B);
size_t g1_ntt_scratch_bytes();   // per concurrently running K5 launch (odd-multiples tables of the resident warps); 0 on error
cudaError_t launch_g1_ntt_phases(G1Jac* pts, int B, int ph0, int ph1, uint32_t* queue, void* scratch, cudaStream_t st);
void set_k5_throughput_hint(bool on);   // this thread's next K5 launches: least work (radix-2) rather than shortest chain, for batches above 64 blobs
cudaError_t launch_fk20_g1_ntts(G1Jac* pts, int B, uint32_t* queue, void* scratch, cudaStream_t st);
cudaError_t launch_g1_compress(const G1Jac* pts, uint8_t* out, int npos, int B, cudaStream_t st);
cudaError_t launch_g1_decompress(const uint8_t* in, G1Affine* out, uint32_t* status, int n, cudaStream_t st);
cudaError_t launch_fk20_setup(const G1Affine* srs, G1Jac* pts_scratch, G1Affine* qaff, G1Affine* table, const DevTables& T,
                              uint32_t* queue, void* ntt_scratch, cudaStream_t st);
cudaError_t launch_srs_table_setup(const G1Affine* srs, int npoints, G1Affine* qaff, G1Affine* table, const MsmTable& T, cudaStream_t st);

// kzg_kernels_4844.cu
cudaError_t launch_blob_challenge(const uint8_t* blobs, const uint8_t* commitments, Fr* z, int B, cudaStream_t st);
cudaError_t launch_scalars_from_be(const uint8_t* in, Fr* out, uint32_t* status, int n, cudaStream_t st);
cudaError_t launch_quotient(const Fr* coeffs, const Fr* z, uint32_t* scalars, uint8_t* y_out, int B, cudaStream_t st);
cudaError_t launch_coset_quotients(const Fr* coeffs, uint32_t* scalars, const DevTables& T, int nblobs, cudaStream_t st);   // [4096][128 nblobs] plain
cudaError_t launch_coeffs_to_scalars(const Fr* coeffs, uint32_t* scalars, int B, cudaStream_t st);
cudaError_t launch_sum_positions(G1Jac* pts, int B, int count, int stride, cudaStream_t st);
cudaError_t launch_g1_subgroup(const G1Affine* pts, uint32_t* status, int n, const G1Affine* pts2, uint32_t* status2, int n2, cudaStream_t st);   // status 2 where a decompressed point is outside G1
cudaError_t launch_g1_validate(const uint8_t* in, G1Affine* out, uint32_t* status, int n, bool check_subgroup, cudaStream_t st);

// kzg_kernels_recover.cu
cudaError_t recover_kernels_init();
cudaError_t launch_recover_coeffs(const uint8_t* cells, const int16_t* slotmap, Fr* ze, Fr* czinv, Fr* bufA, Fr* bufB, Fr* coeffs,
                                  uint32_t* status, const DevTables& T, const Fr* shift_fwd, const Fr* shift_inv, const uint32_t* gen64_mont,
                                  int B, cudaStream_t st, const uint32_t* cell_off = nullptr);

// kzg_kernels_verify.cu
cudaError_t launch_powers_from_hash(const uint8_t* hash, Fr* rpow, int n, cudaStream_t st);
cudaError_t launch_cell_verify_scalars(const Fr* rpow, const uint32_t* col, uint32_t* s1, uint32_t* s2, const DevTables& T, int n, cudaStream_t st);
cudaError_t launch_commitment_weights(const Fr* rpow, const uint32_t* row, uint32_t* wout, int n, int m, cudaStream_t st);
cudaError_t launch_column_sums(const G1Jac* prods, const uint32_t* col, G1Jac* colsum, G1Jac* weighted, int n, cudaStream_t st);
cudaError_t launch_scalar_mul(const G1Affine* pts, const uint32_t* scalars, G1Jac* out, int n, cudaStream_t st);
cudaError_t launch_sum_points(const G1Jac* in, int n, G1Jac* scratch, G1Jac* out, cudaStream_t st);
cudaError_t launch_cell_interp(const uint8_t* cells, const uint32_t* col, const Fr* rpow, Fr* interp, uint32_t* status, const DevTables& T,
                               int n, cudaStream_t st);
cudaError_t launch_interp_column_sum(const Fr* interp, uint32_t* out, int n, cudaStream_t st);
// K7 (kzg_kernels_msm.cu): bucket-method MSM over n variable points for one or two scalar sets
size_t msm_bucket_scratch_bytes(int n, int sets);
constexpr int MSM_BUCKET_MIN = 1 << 30;   // batch size from which the verifier takes the bucket method by itself (measured: see DESIGN.md section 4.3)
cudaError_t launch_msm_bucket(const G1Affine* pts, const uint32_t* scalars0, const uint32_t* scalars1, int n, G1Jac* out0, G1Jac* out1, void* scratch,
                              cudaStream_t st);
constexpr int PAIRING_INPUT_WORDS = 37;   // per point: Jacobian X, Y, Z (Montgomery limbs) + identity flag
cudaError_t launch_pairing_inputs(const G1Jac* a0, const G1Jac* b0, const G1Jac* b1, const G1Jac* b2, uint32_t* out, cudaStream_t st);
cudaError_t launch_kzg_verify_pairs(const G1Affine* commitments, const G1Affine* proofs, const Fr* z, const Fr* y, const Fr* rpow, G1Affine* pts,
                                    uint32_t* scalars, int n, cudaStream_t st);   // 4n (point, scalar) pairs, kind-major
cudaError_t launch_poly_eval(const Fr* coeffs, const Fr* z, Fr* y, uint8_t* y_be, int B, cudaStream_t st);
cudaError_t launch_fr_to_be(const Fr* in, uint8_t* out, int n, cudaStream_t st);
// verdicts per group / per item: masking of malformed items, then the per-group sums of the failure path
cudaError_t launch_cell_canonical(const uint8_t* cells, uint32_t* bad, int n, cudaStream_t st);   // bad[k] = cell k holds a value >= r
cudaError_t launch_mask_openings(Fr* rpow, const uint32_t* stp, const uint32_t* stc, const uint32_t* row, uint32_t* col, const uint32_t* cell_bad,
                                 G1Affine* a_p, G1Affine* a_c, uint32_t* flag, int n, int m, cudaStream_t st);
cudaError_t launch_mask_items(Fr* rpow, const uint32_t* stb, const uint32_t* stc, const uint32_t* stp, G1Affine* a_c, G1Affine* a_p, uint32_t* flag,
                              int n, cudaStream_t st);
cudaError_t launch_gather_points(const G1Affine* pts, const uint32_t* idx, G1Affine* out, int n, cudaStream_t st);
// sums[s * G + g] = sum over the CSR segment of group g of in_s (s = 0, 1, 2); groups listed in `small` get a warp, in `large` a CTA
cudaError_t launch_group_point_sums(const G1Jac* in0, const G1Jac* in1, const G1Jac* in2, const uint32_t* order, const uint32_t* off,
                                    const uint32_t* small, int n_small, const uint32_t* large, int n_large, G1Jac* sums, int G, cudaStream_t st);
cudaError_t launch_group_interp_sums(const Fr* interp, const uint32_t* order, const uint32_t* off, uint32_t* out, int G, cudaStream_t st);   // [64][G] plain
cudaError_t launch_pairing_inputs_n(const G1Jac* a, const G1Jac* b0, const G1Jac* b1, const G1Jac* b2, bool sub_b1, uint32_t* out, int n,
                                    cudaStream_t st);
// verify_blob_cell_proofs_batch: byte comparison of B blobs' recomputed proofs (B x 128 x 48 B) and commitments (B x 48 B) with the
// supplied ones; cell_mm[B][128]: 0 equal, 1 differs, 2 blob_status[b] != 0 (non-canonical blob); blob_mm[B]: BLOB_MM_* bits
enum : uint8_t { BLOB_MM_PROOF = 1, BLOB_MM_COMMITMENT = 2, BLOB_MM_NON_CANONICAL = 4 };
cudaError_t launch_compare_blob_proofs(const uint8_t* computed_proofs, const uint8_t* given_proofs, const uint8_t* computed_c48,
                                       const uint8_t* given_c48, const uint32_t* blob_status, uint8_t* cell_mm, uint8_t* blob_mm, int B,
                                       cudaStream_t st);


}  // namespace ekzg
