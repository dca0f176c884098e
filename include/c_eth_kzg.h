/*
 * C ABI of the B200-native KZG backend: libc_eth_kzg_b200.so.
 *
 * This is the drop-in boundary.  The first block reproduces, symbol for symbol, the header cbindgen
 * generates from the reference's `bindings/c/src/lib.rs` (checked-in rendering:
 * bindings/nim/nim_code/nim_eth_kzg/header.nim:5-140): same names, argument order, types, ownership
 * and error behaviour, so the reference's C#/Nim/Go/Java shims link against this library unchanged.
 * The second block is additive: batch entry points and device-pointer entry points that the
 * reference does not have (its API is one blob per call, SURVEY.md §0.8).
 *
 * Ownership (bindings/c/src/pointer_utils.rs:53-62): every data buffer is caller-allocated; `out_cells`
 * and `out_proofs` are arrays of 128 caller-owned pointers (2048 B / 48 B each).  The library owns only
 * the context and error strings.  A failing call returns {Err, malloc'd message}; free it with
 * eth_kzg_free_error_message.  Verification functions return Ok with *verified = false for a wrong
 * proof and Err for malformed input (bindings/c/src/lib.rs:272-280).
 */
#ifndef C_ETH_KZG_B200_H
#define C_ETH_KZG_B200_H

#include <stdbool.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* bindings/c/src/lib.rs:41-44 (opaque) */
typedef struct DASContext DASContext;

/* bindings/c/src/lib.rs:118-123 */
typedef enum CResultStatus {
    Ok,
    Err,
} CResultStatus;

/* bindings/c/src/lib.rs:128-132 */
typedef struct CResult {
    CResultStatus status;
    char *error_msg;
} CResult;

/* bindings/c/src/lib.rs:79.  Builds the SRS-derived tables on the calling thread's current CUDA device (override
 * with EKZG_DEVICE), or on every device named in EKZG_DEVICES ("all" or a comma list of ordinals): batch calls are
 * then sharded over those devices and single-item calls dealt round-robin, the counterpart of the reference's rayon
 * fan-out over the cores of the box.  The caller's current device is restored before every entry point returns.
 * use_precomp selects the fixed-base window widths (the reference's UsePrecomp, fixed_base_msm.rs:83-89):
 *   false -> 8-bit windows, 3 GiB of tables per device;
 *   true  -> the WIDEST windows whose tables fit the device's free memory minus a 16 GiB reserve (or minus
 *            EKZG_HBM_RESERVE_GIB): on an empty 180 GB B200 that is 14-bit FK20 windows (114 GiB) plus 13-bit SRS windows
 *            (30 GiB), built on the device in about 2 s.  A second context or another tenant on the same GPU gets
 *            narrower windows (more point additions per blob, up to 1.5x slower) -- EKZG_TRACE=1 prints the widths and
 *            bytes chosen; EKZG_FK20_WINDOW / EKZG_SRS_WINDOW (4..16) pin them.
 * Returns NULL if no CUDA device is usable: there is no CPU fallback. */
DASContext *eth_kzg_das_context_new(bool use_precomp);

/* bindings/c/src/lib.rs:109 (null-safe) */
void eth_kzg_das_context_free(DASContext *ctx);

/* bindings/c/src/lib.rs:171 (null-safe) */
void eth_kzg_free_error_message(char *c_message);

/* bindings/c/src/lib.rs:196  blob: 131072 B, out: 48 B */
CResult eth_kzg_blob_to_kzg_commitment(const DASContext *ctx, const uint8_t *blob, uint8_t *out);

/* bindings/c/src/lib.rs:226  out_cells: 128 x 2048 B, out_proofs: 128 x 48 B */
CResult eth_kzg_compute_cells_and_kzg_proofs(const DASContext *ctx, const uint8_t *blob, uint8_t **out_cells,
                                             uint8_t **out_proofs);

/* bindings/c/src/lib.rs:255 */
CResult eth_kzg_compute_cells(const DASContext *ctx, const uint8_t *blob, uint8_t **out_cells);

/* bindings/c/src/lib.rs:309 */
CResult eth_kzg_verify_cell_kzg_proof_batch(const DASContext *ctx, uint64_t commitments_length,
                                            const uint8_t *const *commitments, uint64_t cell_indices_length,
                                            const uint64_t *cell_indices, uint64_t cells_length,
                                            const uint8_t *const *cells, uint64_t proofs_length,
                                            const uint8_t *const *proofs, bool *verified);

/* bindings/c/src/lib.rs:366 */
CResult eth_kzg_recover_cells_and_proofs(const DASContext *ctx, uint64_t cells_length, const uint8_t *const *cells,
                                         uint64_t cell_indices_length, const uint64_t *cell_indices, uint8_t **out_cells,
                                         uint8_t **out_proofs);

/* bindings/c/src/lib.rs:395-405 */
uint64_t eth_kzg_constant_bytes_per_cell(void);
uint64_t eth_kzg_constant_bytes_per_proof(void);
uint64_t eth_kzg_constant_cells_per_ext_blob(void);

/* bindings/c/src/lib.rs:423  z: 32 B, out_proof: 48 B, out_y: 32 B */
CResult eth_kzg_compute_kzg_proof(const DASContext *ctx, const uint8_t *blob, const uint8_t *z, uint8_t *out_proof,
                                  uint8_t *out_y);

/* bindings/c/src/lib.rs:451 */
CResult eth_kzg_compute_blob_kzg_proof(const DASContext *ctx, const uint8_t *blob, const uint8_t *commitment,
                                       uint8_t *out_proof);

/* bindings/c/src/lib.rs:480 */
CResult eth_kzg_verify_kzg_proof(const DASContext *ctx, const uint8_t *commitment, const uint8_t *z, const uint8_t *y,
                                 const uint8_t *proof, bool *verified);

/* bindings/c/src/lib.rs:510 */
CResult eth_kzg_verify_blob_kzg_proof(const DASContext *ctx, const uint8_t *blob, const uint8_t *commitment,
                                      const uint8_t *proof, bool *verified);

/* bindings/c/src/lib.rs:546 */
CResult eth_kzg_verify_blob_kzg_proof_batch(const DASContext *ctx, uint64_t blobs_length, const uint8_t *const *blobs,
                                            uint64_t commitments_length, const uint8_t *const *commitments,
                                            uint64_t proofs_length, const uint8_t *const *proofs, bool *verified);

/* ------------------------------------------------------------------------------------------------
 * Additive B200 entry points (not in the reference; SURVEY.md §8b "Gap vs BASELINE.json configs").
 * ---------------------------------------------------------------------------------------------- */

/* A context over a CALLER-SUPPLIED trusted setup: the C-ABI form of what a Rust user of the reference writes as
 *   DASContext::new(&TrustedSetup::from_json(json), use_precomp)            (subgroup_check = true)
 *   DASContext::new(&TrustedSetup::from_json_unchecked(json), use_precomp)  (subgroup_check = false)
 * (crates/trusted_setup/src/lib.rs:112-127, crates/eip7594/src/lib.rs DASContext::new, crates/eip7594/src/trusted_setup.rs:6-23).
 * `json` is the consensus-specs file layout: {"g1_monomial": 4096 x "0x" + 96 hex digits, "g2_monomial": 65 x "0x" + 192 hex
 * digits, ...}; other keys (g1_lagrange) are skipped as the reference skips them.  The 4096 G1 points are decompressed and
 * checked (curve equation; prime-order subgroup unless subgroup_check is false) on the device, the 65 G2 points on the host;
 * the FK20 and SRS tables are then built from them exactly as for the embedded setup.  Where the reference panics (malformed
 * JSON, missing "0x", wrong length, invalid point) this returns Err and leaves *out_ctx NULL.  Free with
 * eth_kzg_das_context_free. */
CResult eth_kzg_b200_das_context_new_from_json(const char *json, uint64_t json_len, bool subgroup_check, bool use_precomp,
                                               DASContext **out_ctx);

/* n independent blobs in one call, HOST buffers, contiguous: blobs = n*131072 B, out_cells = n*128*2048 B,
 * out_proofs = n*128*48 B.  blob_status[i] (optional, may be NULL) is 0 for a valid blob and 1 for a
 * non-canonical one, whose outputs are left unspecified; the call returns Err iff any blob is invalid.
 * Internally the batch is streamed through the device in chunks with copies overlapped with compute.
 * Batch form of eip7594/src/prover.rs:117-134. */
CResult eth_kzg_b200_compute_cells_and_kzg_proofs_batch(const DASContext *ctx, uint64_t n, const uint8_t *blobs,
                                                        uint8_t *out_cells, uint8_t *out_proofs, uint8_t *blob_status);

/* Same computation on buffers that already live on the context's device (layout as above, 16-byte aligned);
 * d_status is n uint32 (0 ok / 1 invalid blob).  Runs asynchronously on `cuda_stream` (a cudaStream_t; 0 for the
 * default stream); no host synchronisation.  d_cells may be NULL to skip cell output. */
CResult eth_kzg_b200_compute_cells_and_kzg_proofs_device(const DASContext *ctx, uint64_t n, const void *d_blobs,
                                                         void *d_cells, void *d_proofs, void *d_status, void *cuda_stream);

/* Batch forms of eth_kzg_blob_to_kzg_commitment / eth_kzg_compute_blob_kzg_proof (BASELINE.json config #2):
 * contiguous HOST buffers, n*131072 B of blobs (and n*48 B of commitments) in, n*48 B out.  item_status[i]
 * (optional): 0 ok, 1 invalid blob, 2 invalid commitment.  Err iff any item is invalid. */
CResult eth_kzg_b200_blob_to_kzg_commitment_batch(const DASContext *ctx, uint64_t n, const uint8_t *blobs, uint8_t *out,
                                                  uint8_t *item_status);
CResult eth_kzg_b200_compute_blob_kzg_proof_batch(const DASContext *ctx, uint64_t n, const uint8_t *blobs,
                                                  const uint8_t *commitments, uint8_t *out_proofs, uint8_t *item_status);

/* Batch form of eth_kzg_recover_cells_and_proofs (BASELINE.json config #4).  Blob i supplies cell_counts[i] cells;
 * cell_indices and cells (2048 B each) of all blobs are concatenated in blob order.  Outputs contiguous per blob
 * (128*2048 B cells, 128*48 B proofs).  item_status[i] (optional): 0 ok, 3 invalid indices (range / order / count),
 * 1 non-canonical cell scalar, 4 recovered polynomial of degree >= 4096.  Err iff any item is invalid. */
CResult eth_kzg_b200_recover_cells_and_kzg_proofs_batch(const DASContext *ctx, uint64_t n, const uint64_t *cell_counts,
                                                        const uint64_t *cell_indices, const uint8_t *cells, uint8_t *out_cells,
                                                        uint8_t *out_proofs, uint8_t *item_status);

/* verify_cell_kzg_proof_batch with a verdict per caller-defined group of openings (for example the cells of one column
 * sidecar).  Inputs as eth_kzg_verify_cell_kzg_proof_batch (n of each), plus group_of[n] (< n_groups).  group_status[n_groups]:
 * 0 every opening of the group verifies (also: an empty group), 1 the group's openings do not verify, 2 the group holds a
 * malformed item (invalid commitment / proof encoding or subgroup, non-canonical cell scalar, cell index >= 128; an invalid
 * commitment marks every group with a cell that refers to it).  *all_ok = every group is 0.  The challenge is the plain
 * call's, so with no malformed item *all_ok equals its result.  Err only for structural faults: a group id >= n_groups,
 * n_groups above 2^20. */
CResult eth_kzg_b200_verify_cell_kzg_proof_batch_groups(const DASContext *ctx, uint64_t n, const uint8_t *const *commitments,
                                                        const uint64_t *cell_indices, const uint8_t *const *cells,
                                                        const uint8_t *const *proofs, uint64_t n_groups, const uint32_t *group_of,
                                                        uint8_t *group_status, bool *all_ok);

/* verify_blob_kzg_proof_batch with a verdict per blob: item_status[n] 0 verifies, 1 does not, 2 malformed (non-canonical
 * blob, invalid commitment or proof).  *all_ok = every item is 0; with no malformed item it equals the plain call's result. */
CResult eth_kzg_b200_verify_blob_kzg_proof_batch_items(const DASContext *ctx, uint64_t n, const uint8_t *const *blobs,
                                                       const uint8_t *const *commitments, const uint8_t *const *proofs,
                                                       uint8_t *item_status, bool *all_ok);

/* CUDA device ordinal the context lives on, fixed-base window width, and bytes of HBM its tables occupy. */
int eth_kzg_b200_context_device(const DASContext *ctx);
int eth_kzg_b200_context_window(const DASContext *ctx);
uint64_t eth_kzg_b200_context_table_bytes(const DASContext *ctx);
/* window width of the SRS (commitment / proof) tables; how many devices the context spans (EKZG_DEVICES) and the CUDA
 * ordinal of the i-th of them (-1 if out of range).  The three getters above report the first device. */
int eth_kzg_b200_context_srs_window(const DASContext *ctx);
int eth_kzg_b200_context_device_count(const DASContext *ctx);
int eth_kzg_b200_context_device_at(const DASContext *ctx, int i);
/* Measured issue rate (multiply-adds per second) of carry-chained IMAD.WIDE.U32 on the context's first device: the
 * roofline denominator of the point-arithmetic kernels, measured in-process (about 30 ms).  0 on error. */
double eth_kzg_b200_probe_imad_wide(const DASContext *ctx);
/* how a batch of n items is cut over `parts` devices: device i works on items [*lo, *lo + *cnt) -- whole groups of 32
 * (one G1-NTT work unit is 32 blobs wide), sizes differing by at most one group.  Host-only helper. */
void eth_kzg_b200_debug_shard_bounds(uint64_t n, uint64_t parts, uint64_t i, uint64_t *lo, uint64_t *cnt);
/* kernels launched by this library in this process so far (launch accounting in benchmarks) */
uint64_t eth_kzg_b200_kernel_launch_count(void);


/* Per-stage device timing of the FK20 pipeline (CUDA events on the launching stream), for benchmarks.
 * Stages: 0 blob->coefficients/cells, 1 Toeplitz scalars, 2 fixed-base MSMs, 3 G1 NTTs, 4 compress.
 * collect() adds the elapsed milliseconds of all finished batches to ms_out[5] and returns their count.
 * Single-threaded use only. */
void eth_kzg_b200_set_profiling(const DASContext *ctx, bool on);
int eth_kzg_b200_collect_stage_times(const DASContext *ctx, double *ms_out);

/* Test hook: FK20 intermediates of one blob (plain scalars [128][64][8 x u32 LE], 128 compressed MSM
 * outputs in natural order, 64 compressed h commitments).  Synchronous. */
CResult eth_kzg_b200_debug_fk20_stages(const DASContext *ctx, const uint8_t *blob, uint32_t *out_scalars, uint8_t *out_msm,
                                       uint8_t *out_h);
/* Test hook: the 128 points of one blob after the first `phases` (0..14) G1-NTT phases, compressed, in storage order. */
CResult eth_kzg_b200_debug_g1_ntt_prefix(const DASContext *ctx, const uint8_t *blob, int phases, uint8_t *out128x48);

/* Test hook (host only): prod_i e(P_i, Q_i) == 1.  g1_xy: 96 B per point (x then y, plain little-endian 64-bit limbs,
 * all zero = identity); g2_sel[i]: 0 [1]_2, 1 [tau]_2, 2 [tau^64]_2, +3 for the negated point.  Returns 1/0. */
int eth_kzg_b200_debug_pairing_check(int n, const uint8_t *g1_xy, const int *g2_sel);
/* Test hook (host only): the pairing's sparse line product and cyclotomic squaring against its general Fp12 routines; 1 = agree. */
int eth_kzg_b200_debug_pairing_selftest(void);
/* Test hooks of the setup loader (host only, no GPU): the JSON parser (point counts, first G1 / last G2 point as bytes), the G2
 * decompression (out24 = x.c0, x.c1, y.c0, y.c1 as plain little-endian 64-bit limbs; 0 ok, 1 malformed, 2 off the curve,
 * 3 outside the subgroup, 4 infinity) and the whole G2 side of a setup (65 points). */
CResult eth_kzg_b200_debug_parse_trusted_setup_json(const char *json, uint64_t json_len, uint64_t *n_g1, uint64_t *n_g2,
                                                    uint8_t *first_g1_48, uint8_t *last_g2_96);
int eth_kzg_b200_debug_g2_decompress(const uint8_t *in96, uint64_t *out24);
CResult eth_kzg_b200_debug_g2_keys(const uint8_t *g2_65x96, int count, bool subgroup_check);

/* Test hook (host only): SHA-256 of data[0..n) through the library's transcript hasher (x86 SHA extensions when
 * present), fed as two updates split at `split`; force_portable != 0 runs the portable C block function instead. */
void eth_kzg_b200_debug_sha256(const uint8_t *data, uint64_t n, uint64_t split, int force_portable, uint8_t out[32]);

#ifdef __cplusplus
}
#endif
#endif /* C_ETH_KZG_B200_H */
