// Device-side data layout shared by the kernels (kzg_kernels.cu) and the host runtime (kzg_runtime.cu).
#pragma once
#include <cuda_runtime.h>
#include "g1_mul.cuh"
#include "msm_table.cuh"

namespace ekzg {

constexpr int N_BLOB = 4096;         // FIELD_ELEMENTS_PER_BLOB       (crates/serialization/src/constants.rs)
constexpr int N_EXT = 8192;          // FIELD_ELEMENTS_PER_EXT_BLOB
constexpr int CELL_ELEMS = 64;       // FIELD_ELEMENTS_PER_CELL
constexpr int N_CELLS = 128;         // CELLS_PER_EXT_BLOB
constexpr int BYTES_PER_BLOB = 131072;
constexpr int BYTES_PER_CELL = 2048;
constexpr int BYTES_PER_G1 = 48;
constexpr size_t CELLS_PER_BLOB = (size_t)N_EXT * 32;              // bytes of the 128 cells of a blob
constexpr size_t PROOFS_PER_BLOB = (size_t)N_CELLS * BYTES_PER_G1; // bytes of its 128 proofs
constexpr int FK20_POINTS = 64;      // points per fixed-base MSM  (fk20/prover.rs:95-104)
constexpr int FK20_MSMS = 128;       // MSMs per blob = circulant domain size (fk20/batch_toeplitz.rs:113)

// Read-only tables, built once per device at context creation.  All Fr/Fp values in Montgomery form.
struct DevTables {
    const Fr* tw4096;        // omega_4096^i,  i < 2048
    const Fr* tw4096_inv;    // omega_4096^-i, i < 2048
    const Fr* tw8192;        // omega_8192^i,  i < 4096   (coset shift of the odd half of the 8192-NTT, also the 8192 twiddles)
    const Fr* tw8192_inv;    // omega_8192^-i, i < 4096
    const Fr* tw128;         // omega_128^i,   i < 64
    const Fr* tw64_inv;      // omega_64^-i,   i < 32     (verifier: 64-point coset IFFT)
    // FK20 fixed-base tables: entry (j, k, t, m) = (m+1) * 2^(t*w) * F_k[j], affine.
    // F_k = NTT_128^{G1}(V_k || O^64)  (fk20/batch_toeplitz.rs:49-58); the reference's table holds only
    // the t = 0 slice and pays w doublings per window at MSM time (fixed_base_msm_window.rs:154-165);
    // here every window has its own slice, so an MSM is additions only.
    MsmTable fk20;                     // base point i = j*64 + k  ->  F_k[j]
    // Same construction over the 4096 monomial SRS points, for commitments and single-point proofs
    // (reference: g1_lincomb -> blst Pippenger, bls12_381/src/lincomb.rs:7-30; fixed bases make it additions only).
    MsmTable srs;
    const G1Affine* srs_g1;            // g1_monomial[4096]
    const G1Affine* srs_g1_lagrange;   // g1_lagrange[4096] in the JSON's (bit-reversed) order
};

}  // namespace ekzg
