// sm_100a kernels of erasure recovery (recover_cells_and_kzg_proofs: cells -> polynomial coefficients).
//   reference: crates/eip7594/src/recovery.rs:22-66, kzg_multi_open/src/fk20/cosets.rs:141-198,
//              crates/cryptography/erasure_codes/src/reed_solomon.rs:220-262,332-384 (SURVEY.md A.7).
// What changes against the reference's data flow:
//  * Z(X) = Z0(X^64) vanishes on whole cosets, so its 8192 evaluations (and its 8192 coset evaluations) take only
//    128 distinct values Z0(w128^m) / Z0(7^64 w128^m): two 128-point evaluations and 128 inversions per blob replace two
//    8192-point transforms and an 8192-element batch inversion.
//  * every 8192-point transform is a decimation-in-frequency pass whose first stage is fused into the load, leaving two
//    independent 4096-point transforms that each fit one SM's shared memory (grid = blobs x 2); the bit reversals between
//    transforms are gathers on the 32-byte elements of the next load.
#include "kzg_kernels.h"
#include "fr_ntt.cuh"

namespace ekzg {

__device__ __forceinline__ int rbits(int x, int bits) { return (int)(__brev((unsigned)x) >> (32 - bits)); }

// omega_128^m for any m in [0,128) from the 64-entry table
__device__ __forceinline__ Fr omega128(const DevTables& T, int m) {
    Fr w = ld_vec(&T.tw128[m & 63]);
    if (m & 64) fe_neg(w, w);
    return w;
}

// R0: per blob, from the presence map: Z0 coefficients -> ze[m] = Z0(w^m), czinv[m] = 1 / Z0(7^64 w^m)
//     (reed_solomon.rs:220-262 construct_vanishing_poly_from_block_erasures + :343,:353-358)
__global__ void __launch_bounds__(128)
k_recover_prep(const int16_t* __restrict__ slotmap, Fr* __restrict__ ze, Fr* __restrict__ czinv, DevTables T, Fr gen64) {
    __shared__ Fr z0[2][130];
    __shared__ int missing[128];
    __shared__ int nmiss;
    const int b = blockIdx.x, m = threadIdx.x;
    if (m == 0) {
        int c = 0;
        for (int i = 0; i < 128; i++)
            if (slotmap[b * 128 + i] < 0) missing[c++] = i;
        nmiss = c;
    }
    Fr v;
    fe_set_zero(v);
    z0[0][m] = v;
    z0[1][m] = v;
    if (m < 2) { z0[0][128 + m] = v; z0[1][128 + m] = v; }
    __syncthreads();
    if (m == 0) fe_set_one(z0[0][0]);
    __syncthreads();
    int cur = 0;
    const int n = nmiss;
    for (int s = 0; s < n; s++) {  // multiply by (X - rho): new[i] = old[i-1] - rho*old[i]
        Fr rho = omega128(T, missing[s]);
        if (m <= s + 1) {
            Fr lo = z0[cur][m], t;
            fe_mul(t, rho, lo);
            Fr up;
            if (m >= 1) up = z0[cur][m - 1]; else fe_set_zero(up);
            fe_sub(t, up, t);
            z0[cur ^ 1][m] = t;
        }
        __syncthreads();
        cur ^= 1;
    }
    // Horner at x = w^m and at x = 7^64 w^m; degree n <= 128 is impossible (>= 64 present), n <= 64
    Fr x = omega128(T, m), xc;
    fe_mul(xc, x, gen64);
    Fr a, c;
    fe_set_zero(a);
    fe_set_zero(c);
    for (int i = n; i >= 0; i--) {
        Fr co = z0[cur][i];
        fe_mul(a, a, x); fe_add(a, a, co);
        fe_mul(c, c, xc); fe_add(c, c, co);
    }
    st_vec(&ze[b * 128 + m], a);
    Fr ci;
    fr_inv(ci, c);  // never zero: the coset 7*<w> contains no root of Z (reed_solomon.rs:355-357)
    st_vec(&czinv[b * 128 + m], ci);
}

constexpr int RN_THREADS = 1024;

// R1..R3: one half of an 8192-point DIF transform per CTA (blockIdx.y = half).
//  MODE 1: x[p] = E'[p] * ze[p % 128], E' scattered from the cells; inverse transform -> bufA (bit-reversed order)
//  MODE 2: x[i] = bufA[rev13(i)] * 7^i / 8192; forward transform; out = value * czinv[rev13(q) % 128] -> bufB (bit-reversed)
//  MODE 3: x[p] = bufB[rev13(p)]; inverse transform; c'[idx] = value * 7^-idx / 8192 at idx = rev13(q):
//          idx >= 4096 must be zero (status |= 4 otherwise), idx < 4096 -> coeffs[b][idx]
//  The cells of MODE 1 lie in 128-slot rows (blob b's cell of slot s at cells[b][s]) or, PACKED, as the caller concatenated
//  them: blob b's cell of slot s at cells[cell_off[b] + s].
template <int MODE, bool PACKED>
__device__ __forceinline__ void
recover_ntt(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ cell_off, const int16_t* __restrict__ slotmap,
            const Fr* __restrict__ ze, const Fr* __restrict__ czinv, const Fr* __restrict__ src, Fr* __restrict__ dst,
            Fr* __restrict__ coeffs, uint32_t* __restrict__ status, const Fr* __restrict__ shift, const DevTables& T) {
    extern __shared__ uint32_t sm[];
    const int b = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
    const Fr r2 = fe_const_r2<FrParams>();
    const Fr* tw_first = (MODE == 2) ? T.tw8192 : T.tw8192_inv;
    const uint8_t* row = (MODE == 1) ? cells + (PACKED ? (size_t)cell_off[b] : (size_t)b * N_CELLS) * BYTES_PER_CELL : nullptr;
    bool bad = false;
    for (int i = tid; i < N_BLOB; i += RN_THREADS) {
        Fr x[2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int p = i + u * N_BLOB;
            if (MODE == 1) {
                const int mpos = p & 127, a = p >> 7;
                const int slot = slotmap[b * 128 + mpos];
                if (slot < 0) {
                    fe_set_zero(x[u]);
                } else {
                    Fr e = fr_load_be(row + (size_t)slot * BYTES_PER_CELL + 32 * rbits(a, 6));
                    bad |= fe_plain_ge_mod(e);
                    fe_mul(e, e, r2);
                    Fr z = ld_vec(&ze[b * 128 + mpos]);
                    fe_mul(x[u], e, z);
                }
            } else if (MODE == 2) {
                Fr d = ld_vec(&src[(size_t)b * N_EXT + rbits(p, 13)]);
                Fr s = ld_vec(&shift[p]);
                fe_mul(x[u], d, s);
            } else {
                x[u] = ld_vec(&src[(size_t)b * N_EXT + rbits(p, 13)]);
            }
        }
        Fr v;
        if (h == 0) {
            fe_add(v, x[0], x[1]);
        } else {
            fe_sub(v, x[0], x[1]);
            Fr w = ld_vec(&tw_first[i]);
            fe_mul(v, v, w);
        }
        smem_st(sm, N_BLOB, i, v);
    }
    if (MODE == 1 && bad) atomicOr(&status[b], 1u);
    __syncthreads();
    ntt_dif_shared<12>(sm, N_BLOB, 1, (MODE == 2) ? T.tw4096 : T.tw4096_inv, tid, RN_THREADS);
    for (int p = tid; p < N_BLOB; p += RN_THREADS) {
        const int q = h * N_BLOB + p;
        Fr v = smem_ld(sm, N_BLOB, p);
        if (MODE == 1) {
            st_vec(&dst[(size_t)b * N_EXT + q], v);
        } else if (MODE == 2) {
            const int idx = 2 * rbits(p, 12) + h;  // rev13(q)
            Fr zi = ld_vec(&czinv[b * 128 + (idx & 127)]);
            fe_mul(v, v, zi);
            st_vec(&dst[(size_t)b * N_EXT + q], v);
        } else {
            const int idx = 2 * rbits(p, 12) + h;
            Fr s = ld_vec(&shift[idx]);
            fe_mul(v, v, s);
            if (idx >= N_BLOB) {
                if (!fe_is_zero(v)) atomicOr(&status[b], 4u);
            } else {
                st_vec(&coeffs[(size_t)b * N_BLOB + idx], v);
            }
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(RN_THREADS, 1)
k_recover_ntt(const uint8_t* __restrict__ cells, const int16_t* __restrict__ slotmap, const Fr* __restrict__ ze, const Fr* __restrict__ czinv,
              const Fr* __restrict__ src, Fr* __restrict__ dst, Fr* __restrict__ coeffs, uint32_t* __restrict__ status,
              const Fr* __restrict__ shift, DevTables T) {
    recover_ntt<MODE, false>(cells, nullptr, slotmap, ze, czinv, src, dst, coeffs, status, shift, T);
}

// R1 on packed cells: one H2D copy brings a run of blobs' cells up as the caller laid them out, with no re-layout on the host
__global__ void __launch_bounds__(RN_THREADS, 1)
k_recover_ntt_packed(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ cell_off, const int16_t* __restrict__ slotmap,
                     const Fr* __restrict__ ze, Fr* __restrict__ dst, uint32_t* __restrict__ status, DevTables T) {
    recover_ntt<1, true>(cells, cell_off, slotmap, ze, nullptr, nullptr, dst, nullptr, status, nullptr, T);
}


cudaError_t recover_kernels_init() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_recover_ntt<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_recover_ntt<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_recover_ntt<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_recover_ntt_packed, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4);
}

// cells: [B][128 slots][2048] wire bytes (slot = rank of the cell in the caller's list), or with cell_off (packed) blob b's
// cells from cells + cell_off[b] * 2048 on; slotmap: [B][128] slot of domain position m = rev7(cell index) or -1.
// bufA/bufB: [B][8192] Fr scratch.  Result: coeffs [B][4096], status bits 1 (cell scalar not canonical) / 4 (recovered
// polynomial has degree >= 4096).
cudaError_t launch_recover_coeffs(const uint8_t* cells, const int16_t* slotmap, Fr* ze, Fr* czinv, Fr* bufA, Fr* bufB, Fr* coeffs,
                                  uint32_t* status, const DevTables& T, const Fr* shift_fwd, const Fr* shift_inv, const uint32_t* gen64_mont,
                                  int B, cudaStream_t st, const uint32_t* cell_off) {
    Fr g;
    for (int i = 0; i < 8; i++) g.v[i] = gen64_mont[i];
    k_recover_prep<<<B, 128, 0, st>>>(slotmap, ze, czinv, T, g);
    EKZG_LAUNCH_CHECK();
    const size_t smem = 8 * N_BLOB * 4;
    if (cell_off) k_recover_ntt_packed<<<dim3(B, 2), RN_THREADS, smem, st>>>(cells, cell_off, slotmap, ze, bufA, status, T);
    else k_recover_ntt<1><<<dim3(B, 2), RN_THREADS, smem, st>>>(cells, slotmap, ze, czinv, nullptr, bufA, nullptr, status, nullptr, T);
    EKZG_LAUNCH_CHECK();
    k_recover_ntt<2><<<dim3(B, 2), RN_THREADS, smem, st>>>(nullptr, slotmap, ze, czinv, bufA, bufB, nullptr, status, shift_fwd, T);
    EKZG_LAUNCH_CHECK();
    k_recover_ntt<3><<<dim3(B, 2), RN_THREADS, smem, st>>>(nullptr, slotmap, ze, czinv, bufB, nullptr, coeffs, status, shift_inv, T);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

}  // namespace ekzg
