// sm_100a kernels of the verifiers: verify_cell_kzg_proof_batch (universal FK20 verification equation) and the EIP-4844
// verify_* functions.  Everything up to the two G1 points of the final pairing check runs here; the pairing itself is a
// single latency-bound computation on the host (host_pairing.cpp).
//   reference: kzg_multi_open/src/fk20/verifier.rs:129-260, 333-384; kzg_single_open/src/verifier.rs:33-108;
//              crates/serialization/src/lib.rs:69-126.
// The reference's three variable-base MSMs (blst Pippenger, N up to 16384) become one scalar multiplication per thread
// followed by a tree reduction: the bases change with every call, so there is nothing to precompute, and at N x 255-bit the
// whole job is ~1e8 field multiplications = a few milliseconds of one B200.
#include "kzg_kernels.h"
#include "fr_ntt.cuh"

namespace ekzg {

__device__ __forceinline__ int vbits(int x, int bits) { return (int)(__brev((unsigned)x) >> (32 - bits)); }

__device__ __forceinline__ Fr fr_from_hash_dev(const uint8_t* p) {
    Fr x;
#pragma unroll
    for (int l = 0; l < 8; l++) {
        const uint8_t* q = p + 4 * (7 - l);
        x.v[l] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
    }
    fe_final_sub<FrParams>(x.v);
    fe_final_sub<FrParams>(x.v);
    fe_to_mont(x, x);
    return x;
}

__device__ __forceinline__ void store_plain(uint32_t* dst, const Fr& mont) {
    Fr p;
    fe_from_mont(p, mont);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    d4[0] = make_uint4(p.v[0], p.v[1], p.v[2], p.v[3]);
    d4[1] = make_uint4(p.v[4], p.v[5], p.v[6], p.v[7]);
}

// rpow[k] = r^k, r = SHA-256 digest reduced mod r  (fk20/verifier.rs:333-343 compute_powers)
__global__ void k_powers_from_hash(const uint8_t* __restrict__ hash, Fr* __restrict__ rpow, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Fr b = fr_from_hash_dev(hash), acc;
    fe_set_one(acc);
    for (int e = k; e; e >>= 1) {
        if (e & 1) fe_mul(acc, acc, b);
        fe_sqr(b, b);
    }
    st_vec(&rpow[k], acc);
}

// per opening k: s1 = rho_k, s2 = rho_k * h_col^64 with h_col^64 = w128^rev7(col)  (verifier.rs:188-201), plain integers
__global__ void k_cell_verify_scalars(const Fr* __restrict__ rpow, const uint32_t* __restrict__ col, uint32_t* __restrict__ s1,
                                      uint32_t* __restrict__ s2, DevTables T, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Fr rho = ld_vec(&rpow[k]);
    int m = vbits((int)col[k], 7);
    Fr w = ld_vec(&T.tw128[m & 63]);
    if (m & 64) fe_neg(w, w);
    Fr t;
    fe_mul(t, rho, w);
    store_plain(s1 + (size_t)k * 8, rho);
    store_plain(s2 + (size_t)k * 8, t);
}

// weights[i] = sum_{k: row_k == i} rho_k  (verifier.rs:216-219), plain integers.  One CTA per row.
__global__ void __launch_bounds__(128)
k_commitment_weights(const Fr* __restrict__ rpow, const uint32_t* __restrict__ row, uint32_t* __restrict__ wout, int n, int m) {
    __shared__ Fr sm[128];
    const int i = blockIdx.x;
    Fr acc;
    fe_set_zero(acc);
    for (int k = threadIdx.x; k < n; k += 128)
        if ((int)row[k] == i) {
            Fr r = ld_vec(&rpow[k]);
            fe_add(acc, acc, r);
        }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s >= 1; s >>= 1) {
        if (threadIdx.x < s) {
            Fr a = sm[threadIdx.x], b = sm[threadIdx.x + s];
            fe_add(a, a, b);
            sm[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) store_plain(wout + (size_t)i * 8, sm[0]);
}

// The second random-linear-combination MSM of the verification equation, sum_k rho_k h_k^64 pi_k (verifier.rs:188-201),
// shares its points with the first one and its extra factor h_k^64 = omega_128^rev7(col_k) only depends on the cell
// index.  So: colsum[c] = sum_{k: col_k == c} rho_k pi_k (one CTA per column over the products the first MSM already
// made), then  sum_k rho_k pi_k = sum_c colsum[c]  and  sum_k rho_k h_k^64 pi_k = sum_c omega^rev7(c) colsum[c]
// -- 128 multiplications by FIXED roots of unity (the op-list ladder of the G1 NTT) instead of N variable ones.
__constant__ uint16_t c_verify_twiddle_ops[128][MULOPS_STRIDE] =
#include "twiddle_ops.inc"
    ;

__global__ void __launch_bounds__(128)
k_column_sums(const G1Jac* __restrict__ prods, const uint32_t* __restrict__ col, G1Jac* __restrict__ colsum, int n) {
    __shared__ G1Jac sm[128];
    const int c = blockIdx.x;
    G1Jac acc;
    jac_set_inf(acc);
    for (int k = threadIdx.x; k < n; k += 128)
        if ((int)col[k] == c) {
            G1Jac q = ld_vec(&prods[k]);
            jac_add(acc, q);
        }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s >= 1; s >>= 1) {
        if (threadIdx.x < s) {
            G1Jac a = sm[threadIdx.x];
            jac_add(a, sm[threadIdx.x + s]);
            sm[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) st_vec(&colsum[c], sm[0]);
}

// weighted[c] = omega_128^rev7(c) * colsum[c]
__global__ void __launch_bounds__(32)
k_column_twiddle(const G1Jac* __restrict__ colsum, G1Jac* __restrict__ weighted) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= N_CELLS) return;
    G1Jac q = ld_vec(&colsum[c]);
    const int e = vbits(c, 7);
    if (e != 0 && !jac_is_inf(q)) jac_mul_ops(q, q, c_verify_twiddle_ops[e]);
    st_vec(&weighted[c], q);
}

// out[i] = scalar_i * P_i  (identity points / zero scalars give the identity, like lincomb.rs:13-27 filters them)
__global__ void __launch_bounds__(64)
k_scalar_mul(const G1Affine* __restrict__ pts, const uint32_t* __restrict__ scalars, G1Jac* __restrict__ out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    G1Affine a = ld_vec(&pts[i]);
    G1Jac p, r;
    jac_from_affine(p, a);
    uint32_t k[8];
    const uint4* s4 = reinterpret_cast<const uint4*>(scalars + (size_t)i * 8);
    uint4 lo = s4[0], hi = s4[1];
    k[0] = lo.x; k[1] = lo.y; k[2] = lo.z; k[3] = lo.w; k[4] = hi.x; k[5] = hi.y; k[6] = hi.z; k[7] = hi.w;
    if (g1a_is_inf(a)) jac_set_inf(r);
    else jac_mul_fr_glv(r, p, k);   // scalars are canonical Fr values (< r): GLV halves the doublings
    st_vec(&out[i], r);
}

// the same with the two GLV halves of every multiplication on two lanes (small batches: the call is bound by the latency of ONE
// ladder, and half the additions of a ladder are the other half's).  Thread 2i + h: half h of item i; the pair meets through
// shared memory.
__global__ void __launch_bounds__(64)
k_scalar_mul_split(const G1Affine* __restrict__ pts, const uint32_t* __restrict__ scalars, G1Jac* __restrict__ out, int n) {
    __shared__ G1Jac part[32];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = t >> 1, h = t & 1;
    const bool live = i < n;
    G1Jac r;
    jac_set_inf(r);
    if (live) {
        G1Affine a = ld_vec(&pts[i]);
        if (!g1a_is_inf(a)) {
            G1Jac p;
            jac_from_affine(p, a);
            uint32_t k[8];
            const uint4* s4 = reinterpret_cast<const uint4*>(scalars + (size_t)i * 8);
            uint4 lo = s4[0], hi = s4[1];
            k[0] = lo.x; k[1] = lo.y; k[2] = lo.z; k[3] = lo.w; k[4] = hi.x; k[5] = hi.y; k[6] = hi.z; k[7] = hi.w;
            int8_t d[66];
            glv_split_digits(d, k);
            if (h) jac_endo(p, p);
            jac_mul_half16(r, p, d + 33 * h);
        }
    }
    if (h) part[threadIdx.x >> 1] = r;
    __syncthreads();
    if (live && !h) {
        jac_add(r, part[threadIdx.x >> 1]);
        st_vec(&out[i], r);
    }
}

// partial[blockIdx] = sum of in[i] for i = blockIdx*blockDim + tid, strided by the whole grid; block tree in shared memory
__global__ void __launch_bounds__(128)
k_reduce_points(const G1Jac* __restrict__ in, G1Jac* __restrict__ partial, int n) {
    __shared__ G1Jac sm[128];
    G1Jac acc;
    jac_set_inf(acc);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        G1Jac q = ld_vec(&in[i]);
        jac_add(acc, q);
    }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s >= 1; s >>= 1) {
        if (threadIdx.x < s) {
            G1Jac a = sm[threadIdx.x];
            jac_add(a, sm[threadIdx.x + s]);
            sm[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) st_vec(&partial[blockIdx.x], sm[0]);
}

// Interpolation polynomial of one cell, scaled: interp[k][t] = rho_k * INTT_64(BRP(cell_k))[t] * h_col^-t
// (verifier.rs:348-384 compute_sum_interpolation_poly; coset_ifft_scalars domain.rs:214-223).  64 threads per cell.
constexpr int VI_CELLS = 2;
__global__ void __launch_bounds__(64 * VI_CELLS)
k_cell_interp(const uint8_t* __restrict__ cells, const uint32_t* __restrict__ col, const Fr* __restrict__ rpow, Fr* __restrict__ interp,
              uint32_t* __restrict__ status, DevTables T, int n) {
    __shared__ uint32_t sm[8 * 64 * VI_CELLS];
    constexpr int STRIDE = 64 * VI_CELLS;
    const int tid = threadIdx.x, q = tid >> 6, t = tid & 63;
    const int k = blockIdx.x * VI_CELLS + q;
    const bool active = k < n;
    Fr e;
    fe_set_zero(e);
    if (active) {
        e = fr_load_be(cells + (size_t)k * BYTES_PER_CELL + 32 * t);
        if (fe_plain_ge_mod(e)) atomicOr(status, 1u);
        fe_to_mont(e, e);
    }
    smem_st(sm, STRIDE, tid, e);
    __syncthreads();
    // the cell is in bit-reversed order: a DIT pass on the array as it lies is INTT_64(BRP(cell))
    ntt_dit_shared<6>(sm, STRIDE, VI_CELLS, T.tw64_inv, tid, 64 * VI_CELLS);
    if (!active) return;
    Fr v = smem_ld(sm, STRIDE, tid);
    const int m = vbits((int)col[k], 7);          // h_col = w8192^m
    const int ex = (m * t) & 8191;                // h_col^-t = w8192^-(m t)
    Fr w = ld_vec(&T.tw8192_inv[ex & 4095]);
    if (ex & 4096) fe_neg(w, w);
    Fr rho = ld_vec(&rpow[k]);
    fe_mul(v, v, w);
    fe_mul(v, v, rho);
    fe_mul(v, v, fr_inv_64());
    st_vec(&interp[(size_t)k * 64 + t], v);
}

// sum over k of interp[k][t] -> plain integer scalar t (64 CTAs)
__global__ void __launch_bounds__(128)
k_interp_column_sum(const Fr* __restrict__ interp, uint32_t* __restrict__ out, int n) {
    __shared__ Fr sm[128];
    const int t = blockIdx.x;
    Fr acc;
    fe_set_zero(acc);
    for (int k = threadIdx.x; k < n; k += 128) {
        Fr v = ld_vec(&interp[(size_t)k * 64 + t]);
        fe_add(acc, acc, v);
    }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s >= 1; s >>= 1) {
        if (threadIdx.x < s) {
            Fr a = sm[threadIdx.x], b = sm[threadIdx.x + s];
            fe_add(a, a, b);
            sm[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) store_plain(out + (size_t)t * 8, sm[0]);
}

// Final G1 points of a pairing check, as plain affine coordinates for the host:
//   out[0] = a0 ;  out[1] = b0 - b1 + b2      (each term may be null = identity)
// layout per point: X, Y, Z of the Jacobian point (12 limbs each, Montgomery form, little-endian 32-bit) + 1 word identity flag
// = 37 words.  The normalisation (one inversion: ~0.4 ms for a lone device thread, ~25 us on the host) is left to the host, which
// works on the same Montgomery representation (R = 2^384 on both sides).
__global__ void k_pairing_inputs(const G1Jac* a0, const G1Jac* b0, const G1Jac* b1, const G1Jac* b2, uint32_t* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x > 1) return;   // two CTAs, one point each
    const int i = blockIdx.x;
    G1Jac pt;
    if (i == 0) {
        pt = ld_vec(a0);
    } else {
        jac_set_inf(pt);
        if (b0) { G1Jac q = ld_vec(b0); jac_add(pt, q); }
        if (b1) { G1Jac q = ld_vec(b1); jac_neg(q, q); jac_add(pt, q); }
        if (b2) { G1Jac q = ld_vec(b2); jac_add(pt, q); }
    }
    uint32_t* o = out + PAIRING_INPUT_WORDS * i;
    for (int l = 0; l < 12; l++) { o[l] = pt.x.v[l]; o[12 + l] = pt.y.v[l]; o[24 + l] = pt.z.v[l]; }
    o[36] = jac_is_inf(pt) ? 1u : 0u;
}

// EIP-4844 single / batched proof verification inputs (kzg_single_open/src/verifier.rs:33-108), rewritten so that only G1
// arithmetic is needed:  e(sum r^i (C_i - y_i G + z_i pi_i), -[1]_2) * e(sum r^i pi_i, [tau]_2) == 1.
// Per item i the four products  r^i * C_i,  (-r^i y_i) * G,  (r^i z_i) * pi_i  and  r^i * pi_i  are independent: this kernel only writes
// them down as (point, scalar) pairs, kind-major (pair kind*n + i), and the generic scalar-multiplication kernel runs all 4n at once
// (first version: one thread per item, four plain 255-bit ladders in a row -- 9 ms for a single proof).  The left sum is then the
// sum of the first 3n products, the right sum that of the last n.
__global__ void __launch_bounds__(64)
k_kzg_verify_pairs(const G1Affine* __restrict__ commitments, const G1Affine* __restrict__ proofs, const Fr* __restrict__ z,
                   const Fr* __restrict__ y, const Fr* __restrict__ rpow, G1Affine* __restrict__ pts, uint32_t* __restrict__ scalars, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Fr rho = ld_vec(&rpow[i]), zi = ld_vec(&z[i]), yi = ld_vec(&y[i]);
    Fr rz, ry, p;
    fe_mul(rz, rho, zi);
    fe_mul(ry, rho, yi);
    fe_neg(ry, ry);
    const G1Affine c = ld_vec(&commitments[i]), pi = ld_vec(&proofs[i]);
    G1Affine g;
    for (int l = 0; l < 12; l++) { g.x.v[l] = FpParams::gen_x(l); g.y.v[l] = FpParams::gen_y(l); }
    st_vec(&pts[i], c);
    st_vec(&pts[(size_t)n + i], g);
    st_vec(&pts[(size_t)2 * n + i], pi);
    st_vec(&pts[(size_t)3 * n + i], pi);
    fe_from_mont(p, rho);
    for (int l = 0; l < 8; l++) { scalars[(size_t)i * 8 + l] = p.v[l]; scalars[((size_t)3 * n + i) * 8 + l] = p.v[l]; }
    fe_from_mont(p, ry);
    for (int l = 0; l < 8; l++) scalars[((size_t)n + i) * 8 + l] = p.v[l];
    fe_from_mont(p, rz);
    for (int l = 0; l < 8; l++) scalars[((size_t)2 * n + i) * 8 + l] = p.v[l];
}

// y_i = p_i(z_i) on the monomial coefficients (eip4844/src/verifier.rs:83,120 `.eval(&z)`): a warp per blob, lane l runs Horner over
// coefficients [128 l, 128 l + 128), then the 32 partial values are combined with powers of z^128 (one thread per blob took 0.8 ms
// for its 4096 dependent multiplications, which a single-proof call cannot hide)
__global__ void __launch_bounds__(32)
k_poly_eval(const Fr* __restrict__ coeffs, const Fr* __restrict__ z_in, Fr* __restrict__ y_out, uint8_t* __restrict__ y_be, int B) {
    __shared__ Fr part[32];
    const int b = blockIdx.x, lane = threadIdx.x;
    if (b >= B) return;
    const Fr* c = coeffs + (size_t)b * N_BLOB + (size_t)lane * 128;
    const Fr z = ld_vec(&z_in[b]);
    Fr t;
    fe_set_zero(t);
    for (int i = 127; i >= 0; i--) {
        Fr ci = ld_vec(&c[i]);
        fe_mul(t, t, z);
        fe_add(t, t, ci);
    }
    part[lane] = t;
    __syncwarp();
    if (lane == 0) {
        Fr z128 = z;
        for (int i = 0; i < 7; i++) fe_sqr(z128, z128);
        Fr acc = part[31];
        for (int l = 30; l >= 0; l--) {
            fe_mul(acc, acc, z128);
            fe_add(acc, acc, part[l]);
        }
        st_vec(&y_out[b], acc);
        if (y_be) {
            Fr p;
            fe_from_mont(p, acc);
            fr_store_be(y_be + (size_t)b * 32, p);
        }
    }
}

// Montgomery Fr -> 32 big-endian bytes (transcript of verify_blob_kzg_proof_batch needs z and y on the wire format)
__global__ void k_fr_to_be(const Fr* __restrict__ in, uint8_t* __restrict__ out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr p = ld_vec(&in[i]);
    fe_from_mont(p, p);
    fr_store_be(out + (size_t)i * 32, p);
}

// ------------------------------------------------------------------------------------------------
// Verdicts per group of openings / per blob (verify_cell_kzg_proof_batch_groups, verify_blob_kzg_proof_batch_items).
// A malformed item is masked out of every sum: its power of r becomes 0 and its points the identity, so it adds nothing
// and the other items keep their powers.  Then, only when the masked aggregate check fails, the sums are formed again per
// group and checked group by group on the host.
// ------------------------------------------------------------------------------------------------

// bad[k] = 1 when a field element of cell k is not canonical (k_cell_interp ORs one flag for the whole batch).  A warp per cell.
__global__ void __launch_bounds__(128)
k_cell_canonical(const uint8_t* __restrict__ cells, uint32_t* __restrict__ bad, int n) {
    const int k = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= n) return;   // (the whole warp)
    const uint8_t* c = cells + (size_t)k * BYTES_PER_CELL;
    const bool b = fe_plain_ge_mod(fr_load_be(c + 32 * lane)) || fe_plain_ge_mod(fr_load_be(c + 32 * (lane + 32)));
    const bool any = __any_sync(0xffffffffu, b);
    if (lane == 0) bad[k] = any ? 1u : 0u;
}

// Opening k is malformed when its proof, the commitment of its row or its cell is, or its cell index is >= 128:
// flag[k] = 1, rho_k = 0, its proof point becomes the identity and its index 0 (so that no later kernel reads out of
// bounds).  Threads below m set the invalid commitments to the identity.
__global__ void k_mask_openings(Fr* __restrict__ rpow, const uint32_t* __restrict__ stp, const uint32_t* __restrict__ stc,
                                const uint32_t* __restrict__ row, uint32_t* __restrict__ col, const uint32_t* __restrict__ cell_bad,
                                G1Affine* __restrict__ a_p, G1Affine* __restrict__ a_c, uint32_t* __restrict__ flag, int n, int m) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    G1Affine id;
    g1a_set_inf(id);
    if (i < m && stc[i]) st_vec(&a_c[i], id);
    if (i >= n) return;
    const bool bad_col = col[i] >= (uint32_t)N_CELLS;
    const bool bad = stp[i] || stc[row[i]] || cell_bad[i] || bad_col;
    flag[i] = bad ? 1u : 0u;
    if (bad) {
        Fr z;
        fe_set_zero(z);
        st_vec(&rpow[i], z);
        st_vec(&a_p[i], id);
    }
    if (bad_col) col[i] = 0;
}

// EIP-4844 item i is malformed when its blob, commitment or proof is: flag[i] = 1, r^i = 0, both points the identity
__global__ void k_mask_items(Fr* __restrict__ rpow, const uint32_t* __restrict__ stb, const uint32_t* __restrict__ stc,
                             const uint32_t* __restrict__ stp, G1Affine* __restrict__ a_c, G1Affine* __restrict__ a_p,
                             uint32_t* __restrict__ flag, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool bad = stb[i] || stc[i] || stp[i];
    flag[i] = bad ? 1u : 0u;
    if (bad) {
        Fr z;
        fe_set_zero(z);
        st_vec(&rpow[i], z);
        G1Affine id;
        g1a_set_inf(id);
        st_vec(&a_c[i], id);
        st_vec(&a_p[i], id);
    }
}

// out[k] = pts[idx[k]]  (the commitment of every opening, for a ladder per opening)
__global__ void k_gather_points(const G1Affine* __restrict__ pts, const uint32_t* __restrict__ idx, G1Affine* __restrict__ out, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    st_vec(&out[k], ld_vec(&pts[idx[k]]));
}

// Segmented point sums over a CSR layout: the items of group g are order[off[g] .. off[g + 1]).  For s = 0, 1, 2:
// sums[s * G + g] = sum of in_s[order[j]].  TEAM threads per group: a warp for a small group (four per CTA), the whole CTA
// for a large one; `groups[count]` lists the groups of this launch.
template <int TEAM>
__global__ void __launch_bounds__(128)
k_group_point_sums(const G1Jac* __restrict__ in0, const G1Jac* __restrict__ in1, const G1Jac* __restrict__ in2,
                   const uint32_t* __restrict__ order, const uint32_t* __restrict__ off, const uint32_t* __restrict__ groups, int count,
                   G1Jac* __restrict__ sums, int G) {
    __shared__ G1Jac sm[128];
    const int team = blockIdx.x * (128 / TEAM) + threadIdx.x / TEAM, lane = threadIdx.x % TEAM;
    const bool live = team < count;
    const int g = live ? (int)groups[team] : 0;
    const int lo = live ? (int)off[g] : 0, hi = live ? (int)off[g + 1] : 0;
#pragma unroll 1
    for (int s = 0; s < 3; s++) {
        const G1Jac* in = s == 0 ? in0 : (s == 1 ? in1 : in2);
        G1Jac acc;
        jac_set_inf(acc);
        for (int j = lo + lane; j < hi; j += TEAM) {
            G1Jac q = ld_vec(&in[order[j]]);
            jac_add(acc, q);
        }
        sm[threadIdx.x] = acc;
        __syncthreads();
        for (int w = TEAM / 2; w >= 1; w >>= 1) {
            if (lane < w) {
                G1Jac a = sm[threadIdx.x];
                jac_add(a, sm[threadIdx.x + w]);
                sm[threadIdx.x] = a;
            }
            __syncthreads();
        }
        if (live && lane == 0) st_vec(&sums[(size_t)s * G + g], sm[threadIdx.x]);
        __syncthreads();
    }
}

// out[(t * G + g) * 8] = sum over the items of group g of interp[k][t], as plain integers.  t-major ([64][G]): the layout
// in which the fixed-base MSM reads the scalars of G "blobs" (for G = 1 that of k_interp_column_sum).  A CTA per group,
// four lanes per coefficient.
__global__ void __launch_bounds__(256)
k_group_interp_sums(const Fr* __restrict__ interp, const uint32_t* __restrict__ order, const uint32_t* __restrict__ off,
                    uint32_t* __restrict__ out, int G) {
    __shared__ Fr sm[256];
    const int g = blockIdx.x, t = threadIdx.x & 63, q = threadIdx.x >> 6;
    Fr acc;
    fe_set_zero(acc);
    for (int j = (int)off[g] + q; j < (int)off[g + 1]; j += 4) {
        Fr v = ld_vec(&interp[(size_t)order[j] * 64 + t]);
        fe_add(acc, acc, v);
    }
    sm[threadIdx.x] = acc;
    __syncthreads();
    if (q != 0) return;
    for (int r = 1; r < 4; r++) {
        Fr b = sm[threadIdx.x + 64 * r];
        fe_add(acc, acc, b);
    }
    store_plain(out + ((size_t)t * G + g) * 8, acc);
}

// n pairing checks in the layout of k_pairing_inputs, one thread each: P_i = a[i], Q_i = b0[i] + b1[i] + b2[i], or
// b0[i] - b1[i] + b2[i] with sub_b1
__global__ void k_pairing_inputs_n(const G1Jac* __restrict__ a, const G1Jac* __restrict__ b0, const G1Jac* __restrict__ b1,
                                   const G1Jac* __restrict__ b2, bool sub_b1, uint32_t* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    G1Jac pt[2];
    pt[0] = ld_vec(&a[i]);
    pt[1] = ld_vec(&b0[i]);
    G1Jac q = ld_vec(&b1[i]);
    if (sub_b1) jac_neg(q, q);
    jac_add(pt[1], q);
    q = ld_vec(&b2[i]);
    jac_add(pt[1], q);
    for (int h = 0; h < 2; h++) {
        uint32_t* o = out + (size_t)PAIRING_INPUT_WORDS * (2 * i + h);
        for (int l = 0; l < 12; l++) { o[l] = pt[h].x.v[l]; o[12 + l] = pt[h].y.v[l]; o[24 + l] = pt[h].z.v[l]; }
        o[36] = jac_is_inf(pt[h]) ? 1u : 0u;
    }
}


cudaError_t launch_powers_from_hash(const uint8_t* hash, Fr* rpow, int n, cudaStream_t st) {
    k_powers_from_hash<<<(n + 127) / 128, 128, 0, st>>>(hash, rpow, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_cell_verify_scalars(const Fr* rpow, const uint32_t* col, uint32_t* s1, uint32_t* s2, const DevTables& T, int n, cudaStream_t st) {
    k_cell_verify_scalars<<<(n + 127) / 128, 128, 0, st>>>(rpow, col, s1, s2, T, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_commitment_weights(const Fr* rpow, const uint32_t* row, uint32_t* wout, int n, int m, cudaStream_t st) {
    k_commitment_weights<<<m, 128, 0, st>>>(rpow, row, wout, n, m);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
// colsum[128] and weighted[128] from the N products rho_k pi_k (see k_column_sums)
cudaError_t launch_column_sums(const G1Jac* prods, const uint32_t* col, G1Jac* colsum, G1Jac* weighted, int n, cudaStream_t st) {
    k_column_sums<<<N_CELLS, 128, 0, st>>>(prods, col, colsum, n);
    EKZG_LAUNCH_CHECK();
    k_column_twiddle<<<N_CELLS / 32, 32, 0, st>>>(colsum, weighted);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_scalar_mul(const G1Affine* pts, const uint32_t* scalars, G1Jac* out, int n, cudaStream_t st) {
    // up to 8192 items the machine has lanes to spare (2 x 8192 threads per pass, two passes at a time): split every
    // multiplication over two lanes; above that one lane per item keeps the passes to one wave
    if (n <= 8192) k_scalar_mul_split<<<(2 * n + 63) / 64, 64, 0, st>>>(pts, scalars, out, n);
    else k_scalar_mul<<<(n + 63) / 64, 64, 0, st>>>(pts, scalars, out, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
// sum of n points -> out[0]; scratch must hold 148 points
cudaError_t launch_sum_points(const G1Jac* in, int n, G1Jac* scratch, G1Jac* out, cudaStream_t st) {
    int blocks = (n + 127) / 128;
    if (blocks > 148) blocks = 148;
    if (blocks < 1) blocks = 1;
    k_reduce_points<<<blocks, 128, 0, st>>>(in, scratch, n);
    EKZG_LAUNCH_CHECK();
    k_reduce_points<<<1, 128, 0, st>>>(scratch, out, blocks);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_cell_interp(const uint8_t* cells, const uint32_t* col, const Fr* rpow, Fr* interp, uint32_t* status, const DevTables& T,
                               int n, cudaStream_t st) {
    k_cell_interp<<<(n + VI_CELLS - 1) / VI_CELLS, 64 * VI_CELLS, 0, st>>>(cells, col, rpow, interp, status, T, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_interp_column_sum(const Fr* interp, uint32_t* out, int n, cudaStream_t st) {
    k_interp_column_sum<<<64, 128, 0, st>>>(interp, out, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_pairing_inputs(const G1Jac* a0, const G1Jac* b0, const G1Jac* b1, const G1Jac* b2, uint32_t* out, cudaStream_t st) {
    k_pairing_inputs<<<2, 32, 0, st>>>(a0, b0, b1, b2, out);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_kzg_verify_pairs(const G1Affine* commitments, const G1Affine* proofs, const Fr* z, const Fr* y, const Fr* rpow, G1Affine* pts,
                                    uint32_t* scalars, int n, cudaStream_t st) {
    k_kzg_verify_pairs<<<(n + 63) / 64, 64, 0, st>>>(commitments, proofs, z, y, rpow, pts, scalars, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_poly_eval(const Fr* coeffs, const Fr* z, Fr* y, uint8_t* y_be, int B, cudaStream_t st) {
    k_poly_eval<<<B, 32, 0, st>>>(coeffs, z, y, y_be, B);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_fr_to_be(const Fr* in, uint8_t* out, int n, cudaStream_t st) {
    k_fr_to_be<<<(n + 127) / 128, 128, 0, st>>>(in, out, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_cell_canonical(const uint8_t* cells, uint32_t* bad, int n, cudaStream_t st) {
    k_cell_canonical<<<(n + 3) / 4, 128, 0, st>>>(cells, bad, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_mask_openings(Fr* rpow, const uint32_t* stp, const uint32_t* stc, const uint32_t* row, uint32_t* col, const uint32_t* cell_bad,
                                 G1Affine* a_p, G1Affine* a_c, uint32_t* flag, int n, int m, cudaStream_t st) {
    k_mask_openings<<<(std::max(n, m) + 127) / 128, 128, 0, st>>>(rpow, stp, stc, row, col, cell_bad, a_p, a_c, flag, n, m);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_mask_items(Fr* rpow, const uint32_t* stb, const uint32_t* stc, const uint32_t* stp, G1Affine* a_c, G1Affine* a_p, uint32_t* flag,
                              int n, cudaStream_t st) {
    k_mask_items<<<(n + 127) / 128, 128, 0, st>>>(rpow, stb, stc, stp, a_c, a_p, flag, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_gather_points(const G1Affine* pts, const uint32_t* idx, G1Affine* out, int n, cudaStream_t st) {
    k_gather_points<<<(n + 127) / 128, 128, 0, st>>>(pts, idx, out, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_group_point_sums(const G1Jac* in0, const G1Jac* in1, const G1Jac* in2, const uint32_t* order, const uint32_t* off,
                                    const uint32_t* small, int n_small, const uint32_t* large, int n_large, G1Jac* sums, int G, cudaStream_t st) {
    if (n_small) {
        k_group_point_sums<32><<<(n_small + 3) / 4, 128, 0, st>>>(in0, in1, in2, order, off, small, n_small, sums, G);
        EKZG_LAUNCH_CHECK();
    }
    if (n_large) {
        k_group_point_sums<128><<<n_large, 128, 0, st>>>(in0, in1, in2, order, off, large, n_large, sums, G);
        EKZG_LAUNCH_CHECK();
    }
    return cudaSuccess;
}
cudaError_t launch_group_interp_sums(const Fr* interp, const uint32_t* order, const uint32_t* off, uint32_t* out, int G, cudaStream_t st) {
    k_group_interp_sums<<<G, 256, 0, st>>>(interp, order, off, out, G);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}
cudaError_t launch_pairing_inputs_n(const G1Jac* a, const G1Jac* b0, const G1Jac* b1, const G1Jac* b2, bool sub_b1, uint32_t* out, int n,
                                    cudaStream_t st) {
    k_pairing_inputs_n<<<(n + 63) / 64, 64, 0, st>>>(a, b0, b1, b2, sub_b1, out, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

}  // namespace ekzg
