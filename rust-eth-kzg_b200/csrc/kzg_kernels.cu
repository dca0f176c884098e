// sm_100a kernels of the FK20 prover path (compute_cells_and_kzg_proofs) and the one-off table setup.
// Launch wrappers at the bottom; the host runtime (kzg_runtime.cu) only sees kzg_kernels.h.
//
// Batch layout (B blobs per launch, everything resident in HBM):
//   blobs   [B][131072]  bytes as on the wire
//   coeffs  [B][4096]    Fr, Montgomery form (monomial coefficients, A.1 of SURVEY.md)
//   cells   [B][8192*32] bytes as on the wire (cells 0..63 = the blob itself)
//   scalars [128][64][B] plain 256-bit integers: scalar k of MSM j of blob b (blob fastest, so a warp
//                        of 32 blobs working on the same MSM reads 1 KiB contiguous)
//   pts     [128][B]     G1Jac, position-major / blob fastest (same reason)
//   proofs  [B][128*48]  bytes as on the wire
#include "kzg_kernels.h"
#include "fr_ntt.cuh"
#include "fpvm.cuh"
#include "fp_inv_gcd.cuh"
#include "g1_ntt_units.cuh"
#include <algorithm>
#include <cstdlib>

namespace ekzg {

std::atomic<unsigned long long> g_kernel_launches{0};

__device__ __forceinline__ int rev_bits(int x, int bits) { return (int)(__brev((unsigned)x) >> (32 - bits)); }

// ------------------------------------------------------------------------------------------------
// setup: twiddle tables  tw[i] = base^i
// ------------------------------------------------------------------------------------------------
__global__ void k_powers(Fr* out, Fr base, Fr scale, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = scale, b = base;
    for (int e = i; e; e >>= 1) {
        if (e & 1) fe_mul(acc, acc, b);
        fe_sqr(b, b);
    }
    st_vec(&out[i], acc);
}

// ------------------------------------------------------------------------------------------------
// K1  blob bytes -> coefficients (+ the upper 64 cells)
//   reference: deserialize_blob_to_scalars (serialization/src/lib.rs:36-63), reverse_bit_order + ifft_scalars
//   (fk20/prover.rs:177-180), compute_coset_evaluations (fk20/prover.rs:158-165), serialize (lib.rs:132-156).
//   One CTA per blob, the 4096 elements stay in shared memory (128 KiB) from the wire format in to the
//   wire format out.  The 8192-point extension is split by hand: its even outputs are the blob itself
//   (cells 0..63 are a byte copy), its odd outputs are one 4096-point NTT of c[i]*omega_8192^i.
// ------------------------------------------------------------------------------------------------
constexpr int K1_THREADS = 1024;

__global__ void __launch_bounds__(K1_THREADS, 1)
k_blob_to_coeffs_cells(const uint8_t* __restrict__ blobs, Fr* __restrict__ coeffs, uint8_t* __restrict__ cells,
                       uint32_t* __restrict__ status, DevTables T, int want_cells) {
    extern __shared__ uint32_t sm[];
    const int b = blockIdx.x, tid = threadIdx.x;
    const uint8_t* blob = blobs + (size_t)b * BYTES_PER_BLOB;
    const Fr r2 = fe_const_r2<FrParams>();
    bool bad = false;
    for (int i = tid; i < N_BLOB; i += K1_THREADS) {
        Fr e = fr_load_be(blob + 32 * i);
        bad |= fe_plain_ge_mod(e);
        fe_mul(e, e, r2);
        smem_st(sm, N_BLOB, i, e);
    }
    if (bad) atomicOr(&status[b], 1u);
    __syncthreads();
    // c = INTT_4096(BRP(e)): DIT on the array as it lies
    ntt_dit_shared<12>(sm, N_BLOB, 1, T.tw4096_inv, tid, K1_THREADS);
    const Fr ninv = fr_inv_4096();
    Fr* cf = coeffs + (size_t)b * N_BLOB;
    for (int i = tid; i < N_BLOB; i += K1_THREADS) {
        Fr c = smem_ld(sm, N_BLOB, i);
        fe_mul(c, c, ninv);
        st_vec(&cf[i], c);
        if (want_cells) {
            Fr w = ld_vec(&T.tw8192[i]);
            fe_mul(c, c, w);
            smem_st(sm, N_BLOB, i, c);
        }
    }
    if (!want_cells) return;
    __syncthreads();
    ntt_dif_shared<12>(sm, N_BLOB, 1, T.tw4096, tid, K1_THREADS);
    uint8_t* out = cells + (size_t)b * (N_EXT * 32);
    for (int i = tid; i < N_BLOB; i += K1_THREADS) {
        Fr v = smem_ld(sm, N_BLOB, i);
        fe_from_mont(v, v);
        fr_store_be(out + (size_t)(N_BLOB + i) * 32, v);
        // cells 0..63: BRP(NTT_4096(c)) == the blob's own field elements
        const uint4* src = reinterpret_cast<const uint4*>(blob + 32 * i);
        uint4* dst = reinterpret_cast<uint4*>(out + 32 * i);
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

// Half `halfsel` of the 8192-point extension of one blob's coefficients cf, as big-endian bytes at out: BRP(NTT_4096(c))
// (halfsel 0: cells 0..63, i.e. the blob) or BRP(NTT_4096(c[i] w8192^i)) (halfsel 1: cells 64..127).  sm: 128 KiB.
__device__ __forceinline__ void coeffs_half_to_be(const Fr* __restrict__ cf, uint8_t* __restrict__ out, int halfsel, const DevTables& T,
                                                  uint32_t* sm, int tid) {
    for (int i = tid; i < N_BLOB; i += K1_THREADS) {
        Fr c = ld_vec(&cf[i]);
        if (halfsel) {
            Fr w = ld_vec(&T.tw8192[i]);
            fe_mul(c, c, w);
        }
        smem_st(sm, N_BLOB, i, c);
    }
    __syncthreads();
    ntt_dif_shared<12>(sm, N_BLOB, 1, T.tw4096, tid, K1_THREADS);
    for (int i = tid; i < N_BLOB; i += K1_THREADS) {
        Fr v = smem_ld(sm, N_BLOB, i);
        fe_from_mont(v, v);
        fr_store_be(out + (size_t)i * 32, v);
    }
}

// coefficients -> all 128 cells (recovery path: Input::PolyCoeff, fk20/prover.rs:184-188 + 158-165)
__global__ void __launch_bounds__(K1_THREADS, 1)
k_coeffs_to_cells(const Fr* __restrict__ coeffs, uint8_t* __restrict__ cells, DevTables T) {
    extern __shared__ uint32_t sm[];
    const int b = blockIdx.x, tid = threadIdx.x;
    const Fr* cf = coeffs + (size_t)b * N_BLOB;
    uint8_t* out = cells + (size_t)b * (N_EXT * 32);
    for (int halfsel = 0; halfsel < 2; halfsel++) {
        coeffs_half_to_be(cf, out + (size_t)halfsel * BYTES_PER_BLOB, halfsel, T, sm, tid);
        __syncthreads();
    }
}

// coefficients -> the blob (cells 0..63 only: half the transforms and half the bytes of k_coeffs_to_cells)
__global__ void __launch_bounds__(K1_THREADS, 1)
k_coeffs_to_blob(const Fr* __restrict__ coeffs, uint8_t* __restrict__ blobs, DevTables T) {
    extern __shared__ uint32_t sm[];
    const int b = blockIdx.x;
    coeffs_half_to_be(coeffs + (size_t)b * N_BLOB, blobs + (size_t)b * BYTES_PER_BLOB, 0, T, sm, threadIdx.x);
}

// ------------------------------------------------------------------------------------------------
// K2  coefficients -> the 128x64 MSM scalars of a blob
//   reference: compute_h_poly_commitments (fk20/h_poly.rs:36-53), CirculantMatrix::from_toeplitz
//   (fk20/toeplitz.rs:132-144), the 64 fft_scalars(128) + transpose of sum_matrix_vector_mul
//   (fk20/batch_toeplitz.rs:94-107).  a_k = [c[4095-k], 0^64, c[4095-k-64*63], ..., c[4095-k-64]].
//   The 1/128 of the later G1 inverse NTT (domain.rs:172-194) is folded into the scalars here.
//   One CTA handles K2_ROWS of the 64 rows of one blob.
// ------------------------------------------------------------------------------------------------
constexpr int K2_ROWS = 8;
constexpr int K2_THREADS = K2_ROWS * 64;

__global__ void __launch_bounds__(K2_THREADS)
k_toeplitz_scalars(const Fr* __restrict__ coeffs, uint32_t* __restrict__ scalars, DevTables T, int B, int b0) {
    __shared__ uint32_t sm[8 * K2_ROWS * 128];
    constexpr int STRIDE = K2_ROWS * 128;
    const int b = b0 + blockIdx.x, k0 = blockIdx.y * K2_ROWS, tid = threadIdx.x;
    const Fr* cf = coeffs + (size_t)b * N_BLOB;
    const Fr inv128 = fr_inv_128();
    for (int e = tid; e < K2_ROWS * 128; e += K2_THREADS) {
        int q = e >> 7, i = e & 127, k = k0 + q;
        Fr v;
        fe_set_zero(v);
        int src = -1;
        if (i == 0) src = 4095 - k;
        else if (i > 64) src = 4095 - k - 64 * (128 - i);
        if (src >= 0) {
            v = ld_vec(&cf[src]);
            fe_mul(v, v, inv128);
        }
        smem_st(sm, STRIDE, e, v);
    }
    __syncthreads();
    ntt_dif_shared<7>(sm, STRIDE, K2_ROWS, T.tw128, tid, K2_THREADS);
    // array position p of row q holds A_k[rev7(p)]; write plain integers to scalars[j][k][b]
    for (int e = tid; e < K2_ROWS * 128; e += K2_THREADS) {
        int q = e >> 7, p = e & 127, k = k0 + q, j = rev_bits(p, 7);
        Fr v = smem_ld(sm, STRIDE, e);
        fe_from_mont(v, v);
        uint32_t* dst = scalars + ((size_t)(j * FK20_POINTS + k) * B + b) * 8;
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        d4[0] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
        d4[1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
    }
}

// ------------------------------------------------------------------------------------------------
// K4  the 128 fixed-base MSMs of every blob   (HOT LOOP #1)
//   reference: FixedBaseMSMPrecompWindow::msm (fixed_base_msm_window.rs:102-168) with
//   multi_batch_addition_binary_tree_stride (batch_addition.rs:142-232).
//   One thread per (MSM j, blob b, slice of the 64 points): it walks its points and windows, turns each
//   window into a signed Booth digit, gathers the table entry and accumulates in XYZZ coordinates
//   (8M+2S per entry, no doublings at all because every window has its own table slice).  Lanes of a
//   warp are 32 blobs on the same MSM, so table gathers hit the same few KiB and scalar loads coalesce.
//   The slices of one (j, b) are combined through shared memory; the sum is written as a Jacobian point
//   at the BIT-REVERSED position so the inverse G1 NTT can run decimation-in-time without a shuffle.
// ------------------------------------------------------------------------------------------------
template <int NSLICE>
__global__ void __launch_bounds__(128)
k_fk20_msm(const uint32_t* __restrict__ scalars, G1Jac* __restrict__ pts, MsmTable T, int B, int b0, int b1) {
    // block = 128 threads = NSLICE slices x (128/NSLICE) blobs of one MSM j
    constexpr int BLOBS_PER_CTA = 128 / NSLICE;
    constexpr int KPER = FK20_POINTS / NSLICE;
    const int j = blockIdx.y;
    const int lane_b = threadIdx.x % BLOBS_PER_CTA, slice = threadIdx.x / BLOBS_PER_CTA;
    const int b = b0 + blockIdx.x * BLOBS_PER_CTA + lane_b;   // this launch covers blobs [b0, b1) of the batch of B
    const bool active = b < b1;
    G1Xyzz acc;
    xyzz_set_inf(acc);
    if (active) {
        const int w = T.w, nw = T.nw, mg = T.mg;
        const int nreg = mg > 1 ? nw - 1 : nw;   // windows with a slice of their own
        int comb = 0, radix = 1;                 // merged top digits of the current group of mg points (MsmTable)
        for (int kk = 0; kk < KPER; kk++) {
            const int k = slice * KPER + kk;
            const uint4* sp = reinterpret_cast<const uint4*>(scalars + ((size_t)(j * FK20_POINTS + k) * B + b) * 8);
            uint4 s0 = sp[0], s1 = sp[1];
            uint32_t s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
            const G1Affine* tb = T.table + (size_t)(j * FK20_POINTS + k) * T.nw * T.half;
            for (int t = 0; t < nreg; t++) {
                int d = booth_digit(s, t, w);
                if (d != 0) {
                    int m = (d < 0 ? -d : d) - 1;
                    G1Affine e = ld_vec(&tb[(size_t)t * T.half + m]);
                    xyzz_madd(acc, e, d < 0);
                }
            }
            if (mg > 1) {
                comb += booth_digit(s, nw - 1, w) * radix;   // in [0, rtop): scalars are < 2^255
                radix *= T.rtop;
                if ((kk & (mg - 1)) == mg - 1) {
                    if (comb != 0) {
                        const G1Affine* tg = tb - (size_t)(mg - 1) * T.nw * T.half;   // top slice of the group's first point
                        G1Affine e = ld_vec(&tg[(size_t)(nw - 1) * T.half + comb - 1]);
                        xyzz_madd(acc, e, false);
                    }
                    comb = 0;
                    radix = 1;
                }
            }
        }
    }
    __shared__ G1Xyzz red[NSLICE > 1 ? 128 : 1];
    if (NSLICE > 1) {
        for (int step = NSLICE / 2; step >= 1; step >>= 1) {
            if (slice >= step && slice < 2 * step) red[threadIdx.x] = acc;
            __syncthreads();
            if (slice < step) xyzz_add(acc, red[threadIdx.x + step * BLOBS_PER_CTA]);
            __syncthreads();
        }
    }
    if (active && slice == 0) {
        G1Jac r;
        jac_from_xyzz(r, acc);
        st_vec(&pts[(size_t)rev_bits(j, 7) * B + b], r);
    }
}

// ------------------------------------------------------------------------------------------------
// The Fp interpreter shared by the hot kernels (fpvm.cuh): the ONLY copy of the Montgomery multiplier, the squarer and
// the fused two-product multiplier in their instruction stream.  `base` = shared-space address of the calling thread's
// chunk of slot 0; runs instructions [pc, pc + n) of the program table `reps` times; bit i of the result is set when
// instruction i produced zero (the callers test the H / R differences of the addition formulas with it).
// ------------------------------------------------------------------------------------------------
__constant__ uint32_t c_fpvm_prog[fpvm::FPVM_PROG_WORDS] = FPVM_PROG_INIT;

static __device__ __noinline__ uint32_t fpvm_run(uint32_t base, int pc, int n, int reps) {
    fpvm::Smem m{base};
    uint32_t z = 0;
#pragma unroll 1
    for (int r = 0; r < reps; r++) {
#pragma unroll 1
        for (int i = 0; i < n; i++) z |= fpvm::step(m, c_fpvm_prog[pc + i]) << i;
    }
    return z;
}
#define FPVM_RUN(base, NAME) fpvm_run(base, fpvm::PROG_##NAME, fpvm::PROG_##NAME##_LEN, 1)

__device__ __forceinline__ Fp fp_one() {
    Fp r;
    fe_set_one(r);
    return r;
}

// ------------------------------------------------------------------------------------------------
// K4, shared-memory-operand form (the production kernel; the register form above is kept for A/B runs, EKZG_K4=reg).
//   Same thread mapping and table walk as k_fk20_msm.  The XYZZ accumulator of a thread lives in slots 0..3, the table
//   entry is staged into slots 4..5 and slots 6..7 are scratch; one mixed addition = 9 interpreter instructions.
//   The Booth digits come off the low end of the scalar, which is shifted right one window at a time (funnel shifts on
//   statically indexed registers -- the register form indexed its limbs dynamically, which put the scalar in local memory).
//   The entry of the NEXT window is prefetched into L2 before the current one is accumulated, so the 96-byte gather from
//   the 144 GiB of tables is in flight during the ~5000 pipe clocks of an addition (holding it in registers instead
//   would not fit: the interpreter owns 96 of the 128 registers).
// ------------------------------------------------------------------------------------------------
// rare: acc and the entry have the same x.  Same point -> double the entry; opposite -> identity.
static __device__ __noinline__ bool k4_same_x(uint32_t base, const G1Affine* p, bool neg, bool r_is_zero) {
    if (!r_is_zero) return true;          // acc == -e: the sum is the identity
    G1Affine e = ld_vec(p);
    fe_cneg(e.y, e.y, neg);
    G1Xyzz d;
    xyzz_dbl_affine(d, e);
    fpvm::Smem M{base};
    M.st(0, d.x); M.st(1, d.y); M.st(2, d.zz); M.st(3, d.zzz);
    return false;
}
// acc (slots 0..3; `inf`: nothing there yet) += (neg ? -*p : *p)
__device__ __forceinline__ bool k4_accumulate(uint32_t base, const G1Affine* p, bool neg, bool inf) {
    const fpvm::Smem M{base};
    G1Affine e = ld_vec(p);
    if (g1a_is_inf(e)) return inf;
    fe_cneg(e.y, e.y, neg);
    if (inf) {
        M.st(0, e.x); M.st(1, e.y); M.st(2, fp_one()); M.st(3, fp_one());
        return false;
    }
    M.st(4, e.x); M.st(5, e.y);
    const uint32_t z = FPVM_RUN(base, K4_XYZZ_MADD_A);
    if (z & 1u) return k4_same_x(base, p, neg, (z & 2u) != 0);
    FPVM_RUN(base, K4_XYZZ_MADD_B);
    return false;
}
__device__ __forceinline__ void prefetch_entry_l2(const G1Affine* p) {   // 96 bytes, 32-byte aligned: one or two 128-byte lines
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p) + 80));
}
// rare: the two accumulators of a slice reduction have the same x.  Equal points: the sum is twice the OTHER thread's
// accumulator, which still sits untouched in its own slots 0..3.
static __device__ __noinline__ bool k4_same_x_xyzz(uint32_t base, uint32_t other_base, bool r_is_zero) {
    if (!r_is_zero) return true;
    const fpvm::Smem O{other_base};
    G1Xyzz a, d;
    a.x = O.ld(0); a.y = O.ld(1); a.zz = O.ld(2); a.zzz = O.ld(3);
    xyzz_dbl(d, a);
    fpvm::Smem M{base};
    M.st(0, d.x); M.st(1, d.y); M.st(2, d.zz); M.st(3, d.zzz);
    return false;
}

template <int NSLICE>
__global__ void __launch_bounds__(fpvm::NT, 4)
k_fk20_msm_vm(const uint32_t* __restrict__ scalars, G1Jac* __restrict__ pts, MsmTable T, int B, int b0, int b1) {
    extern __shared__ uint4 vm_smem[];
    static_assert(fpvm::NT == 128, "thread mapping below assumes 128-thread CTAs");
    constexpr int BLOBS_PER_CTA = 128 / NSLICE;
    constexpr int KPER = FK20_POINTS / NSLICE;
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(vm_smem) + threadIdx.x * 16u;
    const fpvm::Smem M{base};
    const int j = blockIdx.y;
    const int lane_b = threadIdx.x % BLOBS_PER_CTA, slice = threadIdx.x / BLOBS_PER_CTA;
    const int b = b0 + blockIdx.x * BLOBS_PER_CTA + lane_b;
    const bool active = b < b1;
    bool inf = true;                       // accumulator is the identity (nothing in slots 0..3 yet)
    int comb = 0, radix = 1;               // digits of the merged top window collected so far
    if (active) {
        const int w = T.w, nw = T.nw, mg = T.mg;
        const int nreg = mg > 1 ? nw - 1 : nw;
        const uint32_t vmask = (2u << w) - 1u;
        // one entry ahead: the next window's table entry is pulled into L2 while the current one is accumulated
        const G1Affine* pend = nullptr;
        bool pend_neg = false;
#define K4_EMIT(ptr, negflag)                                     \
    do {                                                          \
        const G1Affine* np_ = (ptr);                              \
        prefetch_entry_l2(np_);                                   \
        if (pend) inf = k4_accumulate(base, pend, pend_neg, inf); \
        pend = np_;                                               \
        pend_neg = (negflag);                                     \
    } while (0)
        for (int kk = 0; kk < KPER; kk++) {
            const int k = slice * KPER + kk;
            const uint4* sp = reinterpret_cast<const uint4*>(scalars + ((size_t)(j * FK20_POINTS + k) * B + b) * 8);
            const uint4 s0 = sp[0], s1 = sp[1];
            uint32_t s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
            uint32_t prev = 0;             // bit t*w - 1 of the scalar
            const G1Affine* tb = T.table + (size_t)(j * FK20_POINTS + k) * T.nw * T.half;
            for (int t = 0; t <= nreg; t++) {
                const uint32_t v = ((s[0] << 1) | prev) & vmask;
                const int d = (int)((v + 1) >> 1) - (int)((v >> w) << w);   // booth_digit, g1_mul.cuh
                if (t == nreg) {           // t = nw - 1 when the top window is merged, else one past the top (d == 0)
                    if (mg > 1) { comb += d * radix; radix *= T.rtop; }
                    break;
                }
                prev = (s[0] >> (w - 1)) & 1u;
#pragma unroll
                for (int i = 0; i < 7; i++) s[i] = __funnelshift_r(s[i], s[i + 1], w);
                s[7] >>= w;
                if (d != 0) K4_EMIT(&tb[(size_t)t * T.half + ((d < 0 ? -d : d) - 1)], d < 0);
            }
            if (mg > 1 && (kk & (mg - 1)) == mg - 1) {
                if (comb != 0) {
                    const G1Affine* tg = tb - (size_t)(mg - 1) * T.nw * T.half;   // top slice of the group's first point
                    K4_EMIT(&tg[(size_t)(nw - 1) * T.half + comb - 1], false);
                }
                comb = 0;
                radix = 1;
            }
        }
        if (pend) inf = k4_accumulate(base, pend, pend_neg, inf);
#undef K4_EMIT
    }
    if (KPER < 4 && T.mg > 1) {
        // fewer points per thread than the merged top window ties together (64 slices: ONE point per thread): the top digits of a group
        // of mg consecutive points sit in mg neighbouring slices -- threads BLOBS_PER_CTA apart, in one warp -- and the thread of the
        // group's first point adds the merged entry.  (Every thread of the CTA is here: inactive ones contribute zero digits.)
        static_assert(KPER >= 4 || KPER == 1, "one point per thread, or whole merge groups");
        const int mg = T.mg;
        int total = comb, rad = T.rtop;
        for (int i = 1; i < mg; i++) {
            total += rad * __shfl_down_sync(0xffffffffu, comb, i * BLOBS_PER_CTA);
            rad *= T.rtop;
        }
        if (active && (slice & (mg - 1)) == 0 && total != 0) {
            const G1Affine* tg = T.table + (size_t)(j * FK20_POINTS + slice) * T.nw * T.half;   // top slice of the group's first point
            inf = k4_accumulate(base, &tg[(size_t)(T.nw - 1) * T.half + total - 1], false, inf);
        }
    }
    if (NSLICE > 1) {
        __shared__ uint8_t s_inf[128];
        for (int step = NSLICE / 2; step >= 1; step >>= 1) {
            s_inf[threadIdx.x] = inf ? 1 : 0;
            __syncthreads();
            if (slice < step) {
                const int other = threadIdx.x + step * BLOBS_PER_CTA;
                if (!s_inf[other]) {
                    const fpvm::Smem O{base + (uint32_t)(step * BLOBS_PER_CTA) * 16u};
                    if (inf) {
                        for (int c = 0; c < 4; c++) M.st(c, O.ld(c));
                        inf = false;
                    } else {
                        for (int c = 0; c < 4; c++) M.st(4 + c, O.ld(c));
                        const uint32_t z = FPVM_RUN(base, K4_XYZZ_ADD_A);
                        if (z & 2u) inf = k4_same_x_xyzz(base, O.base, (z & 8u) != 0);
                        else FPVM_RUN(base, K4_XYZZ_ADD_B);
                    }
                }
            }
            __syncthreads();
        }
    }
    if (active && slice == 0) {
        G1Jac r;
        if (inf) {
            jac_set_inf(r);
        } else {
            FPVM_RUN(base, K4_XYZZ_TO_JAC);
            r.x = M.ld(0); r.y = M.ld(1); r.z = M.ld(2);
        }
        st_vec(&pts[(size_t)rev_bits(j, 7) * B + b], r);
    }
}

// ------------------------------------------------------------------------------------------------
// K4a  the fixed-base MSMs with BATCHED AFFINE additions (opt-in: EKZG_K4=a)
//   reference: the same FixedBaseMSMPrecompWindow::msm, which also adds in affine coordinates and shares inversions
//   (batch_addition.rs:142-232 multi_batch_addition_binary_tree_stride, batch_inversion.rs) -- there across a tree of
//   points, here across the WINDOWS of one scalar:
//     a thread owns one accumulator PER WINDOW (affine, in a per-thread scratch block in global memory / L2).  Round k
//     adds, for every window t, the table entry picked by digit t of scalar k to accumulator t: ~19 independent
//     additions whose denominators x_e - x_acc are inverted together (Montgomery's trick: one product chain forward,
//     ONE inversion by division steps -- fp_inv_gcd.cuh, mostly ALU work -- one chain backward).  An addition then costs
//     5M + 1S + 1/19 inversion (~2000 wide multiply-adds) instead of the 8M + 2S = 2712 of an XYZZ mixed addition.
//     After the last round the window accumulators are summed (XYZZ, 18 additions per thread) and the slices of one
//     (MSM, blob) combined through shared memory as in k_fk20_msm.
//   Equal-x cases stay complete: accumulator == entry puts 2y / 3x^2 into the same batch (affine doubling),
//   accumulator == -entry empties the accumulator, digit 0 and empty accumulators take no part in the product chain.
//   Scratch: [CTA slot][window][x0 x1 x2 y0 y1 y2][thread] and [CTA slot][batch slot][p0 p1 p2][thread] in 16-byte
//   granules, so a warp's access to one granule is 512 contiguous bytes.
// ------------------------------------------------------------------------------------------------
constexpr int K4A_HALF = 16;               // additions of one half-batch (slots that share one inversion per thread)
constexpr int K4A_THREADS = 128;           // worker threads of a CTA (its fifth warp only inverts)
constexpr int K4A_CTA = K4A_THREADS + 32;

struct K4aScratch {
    uint4* acc;     // this thread's granule 0 of window 0
    uint4* pre;     // this thread's granule 0 of batch slot 0
    __device__ __forceinline__ Fp ld(const uint4* p) const {
        Fp r;
        #pragma unroll
        for (int q = 0; q < 3; q++) { const uint4 g = __ldcg(p + q * K4A_THREADS); r.v[4 * q] = g.x; r.v[4 * q + 1] = g.y; r.v[4 * q + 2] = g.z; r.v[4 * q + 3] = g.w; }
        return r;
    }
    __device__ __forceinline__ void st(uint4* p, const Fp& v) const {
        #pragma unroll
        for (int q = 0; q < 3; q++) __stcg(p + q * K4A_THREADS, make_uint4(v.v[4 * q], v.v[4 * q + 1], v.v[4 * q + 2], v.v[4 * q + 3]));
    }
    __device__ __forceinline__ void prefetch(const uint4* p) const {   // one element (three granules) towards L2
#pragma unroll
        for (int q = 0; q < 3; q++) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + q * K4A_THREADS));
    }
    __device__ __forceinline__ uint4* ax(int t) const { return acc + (size_t)t * 6 * K4A_THREADS; }
    __device__ __forceinline__ uint4* ay(int t) const { return acc + ((size_t)t * 6 + 3) * K4A_THREADS; }
    __device__ __forceinline__ uint4* pr(int t) const { return pre + (size_t)t * 3 * K4A_THREADS; }
};

enum : uint32_t { K4A_SKIP = 0, K4A_INIT = 1, K4A_ADD = 2, K4A_DBL = 3, K4A_CANCEL = 4 };

static __device__ __noinline__ Fp k4a_inverse(Fp a) {
    Fp r;
    fp_inv_gcd(r, a);
    return r;
}

// shared-memory exchange of the per-thread denominator products: element of thread i as three 16-byte granules at
// [q][i], so a warp's access is conflict-free
struct K4aXchg {
    uint4* base;   // granule 0 of thread 0
    __device__ __forceinline__ Fp ld(int thread) const {
        Fp r;
        #pragma unroll
        for (int q = 0; q < 3; q++) { const uint4 g = base[q * K4A_THREADS + thread]; r.v[4 * q] = g.x; r.v[4 * q + 1] = g.y; r.v[4 * q + 2] = g.z; r.v[4 * q + 3] = g.w; }
        return r;
    }
    __device__ __forceinline__ void st(int thread, const Fp& v) const {
        #pragma unroll
        for (int q = 0; q < 3; q++) base[q * K4A_THREADS + thread] = make_uint4(v.v[4 * q], v.v[4 * q + 1], v.v[4 * q + 2], v.v[4 * q + 3]);
    }
};

// named barriers (0 is __syncthreads): products of half h posted / inverses of half h ready / workers only
__device__ __forceinline__ void k4a_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void k4a_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
enum { K4A_BAR_POSTED = 1, K4A_BAR_READY = 3, K4A_BAR_WORKERS = 5 };

// forward pass over the slots [lo, hi) of one half-batch: classify, chain the denominators; returns the chain product
__device__ __forceinline__ Fp k4a_forward(const K4aScratch& S, uint32_t (*info_rows)[K4A_THREADS], int lo, int hi, int nreg, const G1Affine* tb,
                                          const G1Affine* tg, uint64_t has) {
    Fp run;
    bool run_set = false;
    if (lo < hi) S.prefetch(S.ax(lo));
    for (int t = lo; t < hi; t++) {
        const uint32_t info = info_rows[t - lo][threadIdx.x];
        if (t + 1 < hi) S.prefetch(S.ax(t + 1));
        if ((info & 7u) == K4A_SKIP) continue;
        const G1Affine* ep = (t < nreg ? tb : tg) + (info >> 4);
        const bool neg = (info & 8u) != 0;
        const Fp ex = ld_vec(&ep->x);
        bool e_inf = false;
        if (fe_is_zero(ex)) { const Fp ey = ld_vec(&ep->y); e_inf = fe_is_zero(ey); }
        uint32_t mode = K4A_ADD;
        if (e_inf) {
            mode = K4A_SKIP;
        } else if (!((has >> t) & 1ull)) {
            mode = K4A_INIT;
        } else {
            Fp den;
            const Fp ax = S.ld(S.ax(t));
            fe_sub(den, ex, ax);
            if (fe_is_zero(den)) {           // same x: the same point (double it) or its negative (cancel)
                Fp ey = ld_vec(&ep->y);
                fe_cneg(ey, ey, neg);
                const Fp ay = S.ld(S.ay(t));
                if (fe_eq(ey, ay)) { mode = K4A_DBL; fe_dbl(den, ay); } else mode = K4A_CANCEL;
            }
            if (mode != K4A_CANCEL) {
                if (run_set) {
                    S.st(S.pr(t), run);
                    fe_mul(run, run, den);
                } else {
                    S.st(S.pr(t), fp_one());
                    run = den;
                    run_set = true;
                }
            }
        }
        info_rows[t - lo][threadIdx.x] = (info & ~7u) | mode;
    }
    return run_set ? run : fp_one();
}

// backward pass: peel the slot inverses off `inv` (the inverse of the chain product) and finish the additions
__device__ __forceinline__ uint64_t k4a_backward(const K4aScratch& S, uint32_t (*info_rows)[K4A_THREADS], int lo, int hi, int nreg, const G1Affine* tb,
                                                 const G1Affine* tg, uint64_t has, Fp inv) {
    for (int t = hi - 1; t >= lo; t--) {
        const uint32_t info = info_rows[t - lo][threadIdx.x];
        const uint32_t mode = info & 7u;
        if (t > lo) { S.prefetch(S.pr(t - 1)); S.prefetch(S.ax(t - 1)); S.prefetch(S.ay(t - 1)); }
        if (mode == K4A_SKIP) continue;
        if (mode == K4A_CANCEL) { has &= ~(1ull << t); continue; }
        const G1Affine* ep = (t < nreg ? tb : tg) + (info >> 4);
        const Fp ex = ld_vec(&ep->x);
        Fp ey = ld_vec(&ep->y);
        fe_cneg(ey, ey, (info & 8u) != 0);
        if (mode == K4A_INIT) {
            S.st(S.ax(t), ex);
            S.st(S.ay(t), ey);
            has |= 1ull << t;
            continue;
        }
        const Fp ax = S.ld(S.ax(t)), ay = S.ld(S.ay(t));
        Fp den, num, dinv, lam, x3, y3;
        {
            const Fp pre = S.ld(S.pr(t));
            fe_mul(dinv, inv, pre);              // 1 / denominator of this slot
        }
        if (mode == K4A_DBL) {
            fe_dbl(den, ay);
            fe_sqr(num, ax);
            fe_dbl(x3, num);
            fe_add(num, num, x3);                // 3 x^2
        } else {
            fe_sub(den, ex, ax);
            fe_sub(num, ey, ay);
        }
        fe_mul(inv, inv, den);                   // inverse of the remaining chain
        fe_mul(lam, num, dinv);
        fe_sqr(x3, lam);
        fe_sub(x3, x3, ax);
        fe_sub(x3, x3, ex);
        fe_sub(y3, ax, x3);
        fe_mul(y3, y3, lam);
        fe_sub(y3, y3, ay);
        S.st(S.ax(t), x3);
        S.st(S.ay(t), y3);
    }
    return has;
}

// Schedule.  The windows of a scalar are split into a low half A and a high half B (the merged top window is in B).  The
// four worker warps run, per point k:
//     forward(A_k), post | wait, backward(B_k-1) | forward(B_k), post | wait, backward(A_k)
// and the fifth warp does nothing but: wait for the 128 posted products of a half, multiply the four of each lane column
// together, invert (division steps: ALU work, off the multiply pipe the workers saturate), hand the four inverses back.
// Between posting a product and needing its inverse a worker has ~55 field multiplications of the other half to do, about
// twice what the inverter needs, so nobody waits; an inversion serves 128 threads x ~10 additions.
__global__ void __launch_bounds__(K4A_CTA, 3)
k_fk20_msm_affine(const uint32_t* __restrict__ scalars, G1Jac* __restrict__ pts, MsmTable T, int B, int b0, int b1, int nslice, int nitems_x,
                  int ngroups, uint4* __restrict__ scratch, size_t scratch_cta_granules) {
    // slot descriptors of half A, and of half B double-buffered (B of point k is finished after the digits of point k+1 are
    // taken); the slice reduction at the end of an item reuses the same 24 KB
    __shared__ __align__(16) uint32_t s_info[3][K4A_HALF][K4A_THREADS];
    static_assert(sizeof(G1Xyzz) * K4A_THREADS <= sizeof(uint32_t) * 3 * K4A_HALF * K4A_THREADS, "the slice reduction reuses the slot descriptors");
    uint32_t (*s_info_a)[K4A_THREADS] = s_info[0];
    G1Xyzz* red = reinterpret_cast<G1Xyzz*>(&s_info[0][0][0]);
    __shared__ uint4 s_xchg[2][3 * K4A_THREADS];
    const int w = T.w, nw = T.nw, mg = T.mg;
    const int nreg = mg > 1 ? nw - 1 : nw;          // windows with a table slice of their own
    const int nslots = mg > 1 ? nreg + 1 : nreg;    // + the merged top window
    const int n_a = (nslots + 1) / 2;               // half A = slots [0, n_a), half B = [n_a, nslots)
    const int blobs_per_cta = K4A_THREADS / nslice, kper = FK20_POINTS / nslice;
    const int nitems = nitems_x * ngroups;
    if (threadIdx.x >= K4A_THREADS) {
        // ---- the inverter warp ----
        const int lane = threadIdx.x - K4A_THREADS;
        constexpr int NWARP = K4A_THREADS / 32;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            for (int r = 0; r < 2 * kper; r++) {
                const int h = r & 1;
                const K4aXchg X{s_xchg[h]};
                k4a_bar_sync(K4A_BAR_POSTED + h, K4A_CTA);
                Fp acc = X.ld(lane);
                Fp part[NWARP - 1];                  // products of the first 1, 2, .. chains (statically indexed: registers)
#pragma unroll
                for (int q = 1; q < NWARP; q++) {
                    part[q - 1] = acc;
                    const Fp a = X.ld(q * 32 + lane);
                    fe_mul(acc, acc, a);
                }
                Fp iv = k4a_inverse(acc);
#pragma unroll
                for (int q = NWARP - 1; q >= 1; q--) {
                    const Fp a = X.ld(q * 32 + lane);
                    Fp mine;
                    fe_mul(mine, iv, part[q - 1]);   // 1 / chain q
                    fe_mul(iv, iv, a);
                    X.st(q * 32 + lane, mine);
                }
                X.st(lane, iv);
                k4a_bar_arrive(K4A_BAR_READY + h, K4A_CTA);
            }
        }
        return;
    }
    // ---- the workers ----
    const int lane_b = threadIdx.x % blobs_per_cta, slice = threadIdx.x / blobs_per_cta;
    const uint32_t vmask = (2u << w) - 1u;
    const K4aXchg XA{s_xchg[0]}, XB{s_xchg[1]};
    K4aScratch S;
    S.acc = scratch + (size_t)blockIdx.x * scratch_cta_granules + threadIdx.x;
    S.pre = S.acc + (size_t)nslots * 6 * K4A_THREADS;
    const size_t point_stride = (size_t)nw * T.half;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int j = item / nitems_x, bx = item - j * nitems_x;
        const int b = b0 + bx * blobs_per_cta + lane_b;
        const bool active = b < b1;                  // (inactive threads walk the same loops: the CTA shares its inversions)
        uint64_t has = 0;                            // bit t: accumulator t holds a point
        int comb = 0, radix = 1;
        for (int kk = 0; kk < kper; kk++) {
            const int k = slice * kper + kk;
            const G1Affine* tb = T.table + (size_t)(j * FK20_POINTS + k) * point_stride;
            const G1Affine* tg = tb - (size_t)(mg - 1) * point_stride;   // first point of this point's merge group
            uint32_t (*info_b)[K4A_THREADS] = s_info[1 + (kk & 1)];
            {
                // digits of scalar k -> table offsets of all its windows; the entries start their way in from HBM
                uint32_t s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                if (active) {
                    const uint4* sp = reinterpret_cast<const uint4*>(scalars + ((size_t)(j * FK20_POINTS + k) * B + b) * 8);
                    const uint4 s0 = sp[0], s1 = sp[1];
                    s[0] = s0.x; s[1] = s0.y; s[2] = s0.z; s[3] = s0.w; s[4] = s1.x; s[5] = s1.y; s[6] = s1.z; s[7] = s1.w;
                }
                uint32_t prev = 0;                   // bit t*w - 1 of the scalar
                const bool top_round = mg > 1 && (kk & (mg - 1)) == mg - 1;
                for (int t = 0; t < nslots; t++) {
                    const uint32_t v = ((s[0] << 1) | prev) & vmask;
                    const int d = (int)((v + 1) >> 1) - (int)((v >> w) << w);   // booth_digit, g1_mul.cuh
                    uint32_t info = K4A_SKIP;        // bits 0..2 mode, bit 3 negate, bits 4.. offset of the entry
                    if (t < nreg) {
                        prev = (s[0] >> (w - 1)) & 1u;
#pragma unroll
                        for (int i = 0; i < 7; i++) s[i] = __funnelshift_r(s[i], s[i + 1], w);
                        s[7] >>= w;
                        if (d != 0) {
                            const uint32_t off = (uint32_t)t * T.half + (uint32_t)((d < 0 ? -d : d) - 1);
                            info = K4A_ADD | (d < 0 ? 8u : 0u) | (off << 4);
                            prefetch_entry_l2(tb + off);
                        }
                    } else {                         // merged top window: the digits of mg consecutive points index one entry
                        comb += d * radix;
                        radix *= T.rtop;
                        if (top_round) {
                            if (comb != 0) {
                                const uint32_t off = (uint32_t)(nw - 1) * T.half + (uint32_t)(comb - 1);
                                info = K4A_ADD | (off << 4);
                                prefetch_entry_l2(tg + off);
                            }
                            comb = 0;
                            radix = 1;
                        }
                    }
                    if (t < n_a) s_info_a[t][threadIdx.x] = info; else info_b[t - n_a][threadIdx.x] = info;
                }
            }
            XA.st(threadIdx.x, k4a_forward(S, s_info_a, 0, n_a, nreg, tb, tg, has));
            k4a_bar_arrive(K4A_BAR_POSTED + 0, K4A_CTA);
            if (kk > 0) {                            // finish half B of the previous point
                k4a_bar_sync(K4A_BAR_READY + 1, K4A_CTA);
                has = k4a_backward(S, s_info[1 + ((kk - 1) & 1)], n_a, nslots, nreg, tb - point_stride, tg - point_stride, has, XB.ld(threadIdx.x));
            }
            XB.st(threadIdx.x, k4a_forward(S, info_b, n_a, nslots, nreg, tb, tg, has));
            k4a_bar_arrive(K4A_BAR_POSTED + 1, K4A_CTA);
            k4a_bar_sync(K4A_BAR_READY + 0, K4A_CTA);
            has = k4a_backward(S, s_info_a, 0, n_a, nreg, tb, tg, has, XA.ld(threadIdx.x));
        }
        {
            const int k = slice * kper + kper - 1;
            const G1Affine* tb = T.table + (size_t)(j * FK20_POINTS + k) * point_stride;
            k4a_bar_sync(K4A_BAR_READY + 1, K4A_CTA);
            has = k4a_backward(S, s_info[1 + ((kper - 1) & 1)], n_a, nslots, nreg, tb, tb - (size_t)(mg - 1) * point_stride, has, XB.ld(threadIdx.x));
        }
        // the window accumulators of this thread, then the slices of one (MSM, blob)
        G1Xyzz acc;
        xyzz_set_inf(acc);
        for (int t = 0; t < nslots; t++) {
            if ((has >> t) & 1ull) {
                G1Affine e;
                e.x = S.ld(S.ax(t));
                e.y = S.ld(S.ay(t));
                xyzz_madd(acc, e, false);
            }
        }
        if (nslice > 1) k4a_bar_sync(K4A_BAR_WORKERS, K4A_THREADS);   // everybody is done with the slot descriptors `red` overlays
        for (int step = nslice / 2; step >= 1; step >>= 1) {
            if (slice >= step && slice < 2 * step) red[threadIdx.x] = acc;
            k4a_bar_sync(K4A_BAR_WORKERS, K4A_THREADS);
            if (slice < step) xyzz_add(acc, red[threadIdx.x + step * blobs_per_cta]);
            k4a_bar_sync(K4A_BAR_WORKERS, K4A_THREADS);
        }
        if (active && slice == 0) {
            G1Jac r;
            jac_from_xyzz(r, acc);
            st_vec(&pts[(size_t)rev_bits(j, 7) * B + b], r);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K5  the two 128-point G1 NTTs of every blob   (HOT LOOP #2)
//   reference: Domain::ifft_g1_take_n / fft_g1 (polynomial/src/domain.rs:149-194) over the generic
//   butterfly `dit` (fft.rs:164-177) whose `*b * twiddle` is a full scalar multiplication.
//
//   Work unit = one butterfly of 32 blobs (a warp; blob fastest), so the twiddle -- hence the whole
//   double-and-add schedule of jac_mul_ops -- is warp-uniform.  A butterfly with a non-trivial twiddle
//   costs ~1500 Fp multiplications per lane, one with twiddle 1 costs ~30, and a phase of a batch holds
//   only 64*B/32 units: per-stage launches leave most SMs idle in every tail.  So the 14 phases run in
//   ONE persistent kernel: warps pull units from a global ticket counter in (phase, blob group,
//   butterfly) order; a unit of phase p waits until the 64 units of phase p-1 of ITS blob group are
//   done (release/acquire counter per (group, phase)).  A unit only ever waits for tickets handed out
//   before its own, each held by a running warp, so there is no deadlock whatever the residency.
//   phase 0..6 : inverse DIT stage `ph` (input bit-reversed, written that way by K4).  The last one only
//                produces the 64 kept outputs (ifft_g1_take_n(.., 64)); the 1/128 is already in the scalars.
//   phase 7..13: forward DIF stage 13-ph on (h || O^64): the first (stage 6) is h[i] -> (h[i], w^i h[i]).
//                The output of the last stage is in bit-reversed order = proof order (fk20/prover.rs:222).
// ------------------------------------------------------------------------------------------------
__constant__ uint16_t c_twiddle_ops[128][MULOPS_STRIDE] =
#include "twiddle_ops.inc"
    ;

constexpr int NTT_THREADS = 128;
constexpr int NTT_PHASES = 14;

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_inc(unsigned* p) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}

// queue[0] = ticket counter, queue[1 + g*14 + ph] = finished units of (blob group g, phase ph); zeroed by the launcher
template <int MIN_BLOCKS>
__global__ void __launch_bounds__(NTT_THREADS, MIN_BLOCKS)
k_fk20_g1_ntts(G1Jac* __restrict__ pts, int B, int G, int ph0, int ph1, unsigned* __restrict__ queue) {
    const int lane = threadIdx.x & 31;
    const unsigned per_phase = (unsigned)G * 64u;
    const unsigned total = (unsigned)(ph1 - ph0) * per_phase;
    for (;;) {
        unsigned id = 0;
        if (lane == 0) id = atomicAdd(&queue[0], 1u);
        id = __shfl_sync(0xffffffffu, id, 0);
        if (id >= total) break;
        const unsigned rel = id / per_phase, rem = id - rel * per_phase;
        const int g = (int)(rem >> 6), t = (int)(rem & 63u), ph = ph0 + (int)rel;
        unsigned* cnt = queue + 1 + (size_t)g * NTT_PHASES;
        if (rel > 0) {
            if (lane == 0) {
                while (ld_acquire_u32(cnt + ph - 1) < 64u) __nanosleep(256);
            }
            __syncwarp();
        }
        const int b = g * 32 + lane;
        if (b < B) g1_ntt_butterfly(pts, B, b, t, ph, c_twiddle_ops);
        __threadfence();
        __syncwarp();
        if (lane == 0) red_release_inc(cnt + ph);
    }
}

// ------------------------------------------------------------------------------------------------
// K5, radix-4 form for SMALL batches (latency mode: a lone blob, a coalesced handful, a 128-blob shard of a strong-scaled job)
//   A batch of B blobs gives the radix-2 kernel above only 64*ceil(B/32) warps of work per phase, and its 14 phases are a
//   dependent chain of 12 fixed-scalar multiplications (~1.4 ms each for a warp that has its sub-partition to itself): 20 ms
//   whatever B is.  Here two consecutive radix-2 stages are flattened into one super-phase:
//       inverse DIT stages (s, s+1) on x0..x3 = pts[base + {0, 1, 2, 3} * 2^s]:
//           y0 = x0 + p1 + p2 + p3    y2 = x0 + p1 - p2 - p3    y1 = x0 - p1 + p4 - p5    y3 = x0 - p1 - p4 + p5
//           p1 = W(ea) x1, p2 = W(eb) x2, p3 = W(ea+eb) x3, p4 = W(eb+32) x2, p5 = W(ea+eb+32) x3        (W(e) = omega^-e)
//       middle: inverse stage 6 (only the 64 kept outputs) + forward stage 6:  pts[t] = x0 + W(t) x1,  pts[t+64] = omega^t x0 + x1
//       forward DIF stages (s+1, s):
//           y0 = x0+x1+x2+x3   y1 = w(ea)(x0-x1+x2-x3)   y2 = w(eb)(x0-x2) + w(eb+32)(x1-x3)   y3 = w(ea+eb)(x0-x2) - w(ea+eb+32)(x1-x3)
//   The five products of a radix-4 butterfly are independent, so a super-phase is ONE multiplication deep: 7 instead of 12 on
//   the critical path, for 25 % more multiplications (5 per 4 points and two stages instead of 4) -- which is why the wide
//   launches keep the radix-2 kernel.  Same persistent ticket queue; per blob group and super-phase, 160 (middle: 128)
//   multiplication units write their products to a scratch array, then 32 (64) combination units add them up in place.
// ------------------------------------------------------------------------------------------------
// queue[0] = ticket counter, queue[1 + (g*7 + sp)*2 + kind] = finished multiplication (0) / combination (1) units of blob group g
// in super-phase sp; zeroed by the launcher.  Tickets: super-phase major, then all multiplication units, then all combinations.
// GW = blobs per blob group (= per warp): 32, one lane per blob; or 8 (COOP), where a multiplication unit spreads every field element
// of a blob over four lanes (r4_mul_unit_coop) and a combination unit spreads its independent additions over the four lanes of a
// blob (r4_combine_unit_par) -- for batches so small that the machine is mostly idle and only the latency of the dependent
// products counts (launch_g1_ntt_phases picks; a queue of 1 + 14 ceil(B/8) counters, well inside g1_ntt_queue_words(B)).
template <int GW>
__global__ void __launch_bounds__(NTT_THREADS, 2)
k_fk20_g1_ntts_r4(G1Jac* __restrict__ pts, G1Jac* __restrict__ tmp, int B, int G, int sp_end, unsigned* __restrict__ queue) {
    __shared__ G1Jac xch[GW == 32 ? 1 : NTT_THREADS];   // cooperative form: intermediate sums of the combination units, one slot per lane
    const int lane = threadIdx.x & 31;
    const unsigned per_sp = (unsigned)G * R4_UNITS, total = per_sp * (unsigned)sp_end;
    for (;;) {
        unsigned id = 0;
        if (lane == 0) id = atomicAdd(&queue[0], 1u);
        id = __shfl_sync(0xffffffffu, id, 0);
        if (id >= total) break;
        const int sp = (int)(id / per_sp);
        unsigned rem = id - (unsigned)sp * per_sp;
        const unsigned nmul = (unsigned)r4_nmul(sp), ncomb = R4_UNITS - nmul;
        const bool comb = rem >= (unsigned)G * nmul;
        if (comb) rem -= (unsigned)G * nmul;
        const unsigned per = comb ? ncomb : nmul;
        const int g = (int)(rem / per), u = (int)(rem - (unsigned)g * per);
        unsigned* cnt = queue + 1 + ((size_t)g * R4_SUPER + sp) * 2;
        // a multiplication unit reads what the combinations of the previous super-phase wrote; a combination unit reads the
        // products of its own super-phase (and overwrites the inputs of all of them)
        const unsigned* wait_on = comb ? cnt : (sp > 0 ? cnt - 1 : nullptr);
        const unsigned need = comb ? nmul : (unsigned)(R4_UNITS - r4_nmul(sp - 1));
        if (wait_on) {
            if (lane == 0) {
                while (ld_acquire_u32(wait_on) < need) __nanosleep(128);
            }
            __syncwarp();
        }
        if (GW == 32) {
            const int b = g * 32 + lane;
            if (b < B) {
                if (comb) r4_combine_unit(pts, tmp, B, b, sp, u);
                else r4_mul_unit(pts, tmp, B, b, sp, u, c_twiddle_ops);
            }
        } else if (comb) {
            const int b = g * GW + (lane >> 2);              // all 32 lanes: the four lanes of a blob share the unit's additions
            r4_combine_unit_par(pts, tmp, B, b, lane & 3, b < B, sp, u, &xch[(threadIdx.x >> 5) * 32]);
        } else {
            r4_mul_unit_coop(pts, tmp, B, g * GW + (lane >> 2), sp, u, c_twiddle_ops);   // all 32 lanes: 8 blobs x 4 lanes
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) red_release_inc(cnt + (comb ? 1 : 0));
    }
}

// ------------------------------------------------------------------------------------------------
// K5, shared-memory-operand form (the production kernel; the register form above stays for A/B runs, EKZG_K5=reg).
//   Same persistent ticket queue, but
//   * the whole fixed-scalar ladder (jac_mul_ops, g1_mul.cuh) runs on the Fp interpreter: accumulator, the staged table
//     entry and three temporaries in the eight shared-memory slots of a lane, 128 registers, four 128-thread CTAs per SM
//     (the register form: 255 registers, 3136 bytes of stack, two CTAs);
//   * the eight odd multiples (x, y, beta*x, rescaled to one common Z) live in a per-warp scratch block in global memory
//     (L2): they are written once and read ~43 times per ladder, while the accumulator is touched by every instruction;
//   * a unit waits for the TWO butterflies of the previous phase that produced its inputs (one flag per unit) instead
//     of for all 64 of its blob group, so a blob group's phases overlap and the 4 x 148 x 4 resident warps stay busy.
// ------------------------------------------------------------------------------------------------
constexpr int K5_SCRATCH_FP = 26;                                           // per lane: 8 x (x, y, beta*x), zfix, dz
constexpr size_t K5_SCRATCH_WARP_BYTES = (size_t)K5_SCRATCH_FP * 3 * 32 * 16;

struct GScratch {                 // this lane's view of its warp's scratch block (uint4 granules, lane-interleaved)
    uint4* p;
    __device__ __forceinline__ Fp ld(int idx) const {
        Fp r;
        #pragma unroll
        for (int q = 0; q < 3; q++) { const uint4 g = __ldcg(p + (idx * 3 + q) * 32); r.v[4 * q] = g.x; r.v[4 * q + 1] = g.y; r.v[4 * q + 2] = g.z; r.v[4 * q + 3] = g.w; }
        return r;
    }
    __device__ __forceinline__ void st(int idx, const Fp& v) const {
        #pragma unroll
        for (int q = 0; q < 3; q++) __stcg(p + (idx * 3 + q) * 32, make_uint4(v.v[4 * q], v.v[4 * q + 1], v.v[4 * q + 2], v.v[4 * q + 3]));
    }
};

// slots 0..2 (a Jacobian point P of prime order, not the identity) <- k * P for the fixed scalar behind `ops`
// (twiddle_ops.inc); returns true if the result is the identity.  Mirrors jac_mul_ops step by step.
static __device__ __noinline__ bool k5_mul_ops_vm(uint32_t base, uint4* gsp, const uint16_t* __restrict__ ops) {
    using namespace fpvm;
    const Smem M{base};
    const GScratch G{gsp};
    // P aside (in the slots of table entry 7, which is written last), d = 2P
    G.st(21, M.ld(0)); G.st(22, M.ld(1)); G.st(23, M.ld(2));
    FPVM_RUN(base, K5_JAC_DBL);
    M.st(3, G.ld(21)); M.st(4, G.ld(22));
    FPVM_RUN(base, K5_TBL_ISO);                       // slots 5, 6 = P on the curve isomorphic by Z(2P)
    G.st(25, M.ld(2));                                // Z(2P)
    { const Fp dx = M.ld(0), dy = M.ld(1); M.st(3, dx); M.st(4, dy); }   // 2P as an affine point of that curve
    { const Fp cx = M.ld(5), cy = M.ld(6); M.st(0, cx); M.st(1, cy); G.st(0, cx); G.st(1, cy); }
    M.st(2, G.ld(23));
#pragma unroll 1
    for (int i = 1; i < 8; i++) {                     // (2i+1)P = (2i-1)P + 2P, z-ratio H kept for the rescaling
        FPVM_RUN(base, K5_TBL_MADDZR_A);
        G.st(3 * i + 2, M.ld(5));
        FPVM_RUN(base, K5_TBL_MADDZR_B);
        G.st(3 * i, M.ld(0)); G.st(3 * i + 1, M.ld(1));
    }
    M.st(5, M.ld(2)); M.st(6, G.ld(25));
    FPVM_RUN(base, K5_MUL_T0_T1);                     // zfix = Z(15P) * Z(2P): maps the ladder's result back
    G.st(24, M.ld(5));
    // one common Z for all entries (entry 7 has it already), beta*x beside x
    M.st(0, G.ld(23));                                // running z-ratio, starts at H_7
    {
        Fp beta;
#pragma unroll
        for (int l = 0; l < 12; l++) beta.v[l] = FpParams::beta(l);
        M.st(6, beta);
    }
    M.st(3, G.ld(21));
    FPVM_RUN(base, K5_TBL_BETA);
    G.st(23, M.ld(7));
#pragma unroll 1
    for (int i = 6; i >= 0; i--) {
        M.st(3, G.ld(3 * i)); M.st(4, G.ld(3 * i + 1));
        if (i) M.st(5, G.ld(3 * i + 2));
        FPVM_RUN(base, K5_TBL_RESCALE);
        G.st(3 * i, M.ld(3)); G.st(3 * i + 1, M.ld(4)); G.st(3 * i + 2, M.ld(7));
    }
    // the ladder: mixed additions of table entries (phi applied by taking beta*x), doublings in between
    bool inf = true;
    const int n = ops[0];
#pragma unroll 1
    for (int c = 1; c <= n; c++) {
        const uint32_t op = ops[c];
        const int dbl = (int)(op >> 8);
        if (dbl && !inf) fpvm_run(base, PROG_K5_JAC_DBL, PROG_K5_JAC_DBL_LEN, dbl);
        if (op & 0x20u) {
            const int idx = (int)(op & 7u);
            const Fp ex = G.ld(3 * idx + ((op & 0x10u) ? 2 : 0));
            Fp ey = G.ld(3 * idx + 1);
            fe_cneg(ey, ey, (op & 8u) != 0);
            if (inf) {
                M.st(0, ex); M.st(1, ey); M.st(2, fp_one());
                inf = false;
            } else {
                M.st(3, ex); M.st(4, ey);
                const uint32_t z = FPVM_RUN(base, K5_JAC_MADD_A);
                if (z & 2u) {                         // same x: cannot happen for a point of prime order, handled all the same
                    if (z & 8u) FPVM_RUN(base, K5_JAC_DBL); else inf = true;
                } else {
                    FPVM_RUN(base, K5_JAC_MADD_B);
                }
            }
        }
    }
    if (!inf) {
        M.st(5, G.ld(24));
        FPVM_RUN(base, K5_MUL_Z_T0);
    }
    return inf;
}

// slots 0..2 += slots 3..5 (Jacobian, either may be the identity as flagged); returns "the sum is the identity"
static __device__ __noinline__ bool k5_add_vm(uint32_t base, bool acc_inf, bool q_inf) {
    using namespace fpvm;
    const Smem M{base};
    if (q_inf) return acc_inf;
    if (acc_inf) {
        for (int c = 0; c < 3; c++) M.st(c, M.ld(3 + c));
        return false;
    }
    const uint32_t z = FPVM_RUN(base, K5_JAC_ADD_A);
    if (z & 8u) {                                     // H == 0
        if (!(z & 0x80u)) return true;                // P1 == -P2
        FPVM_RUN(base, K5_MUL_Z_QZ);                  // (U1, S1, Z1*Z2) is P1: double it
        FPVM_RUN(base, K5_JAC_DBL);
        return false;
    }
    FPVM_RUN(base, K5_JAC_ADD_B);
    return false;
}

__device__ __forceinline__ void vm_put_pt(const fpvm::Smem& M, int slot0, const G1Jac& p, bool neg_y) {
    M.st(slot0, p.x);
    if (neg_y) { Fp ny; fe_neg(ny, p.y); M.st(slot0 + 1, ny); } else M.st(slot0 + 1, p.y);
    M.st(slot0 + 2, p.z);
}
__device__ __forceinline__ G1Jac vm_get_pt(const fpvm::Smem& M, bool inf) {
    G1Jac r;
    if (inf) { jac_set_inf(r); return r; }
    r.x = M.ld(0); r.y = M.ld(1); r.z = M.ld(2);
    return r;
}

static __device__ __noinline__ void g1_ntt_butterfly_vm(G1Jac* __restrict__ pts, int B, int b, int t, int ph, uint32_t base, uint4* gsp) {
    const fpvm::Smem M{base};
    const int mode = ph >= 7, st = mode ? 13 - ph : ph;
    const int len = 1 << st;
    const int pos = t & (len - 1);
    const int i = ((t >> st) << (st + 1)) + pos, j = i + len;
    const int e = pos << (6 - st);  // twiddle exponent of omega_128
    G1Jac* pi = &pts[(size_t)i * B + b];
    G1Jac* pj = &pts[(size_t)j * B + b];
    if (mode == 0) {
        // v' = w^-e * v;  pi <- u + v';  pj <- u - v' (not needed in the last inverse stage)
        bool v_inf;
        {
            const G1Jac v = ld_pt(pj);
            v_inf = jac_is_inf(v);
            if (!v_inf) vm_put_pt(M, 0, v, false);
        }
        if (!v_inf && e != 0) v_inf = k5_mul_ops_vm(base, gsp, c_twiddle_ops[(128 - e) & 127]);
        const GScratch G{gsp};
        if (st != 6 && !v_inf) { G.st(0, M.ld(0)); G.st(1, M.ld(1)); G.st(2, M.ld(2)); }   // v' aside (the table is dead now)
        bool u_inf;
        {
            const G1Jac u = ld_pt(pi);
            u_inf = jac_is_inf(u);
            if (!u_inf) vm_put_pt(M, 3, u, false);
        }
        const bool s_inf = k5_add_vm(base, v_inf, u_inf);
        if (st == 6) {
            st_pt(pi, vm_get_pt(M, s_inf));
            return;
        }
        {
            const G1Jac u = ld_pt(pi);
            st_pt(pi, vm_get_pt(M, s_inf));
            if (!u_inf) vm_put_pt(M, 0, u, false);
        }
        if (!v_inf) {
            M.st(3, G.ld(0));
            Fp ny = G.ld(1);
            fe_neg(ny, ny);
            M.st(4, ny);
            M.st(5, G.ld(2));
        }
        const bool d_inf = k5_add_vm(base, u_inf, v_inf);
        st_pt(pj, vm_get_pt(M, d_inf));
    } else if (st == 6) {
        // first forward stage on (h || O^64):  pj <- w^e * h_i
        const G1Jac u = ld_pt(pi);
        bool u_inf = jac_is_inf(u);
        if (u_inf || e == 0) { st_pt(pj, u); return; }
        vm_put_pt(M, 0, u, false);
        u_inf = k5_mul_ops_vm(base, gsp, c_twiddle_ops[e]);
        st_pt(pj, vm_get_pt(M, u_inf));
    } else {
        // pi <- u + v;  pj <- w^e * (u - v)
        bool u_inf, v_inf;
        {
            const G1Jac u = ld_pt(pi);
            u_inf = jac_is_inf(u);
            if (!u_inf) vm_put_pt(M, 0, u, false);
            const G1Jac v = ld_pt(pj);
            v_inf = jac_is_inf(v);
            if (!v_inf) vm_put_pt(M, 3, v, false);
        }
        const bool s_inf = k5_add_vm(base, u_inf, v_inf);
        {
            const G1Jac u = ld_pt(pi);
            st_pt(pi, vm_get_pt(M, s_inf));
            if (!u_inf) vm_put_pt(M, 0, u, false);
            const G1Jac v = ld_pt(pj);
            if (!v_inf) vm_put_pt(M, 3, v, true);
        }
        bool d_inf = k5_add_vm(base, u_inf, v_inf);
        if (!d_inf && e != 0) d_inf = k5_mul_ops_vm(base, gsp, c_twiddle_ops[e]);
        st_pt(pj, vm_get_pt(M, d_inf));
    }
}

// the butterfly of phase ph - 1 that wrote point x (both transforms are in place: each point belongs to exactly one
// butterfly per phase, so these are also the only earlier readers of the points a unit is about to overwrite)
__device__ __forceinline__ int ntt_producer(int ph, int x) {
    if (ph <= 6) {                      // inverse DIT stage st = ph, producer at stage st - 1
        const int sp = ph - 1;
        return ((x >> (sp + 1)) << sp) + (x & ((1 << sp) - 1));
    }
    if (ph == 7) return x & 63;         // last inverse stage, butterfly x (x < 64; point x + 64 was only read there)
    const int sp = 13 - ph + 1;         // forward DIF stage st = 13 - ph, producer at stage st + 1
    return ((x >> (sp + 1)) << sp) + (x & ((1 << sp) - 1));
}

// queue[0] = ticket counter, queue[1 + (g*14 + ph)*64 + t] = 1 when unit (blob group g, phase ph, butterfly t) is done
__global__ void __launch_bounds__(fpvm::NT, 4)
k_fk20_g1_ntts_vm(G1Jac* __restrict__ pts, int B, int G, int ph0, int ph1, unsigned* __restrict__ queue, uint4* __restrict__ scratch) {
    extern __shared__ uint4 vm_smem[];
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(vm_smem) + threadIdx.x * 16u;
    const int lane = threadIdx.x & 31;
    uint4* gsp = scratch + ((size_t)blockIdx.x * (fpvm::NT / 32) + (threadIdx.x >> 5)) * (K5_SCRATCH_WARP_BYTES / 16) + lane;
    const unsigned per_phase = (unsigned)G * 64u;
    const unsigned total = (unsigned)(ph1 - ph0) * per_phase;
    for (;;) {
        unsigned id = 0;
        if (lane == 0) id = atomicAdd(&queue[0], 1u);
        id = __shfl_sync(0xffffffffu, id, 0);
        if (id >= total) break;
        const unsigned rel = id / per_phase, rem = id - rel * per_phase;
        const int g = (int)(rem >> 6), t = (int)(rem & 63u), ph = ph0 + (int)rel;
        unsigned* flags = queue + 1 + (size_t)g * (NTT_PHASES * 64);
        if (rel > 0) {
            if (lane < 2) {
                const int mode = ph >= 7, st = mode ? 13 - ph : ph;
                const int pos = t & ((1 << st) - 1);
                const int i = ((t >> st) << (st + 1)) + pos;
                const int x = lane == 0 ? i : i + (1 << st);
                const unsigned* f = flags + (ph - 1) * 64 + ntt_producer(ph, x);
                while (ld_acquire_u32(f) == 0u) __nanosleep(200);
            }
            __syncwarp();
        }
        const int b = g * 32 + lane;
        if (b < B) g1_ntt_butterfly_vm(pts, B, b, t, ph, base, gsp);
        __threadfence();
        __syncwarp();
        if (lane == 0) red_release_inc(flags + ph * 64 + t);
    }
}

// ------------------------------------------------------------------------------------------------
// K6  Jacobian -> affine -> 48-byte compressed
//   reference: g1_batch_normalize (bls12_381/src/lib.rs:56-104) + serialize_g1_compressed
//   (serialization/src/lib.rs:84-86, 138).  One thread per point, blob-fastest input.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_g1_compress(const G1Jac* __restrict__ pts, uint8_t* __restrict__ out, int npos, int B) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= npos * B) return;
    const int p = gid / B, b = gid - p * B;
    G1Jac q = ld_vec(&pts[(size_t)p * B + b]);
    G1Affine a;
    if (jac_is_inf(q)) {
        g1a_set_inf(a);
    } else {
        Fp zi;
        fp_inv(zi, q.z);
        jac_to_affine_with_inv(a, q, zi);
    }
    uint8_t buf[48];
    g1a_compress(buf, a);
    uint8_t* dst = out + ((size_t)b * npos + p) * BYTES_PER_G1;
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(buf);
    (void)w;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        uint4 v;
        v.x = buf[16 * c + 0] | (buf[16 * c + 1] << 8) | (buf[16 * c + 2] << 16) | ((uint32_t)buf[16 * c + 3] << 24);
        v.y = buf[16 * c + 4] | (buf[16 * c + 5] << 8) | (buf[16 * c + 6] << 16) | ((uint32_t)buf[16 * c + 7] << 24);
        v.z = buf[16 * c + 8] | (buf[16 * c + 9] << 8) | (buf[16 * c + 10] << 16) | ((uint32_t)buf[16 * c + 11] << 24);
        v.w = buf[16 * c + 12] | (buf[16 * c + 13] << 8) | (buf[16 * c + 14] << 16) | ((uint32_t)buf[16 * c + 15] << 24);
        d4[c] = v;
    }
}

// Same, CH consecutive positions of one blob per thread sharing ONE inversion (Montgomery's trick, the device twin of
// the reference's shared inversion in g1_batch_normalize): 460/CH + 3 multiplications per point instead of 460.
// Identities (z = 0) are kept out of the product and re-inserted, like the reference does (lib.rs:60-76).
constexpr int K6_CH = 8;
__global__ void __launch_bounds__(128)
k_g1_compress_batched(const G1Jac* __restrict__ pts, uint8_t* __restrict__ out, int npos, int B) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nch = npos / K6_CH;
    if (gid >= nch * B) return;
    const int ch = gid / B, b = gid - ch * B;
    const int p0 = ch * K6_CH;
    Fp prefix[K6_CH];
    Fp run;
    fe_set_one(run);
#pragma unroll 1
    for (int i = 0; i < K6_CH; i++) {
        Fp z = ld_vec(&pts[(size_t)(p0 + i) * B + b].z);
        prefix[i] = run;
        if (!fe_is_zero(z)) fe_mul(run, run, z);
    }
    Fp inv;
    fp_inv(inv, run);
#pragma unroll 1
    for (int i = K6_CH - 1; i >= 0; i--) {
        G1Jac q = ld_vec(&pts[(size_t)(p0 + i) * B + b]);
        G1Affine a;
        if (jac_is_inf(q)) {
            g1a_set_inf(a);
        } else {
            Fp zi;
            fe_mul(zi, inv, prefix[i]);
            fe_mul(inv, inv, q.z);
            jac_to_affine_with_inv(a, q, zi);
        }
        uint8_t buf[48];
        g1a_compress(buf, a);
        uint4* d4 = reinterpret_cast<uint4*>(out + ((size_t)b * npos + p0 + i) * BYTES_PER_G1);
#pragma unroll
        for (int c = 0; c < 3; c++) {
            uint4 v;
            v.x = buf[16 * c + 0] | (buf[16 * c + 1] << 8) | (buf[16 * c + 2] << 16) | ((uint32_t)buf[16 * c + 3] << 24);
            v.y = buf[16 * c + 4] | (buf[16 * c + 5] << 8) | (buf[16 * c + 6] << 16) | ((uint32_t)buf[16 * c + 7] << 24);
            v.z = buf[16 * c + 8] | (buf[16 * c + 9] << 8) | (buf[16 * c + 10] << 16) | ((uint32_t)buf[16 * c + 11] << 24);
            v.w = buf[16 * c + 12] | (buf[16 * c + 13] << 8) | (buf[16 * c + 14] << 16) | ((uint32_t)buf[16 * c + 15] << 24);
            d4[c] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// setup kernels
// ------------------------------------------------------------------------------------------------
// 48-byte compressed points -> affine Montgomery; status[i] != 0 on malformed input.
__global__ void k_g1_decompress(const uint8_t* __restrict__ in, G1Affine* __restrict__ out, uint32_t* __restrict__ status, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t buf[48];
    for (int c = 0; c < 48; c++) buf[c] = in[(size_t)i * 48 + c];
    G1Affine a;
    int rc = g1a_decompress(a, buf);
    if (rc) { g1a_set_inf(a); status[i] = 1; }
    st_vec(&out[i], a);
}

// FK20 setup, step 1 (fk20/prover.rs:88-104): lay the 64 strided SRS vectors V_k out as the lower half of
// a 128-point G1 NTT input, "blob" index := k.   pts[m][k] = srs[4031 - (k + 64 m)], m < 63; identity else.
__global__ void k_fk20_setup_vectors(const G1Affine* __restrict__ srs, G1Jac* __restrict__ pts) {
    int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= 128 * 64) return;
    int m = gid / 64, k = gid % 64;
    G1Jac r;
    jac_set_inf(r);
    int idx = k + 64 * m;
    if (m < 63 && idx < 4032) {
        G1Affine a = ld_vec(&srs[4031 - idx]);
        jac_from_affine(r, a);
    }
    st_vec(&pts[(size_t)m * 64 + k], r);
}

// FK20 setup, step 2: per base point P = F_k[j] (at pts[rev7(j)][k] after the DIF NTT) the window
// bases Q_t = 2^(t*w) P, normalised to affine with one shared inversion per thread.
constexpr int MAX_NW = 64;
__global__ void __launch_bounds__(64)
k_fk20_window_bases(const G1Jac* __restrict__ pts, const G1Affine* __restrict__ aff, G1Affine* __restrict__ qaff, int w, int nw, int npoints) {
    int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= npoints) return;
    G1Jac p;
    if (aff) {  // plain list of affine base points
        G1Affine a = ld_vec(&aff[gid]);
        jac_from_affine(p, a);
    } else {    // FK20: base (j, k) sits at pts[rev7(j)][k] after the DIF NTT
        int j = gid / FK20_POINTS, k = gid % FK20_POINTS;
        p = ld_vec(&pts[(size_t)rev_bits(j, 7) * 64 + k]);
    }
    G1Affine* dst = qaff + (size_t)gid * nw;
    G1Jac qs[MAX_NW];
    Fp prefix[MAX_NW];
    G1Jac q = p;
    Fp run;
    fe_set_one(run);
    for (int t = 0; t < nw; t++) {
        if (t) for (int s = 0; s < w; s++) jac_dbl(q, q);
        qs[t] = q;
        prefix[t] = run;          // product of z_0..z_{t-1}
        fe_mul(run, run, q.z);
    }
    Fp inv;
    fp_inv(inv, run);             // 1 / prod z_u   (all z_u != 0: P has prime order)
    for (int t = nw - 1; t >= 0; t--) {
        Fp zi;
        fe_mul(zi, inv, prefix[t]);   // 1/z_t
        fe_mul(inv, inv, qs[t].z);    // drop z_t
        G1Affine a;
        jac_to_affine_with_inv(a, qs[t], zi);
        st_vec(&dst[t], a);
    }
}

// FK20 setup, step 3 (fixed_base_msm_window.rs:69-82 precompute_points, once per window):
// table[(j,k,t)][m] = (m+1) * Q_t for m < half, affine.  One thread per chunk of CH consecutive m.
constexpr int TBL_CH = 64;   // entries sharing one inversion (Montgomery trick): 450/64 + ~19 multiplications per entry
__global__ void __launch_bounds__(128)
k_fk20_table_fill(const G1Affine* __restrict__ qaff, G1Affine* __restrict__ table, int half, size_t nbases) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int chunks = (half + TBL_CH - 1) / TBL_CH;
    if (gid >= nbases * chunks) return;
    const size_t base = gid / chunks;
    const int c = (int)(gid % chunks);
    const G1Affine q = ld_vec(&qaff[base]);
    // start = (c*CH + 1) * Q
    G1Jac acc;
    jac_set_inf(acc);
    uint32_t mult = (uint32_t)c * TBL_CH + 1;
    for (int bit = 31 - __clz(mult); bit >= 0; bit--) {
        jac_dbl(acc, acc);
        if ((mult >> bit) & 1) jac_madd(acc, q, false);
    }
    G1Jac buf[TBL_CH];
    Fp prefix[TBL_CH];
    Fp run;
    fe_set_one(run);
    const int cnt = min(TBL_CH, half - c * TBL_CH);
    for (int i = 0; i < cnt; i++) {
        if (i) jac_madd(acc, q, false);
        buf[i] = acc;
        prefix[i] = run;
        fe_mul(run, run, acc.z);
    }
    Fp inv;
    fp_inv(inv, run);
    G1Affine* dst = table + base * half + (size_t)c * TBL_CH;
    for (int i = cnt - 1; i >= 0; i--) {
        Fp zi;
        fe_mul(zi, inv, prefix[i]);
        fe_mul(inv, inv, buf[i].z);
        G1Affine a;
        jac_to_affine_with_inv(a, buf[i], zi);
        st_vec(&dst[i], a);
    }
}

// FK20 setup, step 4: merged top-window slices (MsmTable::mg).  For every group of mg consecutive points, entry c - 1 of the
// top slice of the group's first point becomes sum_i d_i * Q_i, c = sum_i d_i * rtop^i, Q_i = 2^(w(nw-1)) * P_i (qaff).
// One thread per entry; the d_i are at most 2^tb <= 2^(w-1), a plain double-and-add each.
__global__ void __launch_bounds__(128)
k_fk20_top_merge_fill(const G1Affine* __restrict__ qaff, G1Affine* __restrict__ table, int nw, int half, int rtop, int mg, int ncomb, size_t ngroups) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= ngroups * (size_t)(ncomb - 1)) return;
    const size_t g = gid / (ncomb - 1);
    int c = (int)(gid % (ncomb - 1)) + 1;
    const int c0 = c;
    G1Jac acc;
    jac_set_inf(acc);
    for (int i = 0; i < mg; i++) {
        const int d = c % rtop;
        c /= rtop;
        if (!d) continue;
        const G1Affine q = ld_vec(&qaff[(g * mg + i) * nw + (nw - 1)]);
        G1Jac t;
        jac_set_inf(t);
        for (int bit = 31 - __clz((unsigned)d); bit >= 0; bit--) {
            jac_dbl(t, t);
            if ((d >> bit) & 1) jac_madd(t, q, false);
        }
        jac_add(acc, t);
    }
    Fp zi;
    fp_inv(zi, acc.z);   // a non-trivial combination of independent points of prime order is never the identity
    G1Affine a;
    jac_to_affine_with_inv(a, acc, zi);
    st_vec(&table[((g * mg) * nw + (nw - 1)) * (size_t)half + (c0 - 1)], a);
}

// ------------------------------------------------------------------------------------------------
// launch wrappers
// ------------------------------------------------------------------------------------------------

cudaError_t launch_powers(Fr* out, const uint32_t* base_mont, int n, cudaStream_t st, const uint32_t* scale_mont) {
    Fr b, sc;
    for (int i = 0; i < 8; i++) b.v[i] = base_mont[i];
    for (int i = 0; i < 8; i++) sc.v[i] = scale_mont ? scale_mont[i] : FrParams::one(i);
    k_powers<<<(n + 127) / 128, 128, 0, st>>>(out, b, sc, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}


cudaError_t kernels_init() {
    cudaError_t e = cudaFuncSetAttribute(k_blob_to_coeffs_cells, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4);
    if (e != cudaSuccess) return e;
    // four 48 KB CTAs of the shared-memory-operand kernels per SM
    // (48 KB of dynamic shared memory plus any static bytes is above the 48 KB a kernel gets without opting in)
    e = cudaFuncSetAttribute(k_fk20_msm_vm<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_msm_vm<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, fpvm::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_msm_vm<16>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_msm_vm<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, fpvm::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_msm_vm<64>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_msm_vm<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, fpvm::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_g1_ntts_vm, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fk20_g1_ntts_vm, cudaFuncAttributeMaxDynamicSharedMemorySize, fpvm::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_coeffs_to_cells, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_coeffs_to_blob, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * N_BLOB * 4);
}

cudaError_t launch_blob_to_coeffs_cells(const uint8_t* blobs, Fr* coeffs, uint8_t* cells, uint32_t* status, const DevTables& T,
                                        int B, bool want_cells, cudaStream_t st) {
    k_blob_to_coeffs_cells<<<B, K1_THREADS, 8 * N_BLOB * 4, st>>>(blobs, coeffs, cells, status, T, want_cells ? 1 : 0);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_coeffs_to_cells(const Fr* coeffs, uint8_t* cells, const DevTables& T, int B, cudaStream_t st) {
    k_coeffs_to_cells<<<B, K1_THREADS, 8 * N_BLOB * 4, st>>>(coeffs, cells, T);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_coeffs_to_blob(const Fr* coeffs, uint8_t* blobs, const DevTables& T, int B, cudaStream_t st) {
    k_coeffs_to_blob<<<B, K1_THREADS, 8 * N_BLOB * 4, st>>>(coeffs, blobs, T);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_toeplitz_scalars(const Fr* coeffs, uint32_t* scalars, const DevTables& T, int B, cudaStream_t st, int b0, int cnt) {
    if (cnt < 0) cnt = B - b0;
    k_toeplitz_scalars<<<dim3(cnt, FK20_POINTS / K2_ROWS), K2_THREADS, 0, st>>>(coeffs, scalars, T, B, b0);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

// K4a geometry for a table: granules (16 B) of scratch per resident CTA, and how many CTAs can be resident
static int g_k4a_ctas = 0;
static cudaError_t k4a_query() {
    if (g_k4a_ctas) return cudaSuccess;
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fk20_msm_affine, K4A_CTA, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (const char* env = getenv("EKZG_K4A_OCC")) { const int v = atoi(env); if (v >= 1 && v < per_sm) per_sm = v; }
    g_k4a_ctas = sms * per_sm;
    return cudaSuccess;
}
static size_t k4a_cta_granules(const MsmTable& T) {
    const int nreg = T.mg > 1 ? T.nw - 1 : T.nw, nslots = T.mg > 1 ? nreg + 1 : nreg;
    return (size_t)(nslots * 6 + nslots * 3) * K4A_THREADS;   // accumulators (x, y) and chain prefixes of every window
}
size_t fixed_msm_scratch_bytes(const MsmTable& T) {
    if (k4a_query() != cudaSuccess) return 0;
    return (size_t)g_k4a_ctas * k4a_cta_granules(T) * 16;
}
// 'v' shared-memory-operand XYZZ (default: 50.9 ms per 1024 blobs), 'r' register XYZZ (51.9 ms), 'a' batched affine with
// the accumulators in a global scratch block (63 ms: latency-bound on the scratch traffic, profiles/r2_e_prof_k4a_*;
// kept for A/B runs)
// (the three knobs below are read at every launch, so that a test can switch forms inside one process)
static char k4_form() {
    const char* e = getenv("EKZG_K4");
    return e && (e[0] == 'r' || e[0] == 'a') ? e[0] : 'v';
}
static int k4a_slices() {   // slices per (MSM, blob) in the affine kernel: 1 = a thread walks all 64 points
    const char* e = getenv("EKZG_K4A_SLICES");
    const int x = e ? atoi(e) : 1;
    return x == 2 || x == 4 || x == 8 || x == 16 ? x : 1;
}
static size_t k4a_min_work() {   // launches with fewer (blob, MSM) pairs use the XYZZ kernels, which slice finer
    const char* e = getenv("EKZG_K4A_MIN");
    return e ? (size_t)atoll(e) : (size_t)512 * 128;
}

static bool k4_no_tiny() { const char* e = getenv("EKZG_K4_NO_TINY"); return e && *e == '1'; }   // A/B and test knob: never the 64-slice form

cudaError_t launch_fixed_msm(const uint32_t* scalars, G1Jac* pts, const MsmTable& T, int ngroups, int B, cudaStream_t st, int b0, int cnt,
                             void* scratch) {
    // ngroups MSMs of 64 points each per blob (FK20: 128; SRS commitment: 64 partial sums), blobs [b0, b0 + cnt) of the
    // batch of B (the strides of scalars[][][B] and pts[][B] are those of the whole batch).
    // fewer blobs per launch -> more slices per MSM so the machine still fills
    if (cnt < 0) cnt = B - b0;
    const bool wide = (size_t)B * ngroups >= 512 * 128;
    const char form = k4_form();
    const int nslots_a = T.mg > 1 ? T.nw : T.nw;   // (nw - 1 sliced windows + the merged one, or nw sliced windows)
    if (form == 'a' && scratch && nslots_a <= 2 * K4A_HALF && (size_t)B * ngroups >= k4a_min_work()) {
        cudaError_t e = k4a_query();
        if (e != cudaSuccess) return e;
        const int nslice = k4a_slices(), blobs_per_cta = K4A_THREADS / nslice;
        const int nitems_x = (cnt + blobs_per_cta - 1) / blobs_per_cta;
        const int grid = std::min(g_k4a_ctas, nitems_x * ngroups);
        k_fk20_msm_affine<<<dim3(grid, 1), K4A_CTA, 0, st>>>(scalars, pts, T, B, b0, b0 + cnt, nslice, nitems_x, ngroups,
                                                                   reinterpret_cast<uint4*>(scratch), k4a_cta_granules(T));
    } else if (form == 'r') {
        if (wide) k_fk20_msm<4><<<dim3((cnt + 31) / 32, ngroups), 128, 0, st>>>(scalars, pts, T, B, b0, b0 + cnt);
        else k_fk20_msm<16><<<dim3((cnt + 7) / 8, ngroups), 128, 0, st>>>(scalars, pts, T, B, b0, b0 + cnt);
    } else {
        // a handful of blobs on a table without a merged top window (the SRS tables at w = 13: a thread may own a single point):
        // 64 slices, one point per thread -- 20 additions and a 6-level reduction on the critical path instead of 80 and 4
        // (FK20 tables with a merged top window as well: the digits of a merge group are gathered across its threads; up to 16 blobs)
        const bool tiny = T.mg <= 4 && (size_t)cnt * ngroups <= (T.mg == 1 ? 8 * 64 : 16 * 128) && !k4_no_tiny();
        if (wide) k_fk20_msm_vm<4><<<dim3((cnt + 31) / 32, ngroups), fpvm::NT, fpvm::SMEM_BYTES, st>>>(scalars, pts, T, B, b0, b0 + cnt);
        else if (tiny) k_fk20_msm_vm<64><<<dim3((cnt + 1) / 2, ngroups), fpvm::NT, fpvm::SMEM_BYTES, st>>>(scalars, pts, T, B, b0, b0 + cnt);
        else k_fk20_msm_vm<16><<<dim3((cnt + 7) / 8, ngroups), fpvm::NT, fpvm::SMEM_BYTES, st>>>(scalars, pts, T, B, b0, b0 + cnt);
    }
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

static int g_ntt_sms = 0;
static int ntt_min_blocks() {
    static int v = [] { const char* e = getenv("EKZG_NTT_OCC"); int x = e ? atoi(e) : 2; return x < 2 ? 2 : (x > 4 ? 4 : x); }();
    return v;
}
static bool k5_register_form() {
    // measured on the B200 (profiles/r2_a_*): the shared-memory-operand K5 runs 43.6 ms against 34.7 ms for the register form at
    // 1024 blobs -- a phase holds only 2048 warp-sized units, fewer than the 2368 warps that form keeps resident, so every unit
    // of a phase runs at once at a quarter of a scheduler's pipe and the 12 dependent ladder phases stretch.  EKZG_K5=vm selects it.
    static const bool v = [] { const char* e = getenv("EKZG_K5"); return !(e && e[0] == 'v'); }();
    return v;
}
static cudaError_t ntt_query_sms() {
    if (g_ntt_sms) return cudaSuccess;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    g_ntt_sms = sms;
    return cudaSuccess;
}
constexpr int K5_VM_CTAS_PER_SM = 4;

// ticket counter + one completion flag per (blob group, phase, butterfly)
size_t g1_ntt_queue_words(int B) { return 1 + (size_t)((B + 31) / 32) * NTT_PHASES * 64; }
// odd-multiples tables of the resident warps of k_fk20_g1_ntts_vm (one block per warp slot of the persistent grid)
// A caller that knows the device is busy with other batches anyway (the coalescer with batches in flight) asks for the kernel with
// the least work instead of the shortest dependency chain: the radix-4 form does 25 % more multiplications.
static thread_local bool t_k5_prefer_throughput = false;
void set_k5_throughput_hint(bool on) { t_k5_prefer_throughput = on; }
constexpr int R4_MAX_BLOBS = 256;      // the product scratch of the radix-4 form is sized for this many blobs
static int k5_r4_max() {
    // batches up to this many blobs take the radix-4 kernel (EKZG_K5_R4_MAX; 0 switches it off)
    const char* e = getenv("EKZG_K5_R4_MAX");
    const int v = e ? atoi(e) : 256;   // measured (tools/k5_sweep.py, profiles/r2_i_k5_sweep.jsonl): 10.2 against 17.2 ms up to 64 blobs, 15.3 against 17.2 at 256
    return v < 0 ? 0 : (v > R4_MAX_BLOBS ? R4_MAX_BLOBS : v);
}
static int k5_coop_max() {
    // batches up to this many blobs run their multiplication units cooperatively, four lanes per field element (EKZG_K5_COOP_MAX; 0 = never)
    const char* e = getenv("EKZG_K5_COOP_MAX");
    const int v = e ? atoi(e) : 80;   // measured (tools/k5_sweep.py, profiles/r2_coop_k5_sweep.jsonl): K5 5.4 against 10.2 ms up to 16 blobs, 7.2 at 32, 8.5 at 64, 10.8 against 10.2 at 96
    return v < 0 ? 0 : (v > R4_MAX_BLOBS ? R4_MAX_BLOBS : v);
}
size_t g1_ntt_scratch_bytes() {
    if (ntt_query_sms() != cudaSuccess) return 0;
    return std::max((size_t)g_ntt_sms * K5_VM_CTAS_PER_SM * (fpvm::NT / 32) * K5_SCRATCH_WARP_BYTES,
                    (size_t)R4_TMP_POINTS * R4_MAX_BLOBS * sizeof(G1Jac));
}

// phases [ph0, ph1) of the two transforms over pts[128][B]; queue: g1_ntt_queue_words(B) words, scratch: g1_ntt_scratch_bytes()
cudaError_t launch_g1_ntt_phases(G1Jac* pts, int B, int ph0, int ph1, uint32_t* queue, void* scratch, cudaStream_t st) {
    cudaError_t e = ntt_query_sms();
    if (e != cudaSuccess) return e;
    const int G = (B + 31) / 32;
    e = cudaMemsetAsync(queue, 0, g1_ntt_queue_words(B) * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    const long units = (long)G * 64;                                   // warps that can run at once
    unsigned* q = reinterpret_cast<unsigned*>(queue);
    // latency mode (the memset above covers its 1 + 14 G counters); a phase range [0, 2k) is its first k super-phases (test hook)
    if (ph0 == 0 && (ph1 & 1) == 0 && ph1 >= 2 && ph1 <= NTT_PHASES && scratch && B <= k5_r4_max() && !(t_k5_prefer_throughput && B > 64)) {
        if (B <= k5_coop_max() && !t_k5_prefer_throughput) {   // cooperative multiplication units (40 % less throughput: not beside other batches): 8 blobs per warp (the queue holds 1 + 14 ceil(B/8) counters)
            const int G8 = (B + 7) / 8;
            const int grid = (int)std::min<long>((long)g_ntt_sms * 2, ((long)G8 * 160 + NTT_THREADS / 32 - 1) / (NTT_THREADS / 32));
            k_fk20_g1_ntts_r4<8><<<grid, NTT_THREADS, 0, st>>>(pts, reinterpret_cast<G1Jac*>(scratch), B, G8, ph1 / 2, q);
            EKZG_LAUNCH_CHECK();
            return cudaSuccess;
        }
        const int grid = (int)std::min<long>((long)g_ntt_sms * 2, ((long)G * 160 + NTT_THREADS / 32 - 1) / (NTT_THREADS / 32));
        k_fk20_g1_ntts_r4<32><<<grid, NTT_THREADS, 0, st>>>(pts, reinterpret_cast<G1Jac*>(scratch), B, G, ph1 / 2, q);
        EKZG_LAUNCH_CHECK();
        return cudaSuccess;
    }
    if (!k5_register_form()) {
        const int grid = (int)std::min<long>((long)g_ntt_sms * K5_VM_CTAS_PER_SM, (units + fpvm::NT / 32 - 1) / (fpvm::NT / 32));
        k_fk20_g1_ntts_vm<<<grid, fpvm::NT, fpvm::SMEM_BYTES, st>>>(pts, B, G, ph0, ph1, q, reinterpret_cast<uint4*>(scratch));
        EKZG_LAUNCH_CHECK();
        return cudaSuccess;
    }
    const int mb = ntt_min_blocks();
    const int grid = (int)std::min<long>((long)g_ntt_sms * mb, (units + NTT_THREADS / 32 - 1) / (NTT_THREADS / 32));
    if (mb == 2) k_fk20_g1_ntts<2><<<grid, NTT_THREADS, 0, st>>>(pts, B, G, ph0, ph1, q);
    else if (mb == 3) k_fk20_g1_ntts<3><<<grid, NTT_THREADS, 0, st>>>(pts, B, G, ph0, ph1, q);
    else k_fk20_g1_ntts<4><<<grid, NTT_THREADS, 0, st>>>(pts, B, G, ph0, ph1, q);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_fk20_g1_ntts(G1Jac* pts, int B, uint32_t* queue, void* scratch, cudaStream_t st) {
    return launch_g1_ntt_phases(pts, B, 0, NTT_PHASES, queue, scratch, st);
}

cudaError_t launch_g1_compress(const G1Jac* pts, uint8_t* out, int npos, int B, cudaStream_t st) {
    int n = npos * B;
    if (npos % K6_CH == 0 && n >= 32768) {   // below that both variants are latency-bound
        n /= K6_CH;
        k_g1_compress_batched<<<(n + 127) / 128, 128, 0, st>>>(pts, out, npos, B);
    } else {
        k_g1_compress<<<(n + 127) / 128, 128, 0, st>>>(pts, out, npos, B);
    }
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_g1_decompress(const uint8_t* in, G1Affine* out, uint32_t* status, int n, cudaStream_t st) {
    k_g1_decompress<<<(n + 63) / 64, 64, 0, st>>>(in, out, status, n);
    EKZG_LAUNCH_CHECK();
    return cudaSuccess;
}

static cudaError_t fill_table(const G1Jac* pts, const G1Affine* aff, int npoints, G1Affine* qaff, G1Affine* table, const MsmTable& T, cudaStream_t st) {
    if (T.nw > MAX_NW) return cudaErrorInvalidValue;
    k_fk20_window_bases<<<(npoints + 63) / 64, 64, 0, st>>>(pts, aff, qaff, T.w, T.nw, npoints);
    EKZG_LAUNCH_CHECK();
    size_t nbases = (size_t)npoints * T.nw;
    int chunks = (T.half + TBL_CH - 1) / TBL_CH;
    size_t nthreads = nbases * chunks;
    k_fk20_table_fill<<<(unsigned)((nthreads + 127) / 128), 128, 0, st>>>(qaff, table, T.half, nbases);
    EKZG_LAUNCH_CHECK();
    if (T.mg > 1) {
        if (npoints % T.mg) return cudaErrorInvalidValue;
        int ncomb = 1;
        for (int i = 0; i < T.mg; i++) ncomb *= T.rtop;
        const size_t ngroups = (size_t)npoints / T.mg, n = ngroups * (size_t)(ncomb - 1);
        k_fk20_top_merge_fill<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(qaff, table, T.nw, T.half, T.rtop, T.mg, ncomb, ngroups);
        EKZG_LAUNCH_CHECK();
    }
    return cudaSuccess;
}

cudaError_t launch_fk20_setup(const G1Affine* srs, G1Jac* pts_scratch /*128*64*/, G1Affine* qaff /*8192*nw*/, G1Affine* table,
                              const DevTables& T, uint32_t* queue /*g1_ntt_queue_words(64)*/, void* ntt_scratch, cudaStream_t st) {
    k_fk20_setup_vectors<<<(128 * 64 + 127) / 128, 128, 0, st>>>(srs, pts_scratch);
    EKZG_LAUNCH_CHECK();
    // F_k = NTT_128(V_k || O^64) for the 64 vectors at once: the forward half of K5 with "blob" := k
    cudaError_t e = launch_g1_ntt_phases(pts_scratch, 64, 7, NTT_PHASES, queue, ntt_scratch, st);
    if (e != cudaSuccess) return e;
    return fill_table(pts_scratch, nullptr, FK20_MSMS * FK20_POINTS, qaff, table, T.fk20, st);
}

cudaError_t launch_srs_table_setup(const G1Affine* srs, int npoints, G1Affine* qaff, G1Affine* table, const MsmTable& T, cudaStream_t st) {
    return fill_table(nullptr, srs, npoints, qaff, table, T, st);
}

}  // namespace ekzg
