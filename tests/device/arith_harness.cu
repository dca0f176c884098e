// Device test harness: the field and curve routines of csrc/ compiled for sm_100a with the flags of the library and called
// the way the kernels call them, exported for ctypes.  tests/test_host_emu.py runs its cases a second time through the emu_*
// functions below; tests/test_gpu_device_arith.py checks what only the device has (the warp-cooperative arithmetic of
// g1_coop.cuh and the shared-memory slots of the Fp interpreter).  Test scaffolding only.
//
// Every call copies its host buffers in (cudaMalloc + cudaMemcpy), launches one kernel, synchronises, copies the results back
// and frees its buffers.  The emu_* functions keep the signatures of tests/host_emu/{emu_field,emu_g1}.cpp, and some of those
// return a result rather than a status, so every call also records its CUDA status: harness_error() returns the first error.
// After an error no call launches anything again.
#include "g1_coop.cuh"
#include "fp_inv_gcd.cuh"
#include "fpvm.cuh"
#include <string.h>
using namespace ekzg;

__constant__ uint32_t c_fpvm_prog[fpvm::FPVM_PROG_WORDS] = FPVM_PROG_INIT;
__constant__ uint16_t c_twiddle_ops[128][MULOPS_STRIDE] =
#include "twiddle_ops.inc"
    ;

static cudaError_t g_err = cudaSuccess;

static cudaError_t note(cudaError_t e) {
    if (g_err == cudaSuccess) g_err = e;
    return e;
}

// ---- one item per launch, one thread: the arguments travel as one struct, copied in and back whole ----------------------------
template <class A, void (*F)(A&)>
__global__ void one_item(A* a) { F(*a); }

template <class A, void (*F)(A&)>
static int run_one(A& a) {
    if (g_err != cudaSuccess) return (int)g_err;
    A* d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(A));
    if (e == cudaSuccess) e = cudaMemcpy(d, &a, sizeof(A), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) { one_item<A, F><<<1, 1>>>(d); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(&a, d, sizeof(A), cudaMemcpyDeviceToHost);
    if (d) cudaFree(d);
    return (int)note(e);
}

struct FpArgs { Fp a, b, c, d, r; int ret; };
struct FrArgs { Fr a, b, r; int ret; };
// on the device fe_mul / fe_sqr / fp_mul2_add of Fp are the __noinline__ by-value calls fp_mul_call / fp_sqr_call / fp_mul2_call
__device__ void d_fp_mul(FpArgs& x) { fe_mul(x.r, x.a, x.b); }
__device__ void d_fp_sqr(FpArgs& x) { fe_sqr(x.r, x.a); }
__device__ void d_fp_mul2(FpArgs& x) { fp_mul2_add(x.r, x.a, x.b, x.c, x.d); }
__device__ void d_fp_add(FpArgs& x) { fe_add(x.r, x.a, x.b); }
__device__ void d_fp_sub(FpArgs& x) { fe_sub(x.r, x.a, x.b); }
__device__ void d_fp_neg(FpArgs& x) { fe_neg(x.r, x.a); }
__device__ void d_fp_inv(FpArgs& x) { fp_inv(x.r, x.a); }
__device__ void d_fp_inv_gcd(FpArgs& x) { fp_inv_gcd(x.r, x.a); }
__device__ void d_fp_gt_half(FpArgs& x) { x.ret = fe_plain_gt_half(x.a); }
__device__ void d_fr_mul(FrArgs& x) { fe_mul(x.r, x.a, x.b); }
__device__ void d_fr_sqr(FrArgs& x) { fe_sqr(x.r, x.a); }
__device__ void d_fr_add(FrArgs& x) { fe_add(x.r, x.a, x.b); }
__device__ void d_fr_sub(FrArgs& x) { fe_sub(x.r, x.a, x.b); }
__device__ void d_fr_inv(FrArgs& x) { fr_inv(x.r, x.a); }
__device__ void d_fr_ge_mod(FrArgs& x) { x.ret = fe_plain_ge_mod(x.a); }

template <void (*F)(FpArgs&)>
static int fp_op(const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* r) {
    FpArgs x;
    memset(&x, 0, sizeof(x));
    if (a) memcpy(x.a.v, a, 48);
    if (b) memcpy(x.b.v, b, 48);
    if (c) memcpy(x.c.v, c, 48);
    if (d) memcpy(x.d.v, d, 48);
    run_one<FpArgs, F>(x);
    if (r) memcpy(r, x.r.v, 48);
    return x.ret;
}
template <void (*F)(FrArgs&)>
static int fr_op(const uint32_t* a, const uint32_t* b, uint32_t* r) {
    FrArgs x;
    memset(&x, 0, sizeof(x));
    if (a) memcpy(x.a.v, a, 32);
    if (b) memcpy(x.b.v, b, 32);
    run_one<FrArgs, F>(x);
    if (r) memcpy(r, x.r.v, 32);
    return x.ret;
}

// ---- curve: the bodies of tests/host_emu/emu_g1.cpp, on the device ---------------------------------------------------------
__device__ void to_affine(G1Affine& a, const G1Jac& j) {
    if (jac_is_inf(j)) { g1a_set_inf(a); return; }
    Fp zi; fp_inv(zi, j.z);
    jac_to_affine_with_inv(a, j, zi);
}
__device__ void out48(uint8_t* out, const G1Jac& j) { G1Affine a; to_affine(a, j); g1a_compress(out, a); }
__device__ void out48x(uint8_t* out, const G1Xyzz& p) { G1Jac j; jac_from_xyzz(j, p); out48(out, j); }

constexpr int CHAIN_MAX = 16;
struct G1Args {
    int op, n, e, ret;
    uint8_t p[CHAIN_MAX * 48], q[48], negs[CHAIN_MAX], out[48];
    uint32_t k[8];
    int8_t digits[66];
};

__device__ void d_decompress_roundtrip(G1Args& x) {
    G1Affine a;
    x.ret = g1a_decompress(a, x.p);
    if (x.ret) return;
    if (!g1a_is_inf(a) && !g1a_on_curve(a)) { x.ret = 2; return; }
    g1a_compress(x.out, a);
}
// op: 0 xyzz_madd(P,+Q) 1 xyzz_madd(P,-Q) 2 xyzz_add 3 jac_add 4 jac_madd(+) 5 jac_madd(-) 6 jac_dbl(P) 7 xyzz_dbl(P)
__device__ void d_binop(G1Args& x) {
    G1Affine p, q;
    if (g1a_decompress(p, x.p) || g1a_decompress(q, x.q)) { x.ret = 1; return; }
    G1Xyzz xp, xq; xyzz_from_affine(xp, p); xyzz_from_affine(xq, q);
    G1Jac jp, jq; jac_from_affine(jp, p); jac_from_affine(jq, q);
    x.ret = 0;
    switch (x.op) {
        case 0: xyzz_madd(xp, q, false); out48x(x.out, xp); break;
        case 1: xyzz_madd(xp, q, true); out48x(x.out, xp); break;
        case 2: xyzz_add(xp, xq); out48x(x.out, xp); break;
        case 3: jac_add(jp, jq); out48(x.out, jp); break;
        case 4: jac_madd(jp, q, false); out48(x.out, jp); break;
        case 5: jac_madd(jp, q, true); out48(x.out, jp); break;
        case 6: { G1Jac d; jac_dbl(d, jp); out48(x.out, d); break; }
        case 7: { G1Xyzz d; xyzz_dbl(d, xp); out48x(x.out, d); break; }
        default: x.ret = 3;
    }
}
// mode 0: xyzz_madd chain; 1: jac_madd chain; 2: xyzz_add of two half-chains; 3: jac_add of two half-chains
__device__ void d_chain(G1Args& x) {
    G1Xyzz xa, xb; xyzz_set_inf(xa); xyzz_set_inf(xb);
    G1Jac ja, jb; jac_set_inf(ja); jac_set_inf(jb);
    const int mode = x.op, n = x.n;
    for (int i = 0; i < n; i++) {
        G1Affine p;
        if (g1a_decompress(p, x.p + 48 * i)) { x.ret = 1; return; }
        const bool second = (i >= n / 2), neg = x.negs[i] != 0;
        if (mode == 0) xyzz_madd(xa, p, neg);
        else if (mode == 1) jac_madd(ja, p, neg);
        else if (mode == 2) xyzz_madd(second ? xb : xa, p, neg);
        else jac_madd(second ? jb : ja, p, neg);
    }
    if (mode == 0) out48x(x.out, xa);
    else if (mode == 1) out48(x.out, ja);
    else if (mode == 2) { xyzz_add(xa, xb); out48x(x.out, xa); }
    else { jac_add(ja, jb); out48(x.out, ja); }
    x.ret = 0;
}
// 0 jac_mul_u256(P), 1 jac_mul_fr_glv(2P), 2 jac_mul_glv16(2P, digits), 3 jac_mul_ops(2P, twiddle row e): the last three start
// from a point with Z != 1, the Python side accounts for the factor 2
__device__ void d_scalar_mul(G1Args& x) {
    G1Affine p;
    if (g1a_decompress(p, x.p)) { x.ret = 1; return; }
    G1Jac j, r;
    jac_from_affine(j, p);
    if (x.op) jac_dbl(j, j);
    if (x.op == 0) jac_mul_u256(r, j, x.k);
    else if (x.op == 1) jac_mul_fr_glv(r, j, x.k);
    else if (x.op == 2) jac_mul_glv16(r, j, x.digits);
    else jac_mul_ops(r, j, c_twiddle_ops[x.e & 127]);
    out48(x.out, r);
    x.ret = 0;
}
__device__ void d_in_subgroup(G1Args& x) {
    G1Affine p;
    if (g1a_decompress(p, x.p)) { x.ret = -1; return; }
    x.ret = g1a_is_inf(p) ? 1 : g1a_in_subgroup(p) ? 1 : 0;
}
__device__ void d_booth(G1Args& x) { x.ret = booth_digit(x.k, x.e, x.n); }

template <void (*F)(G1Args&)>
static int g1_op(G1Args& x, uint8_t* out) {
    run_one<G1Args, F>(x);
    if (out) memcpy(out, x.out, 48);
    return x.ret;
}
static G1Args g1_args(const uint8_t* p, int np) {
    G1Args x;
    memset(&x, 0, sizeof(x));
    x.ret = -100;       // what a call that never ran returns (harness_error() says why)
    if (p) memcpy(x.p, p, 48 * np);
    return x;
}

extern "C" {
int harness_error() { return (int)g_err; }
const char* harness_error_name(int e) { return cudaGetErrorName((cudaError_t)e); }

// ---- tests/host_emu/emu_field.cpp on the device: Fp products through fp_mul_call / fp_sqr_call / fp_mul2_call ----------------
void emu_fp_mul(const uint32_t* a, const uint32_t* b, uint32_t* r) { fp_op<d_fp_mul>(a, b, nullptr, nullptr, r); }
void emu_fp_sqr(const uint32_t* a, uint32_t* r) { fp_op<d_fp_sqr>(a, nullptr, nullptr, nullptr, r); }
void emu_fp_mul2(const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* r) { fp_op<d_fp_mul2>(a, b, c, d, r); }
void emu_fp_add(const uint32_t* a, const uint32_t* b, uint32_t* r) { fp_op<d_fp_add>(a, b, nullptr, nullptr, r); }
void emu_fp_sub(const uint32_t* a, const uint32_t* b, uint32_t* r) { fp_op<d_fp_sub>(a, b, nullptr, nullptr, r); }
void emu_fp_neg(const uint32_t* a, uint32_t* r) { fp_op<d_fp_neg>(a, nullptr, nullptr, nullptr, r); }
void emu_fp_inv(const uint32_t* a, uint32_t* r) { fp_op<d_fp_inv>(a, nullptr, nullptr, nullptr, r); }
void emu_fp_inv_gcd(const uint32_t* a, uint32_t* r) { fp_op<d_fp_inv_gcd>(a, nullptr, nullptr, nullptr, r); }
int emu_fp_gt_half(const uint32_t* a) { return fp_op<d_fp_gt_half>(a, nullptr, nullptr, nullptr, nullptr); }
void emu_fr_mul(const uint32_t* a, const uint32_t* b, uint32_t* r) { fr_op<d_fr_mul>(a, b, r); }
void emu_fr_sqr(const uint32_t* a, uint32_t* r) { fr_op<d_fr_sqr>(a, nullptr, r); }
void emu_fr_add(const uint32_t* a, const uint32_t* b, uint32_t* r) { fr_op<d_fr_add>(a, b, r); }
void emu_fr_sub(const uint32_t* a, const uint32_t* b, uint32_t* r) { fr_op<d_fr_sub>(a, b, r); }
void emu_fr_inv(const uint32_t* a, uint32_t* r) { fr_op<d_fr_inv>(a, nullptr, r); }
int emu_fr_ge_mod(const uint32_t* a) { return fr_op<d_fr_ge_mod>(a, nullptr, nullptr); }

// ---- tests/host_emu/emu_g1.cpp on the device ------------------------------------------------------------------------------------
int emu_g1_decompress_roundtrip(const uint8_t* in, uint8_t* out) {
    G1Args x = g1_args(in, 1);
    const int rc = g1_op<d_decompress_roundtrip>(x, nullptr);
    if (rc == 0) memcpy(out, x.out, 48);
    return rc;
}
int emu_g1_binop(int op, const uint8_t* p48, const uint8_t* q48, uint8_t* out) {
    G1Args x = g1_args(p48, 1);
    memcpy(x.q, q48, 48);
    x.op = op;
    return g1_op<d_binop>(x, out);
}
int emu_g1_chain(int mode, int n, const uint8_t* pts48, const uint8_t* negs, uint8_t* out) {
    if (n < 0 || n > CHAIN_MAX) return 4;
    G1Args x = g1_args(pts48, n);
    memcpy(x.negs, negs, n);
    x.op = mode;
    x.n = n;
    return g1_op<d_chain>(x, out);
}
int emu_g1_mul_u256(const uint8_t* p48, const uint32_t* k, uint8_t* out) {
    G1Args x = g1_args(p48, 1);
    memcpy(x.k, k, 32);
    return g1_op<d_scalar_mul>(x, out);
}
int emu_g1_mul_fr_glv(const uint8_t* p48, const uint32_t* k, uint8_t* out) {
    G1Args x = g1_args(p48, 1);
    memcpy(x.k, k, 32);
    x.op = 1;
    return g1_op<d_scalar_mul>(x, out);
}
int emu_g1_mul_twiddle(const uint8_t* p48, int e, uint8_t* out) {
    if (e < 0 || e >= 128) return 4;
    G1Args x = g1_args(p48, 1);
    memcpy(x.digits, GLV_TWIDDLE_DIGITS_HOST[e], 66);
    x.op = 2;
    return g1_op<d_scalar_mul>(x, out);
}
int emu_g1_mul_twiddle_ops(const uint8_t* p48, int e, uint8_t* out) {
    if (e < 0 || e >= 128) return 4;
    G1Args x = g1_args(p48, 1);
    x.op = 3;
    x.e = e;
    return g1_op<d_scalar_mul>(x, out);
}
int emu_g1_in_subgroup(const uint8_t* p48) {
    G1Args x = g1_args(p48, 1);
    return g1_op<d_in_subgroup>(x, nullptr);
}
int emu_booth_digit(const uint32_t* s, int t, int w) {
    G1Args x = g1_args(nullptr, 0);
    memcpy(x.k, s, 32);
    x.e = t;
    x.n = w;
    return g1_op<d_booth>(x, nullptr);
}
}  // extern "C"

// ---- many items per launch --------------------------------------------------------------------------------------------------------
// device copies of one call's host buffers, freed when the call returns
struct Bufs {
    void* p[8];
    int n = 0;
    cudaError_t e = g_err;
    ~Bufs() { for (int i = 0; i < n; i++) cudaFree(p[i]); }
    template <class T> T* in(const T* h, size_t count) {
        T* d = alloc<T>(count);
        if (e == cudaSuccess) e = cudaMemcpy(d, h, count * sizeof(T), cudaMemcpyHostToDevice);
        return d;
    }
    template <class T> T* alloc(size_t count) {
        void* d = nullptr;
        if (e == cudaSuccess) e = cudaMalloc(&d, count * sizeof(T));
        if (e == cudaSuccess) e = cudaMemset(d, 0, count * sizeof(T));
        if (d) p[n++] = d;
        return (T*)d;
    }
    void launched() {
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    template <class T> void back(T* h, const T* d, size_t count) {
        if (e == cudaSuccess) e = cudaMemcpy(h, d, count * sizeof(T), cudaMemcpyDeviceToHost);
    }
    int done() { return (int)note(e); }
};

// The cooperative routines are made of full-mask shuffles and ballots, so every launch is whole warps of eight four-lane groups
// and every lane runs every routine to the end: groups past the batch work on element 0, and only the stores are guarded.
constexpr int COOP_THREADS = 128;
static int coop_blocks(int n) { return (4 * n + COOP_THREADS - 1) / COOP_THREADS; }

__device__ __forceinline__ Fp ld_fp(const uint32_t* src) {
    Fp r;
#pragma unroll
    for (int j = 0; j < 12; j++) r.v[j] = src[j];
    return r;
}

// op 0 cmul(a, b)  1 cmul2(a, b; c, d)  2 cadd(a, b)  3 csub(a, b)  4 cneg(a)  5 from_fp(a).  Element i is 12 limbs of each input;
// raw[2i], raw[2i + 1]: the lanes' limbs of the (two) results as the routine leaves them, canon[2i], canon[2i + 1]: to_fp of them
__global__ void coop_fp_kernel(int op, int n, const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* raw,
                               uint32_t* canon) {
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 2);
    const bool valid = g < n;
    const int src = valid ? g : 0;
    const coop::Ctx ctx = coop::make_ctx();
    const coop::CFp x = coop::from_fp(ctx, ld_fp(a + 12 * src)), y = coop::from_fp(ctx, ld_fp(b + 12 * src));
    coop::CFp r1 = x, r2 = x;
    if (op == 0) coop::cmul(ctx, r1, x, y);
    else if (op == 1) coop::cmul2(ctx, r1, x, y, r2, coop::from_fp(ctx, ld_fp(c + 12 * src)), coop::from_fp(ctx, ld_fp(d + 12 * src)));
    else if (op == 2) coop::cadd(ctx, r1, x, y);
    else if (op == 3) coop::csub(ctx, r1, x, y);
    else if (op == 4) coop::cneg(ctx, r1, x);
    const Fp o1 = coop::to_fp(ctx, r1), o2 = coop::to_fp(ctx, r2);
    if (valid) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            raw[24 * g + 3 * ctx.gl + k] = r1.v[k];
            raw[24 * g + 12 + 3 * ctx.gl + k] = r2.v[k];
        }
        if (ctx.gl == 0)
#pragma unroll
            for (int j = 0; j < 12; j++) {
                canon[24 * g + j] = o1.v[j];
                canon[24 * g + 12 + j] = o2.v[j];
            }
    }
}

__device__ __forceinline__ G1Jac ld_jac(const uint32_t* src) {
    G1Jac r;
    r.x = ld_fp(src); r.y = ld_fp(src + 12); r.z = ld_fp(src + 24);
    return r;
}
__device__ __forceinline__ void st_jac(uint32_t* dst, const G1Jac& p) {
#pragma unroll
    for (int j = 0; j < 12; j++) { dst[j] = p.x.v[j]; dst[12 + j] = p.y.v[j]; dst[24 + j] = p.z.v[j]; }
}

// op 0 cjac_dbl(P)  1 cjac_madd(P, Q)  2 cjac_madd_zr(P, Q) with zr  3 cjac_mul_ops(P, twiddle row rows[warp])  4 jac_mul_ops, one point
// per thread, the same rows.  P: 36 limbs (X, Y, Z), Q: 24 limbs (affine x, y); out: 36 limbs of the result (to_jac: canonical), zr: 12
__global__ void coop_pt_kernel(int op, int n, const uint32_t* p, const uint32_t* q, const int* rows, uint32_t* out, uint32_t* zr_out) {
    const int t = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (op == 4) {
        if (t < n) {
            G1Jac r;
            jac_mul_ops(r, ld_jac(p + 36 * t), c_twiddle_ops[rows[t / 8]]);
            st_jac(out + 36 * t, r);
        }
        return;
    }
    const int g = t >> 2, w = t >> 5;
    const bool valid = g < n;
    const int src = valid ? g : 0;
    const coop::Ctx ctx = coop::make_ctx();
    const coop::CJac cp = coop::from_jac(ctx, ld_jac(p + 36 * src));
    const coop::CFp qx = coop::from_fp(ctx, ld_fp(q + 24 * src)), qy = coop::from_fp(ctx, ld_fp(q + 24 * src + 12));
    coop::CJac r = cp;
    coop::CFp zr = qx;
    if (op == 0) coop::cjac_dbl(ctx, r, cp, coop::const_fp(ctx, coop::three_halves_limb));
    else if (op == 1) coop::cjac_madd(ctx, r, qx, qy);
    else if (op == 2) coop::cjac_madd_zr(ctx, r, cp, qx, qy, zr);
    else coop::cjac_mul_ops(ctx, r, cp, c_twiddle_ops[w < (n + 7) / 8 ? rows[w] : rows[0]]);   // one op list per warp
    const G1Jac o = coop::to_jac(ctx, r);
    const Fp z = coop::to_fp(ctx, zr);
    if (valid && ctx.gl == 0) {
        st_jac(out + 36 * g, o);
#pragma unroll
        for (int j = 0; j < 12; j++) zr_out[12 * g + j] = z.v[j];
    }
}

// ---- the Fp interpreter over fpvm::Smem, with the run loop of fpvm_run in kzg_kernels.cu --------------------------------------
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

// thread `item` = block * NT + t: its eight slots in and out (12 limbs each, Montgomery form) and the zero mask of instructions
// [pc, pc + len).  Slot s of thread t is the three 16-byte chunks at (s * 3 + q) * QS + t * 16 of the block's shared memory
// (fpvm.cuh); they are filled and read back here by that address arithmetic, not through Smem.
__global__ void fpvm_kernel(int pc, int len, const uint4* in, uint4* out, uint32_t* masks) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int t = threadIdx.x, item = blockIdx.x * fpvm::NT + t;
    for (int s = 0; s < fpvm::NSLOT; s++)
        for (int q = 0; q < 3; q++) *(uint4*)(smem + (s * 3 + q) * fpvm::QS + t * 16) = in[(item * fpvm::NSLOT + s) * 3 + q];
    masks[item] = fpvm_run((uint32_t)__cvta_generic_to_shared(smem) + t * 16, pc, len, 1);
    for (int s = 0; s < fpvm::NSLOT; s++)
        for (int q = 0; q < 3; q++) out[(item * fpvm::NSLOT + s) * 3 + q] = *(const uint4*)(smem + (s * 3 + q) * fpvm::QS + t * 16);
}

static bool rows_ok(const int* rows, int k) {
    for (int i = 0; i < k; i++)
        if (rows[i] <= 0 || rows[i] >= 128 || rows[i] == 64) return false;
    return true;
}

extern "C" {
int harness_device_count() {
    int n = 0;
    return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}
int coop_fp(int op, int n, const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* raw, uint32_t* canon) {
    if (op < 0 || op > 5 || n <= 0) return (int)cudaErrorInvalidValue;
    Bufs m;
    const uint32_t *da = m.in(a, 12 * (size_t)n), *db = m.in(b, 12 * (size_t)n), *dc = m.in(c, 12 * (size_t)n), *dd = m.in(d, 12 * (size_t)n);
    uint32_t *dr = m.alloc<uint32_t>(24 * (size_t)n), *dk = m.alloc<uint32_t>(24 * (size_t)n);
    if (m.e == cudaSuccess) coop_fp_kernel<<<coop_blocks(n), COOP_THREADS>>>(op, n, da, db, dc, dd, dr, dk);
    m.launched();
    m.back(raw, dr, 24 * (size_t)n);
    m.back(canon, dk, 24 * (size_t)n);
    return m.done();
}
// rows: one twiddle row per eight points (ops 3 and 4), each in 1..63 or 65..127 -- the rows cjac_mul_ops is used with
int coop_pt(int op, int n, const uint32_t* p, const uint32_t* q, const int* rows, uint32_t* out, uint32_t* zr) {
    const int nrows = (n + 7) / 8;
    if (op < 0 || op > 4 || n <= 0 || ((op == 3 || op == 4) && !rows_ok(rows, nrows))) return (int)cudaErrorInvalidValue;
    Bufs m;
    const uint32_t *dp = m.in(p, 36 * (size_t)n), *dq = m.in(q, 24 * (size_t)n);
    const int* dw = m.in(rows, (size_t)nrows);
    uint32_t *dout = m.alloc<uint32_t>(36 * (size_t)n), *dz = m.alloc<uint32_t>(12 * (size_t)n);
    if (m.e == cudaSuccess) coop_pt_kernel<<<op == 4 ? (n + 127) / 128 : coop_blocks(n), COOP_THREADS>>>(op, n, dp, dq, dw, dout, dz);
    m.launched();
    m.back(out, dout, 36 * (size_t)n);
    m.back(zr, dz, 12 * (size_t)n);
    return m.done();
}
int fpvm_words() { return fpvm::FPVM_PROG_WORDS; }
// nthreads: a multiple of the NT threads of a CTA; slots: nthreads x 8 x 12 limbs in and out; masks: nthreads
int fpvm_smem_run(int pc, int len, int nthreads, uint32_t* slots, uint32_t* masks) {
    if (pc < 0 || len <= 0 || len > 32 || pc + len > fpvm::FPVM_PROG_WORDS || nthreads <= 0 || nthreads % fpvm::NT) return (int)cudaErrorInvalidValue;
    const size_t words = (size_t)nthreads * fpvm::NSLOT * 12;
    Bufs m;
    const uint4* din = m.in((const uint4*)slots, words / 4);
    uint4* dout = m.alloc<uint4>(words / 4);
    uint32_t* dm = m.alloc<uint32_t>(nthreads);
    if (m.e == cudaSuccess) fpvm_kernel<<<nthreads / fpvm::NT, fpvm::NT, fpvm::SMEM_BYTES>>>(pc, len, din, dout, dm);
    m.launched();
    m.back((uint4*)slots, dout, words / 4);
    m.back(masks, dm, (size_t)nthreads);
    return m.done();
}
}  // extern "C"
