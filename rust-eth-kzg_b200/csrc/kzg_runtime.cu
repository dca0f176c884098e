// Host runtime of the B200 KZG backend (see kzg_runtime.h).
#include "kzg_runtime.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <cstring>
#include "fr_consts.cuh"
#include "host_sha256.h"

// The ceremony output (crates/trusted_setup/data/trusted_setup_4096.json, repacked by
// tools/convert_trusted_setup.py) is linked into the library, like the reference embeds its JSON
// (crates/trusted_setup/src/lib.rs:5).
extern "C" {
extern const unsigned char ekzg_trusted_setup_start[];
extern const unsigned char ekzg_trusted_setup_end[];
}

namespace ekzg {

double TraceClock::now() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
TraceClock::TraceClock(const char* w) : what(w) {
    static const bool enabled = getenv("EKZG_TRACE") != nullptr;
    on = enabled;
    t0 = on ? now() : 0;
}
void TraceClock::mark(const char* phase) {
    if (!on) return;
    double t = now();
    fprintf(stderr, "[ekzg trace] %s: %s %.3f ms\n", what, phase, t - t0);
    t0 = t;
}

void host_blob_challenge(const uint8_t* blob, const uint8_t* commitment48, uint8_t z_be[32]) {
    host::Sha256Stream h;
    uint8_t head[32] = {0};
    memcpy(head, "FSBLOBVERIFY_V1_", 16);
    head[30] = 0x10;                      // u128_be(4096)
    h.update(head, 32);
    h.update(blob, BYTES_PER_BLOB);
    h.update(commitment48, 48);
    uint8_t d[32];
    h.final(d);
    // reduce below r (2^256 < 3 r: at most two subtractions)
    static const uint64_t R[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
    uint64_t v[4];
    for (int i = 0; i < 4; i++) {
        uint64_t x = 0;
        for (int b = 0; b < 8; b++) x = (x << 8) | d[8 * (3 - i) + b];
        v[i] = x;
    }
    for (int it = 0; it < 2; it++) {
        bool ge = true;
        for (int i = 3; i >= 0; i--) {
            if (v[i] != R[i]) { ge = v[i] > R[i]; break; }
        }
        if (!ge) break;
        unsigned __int128 br = 0;
        for (int i = 0; i < 4; i++) {
            const unsigned __int128 t = (unsigned __int128)v[i] - R[i] - (uint64_t)br;
            v[i] = (uint64_t)t;
            br = (t >> 64) & 1;
        }
    }
    for (int i = 0; i < 4; i++)
        for (int b = 0; b < 8; b++) z_be[8 * (3 - i) + b] = (uint8_t)(v[i] >> (8 * (7 - b)));
}

static int direct_proofs_max() {
    const char* e = getenv("EKZG_DIRECT_MAX");
    const int v = e ? atoi(e) : 1;   // two blobs: 8.2 ms direct against 7.0 ms through FK20 with the cooperative G1 NTTs (profiles/r2_latency_sweep.jsonl)
    return v < 0 ? 0 : (v > 8 ? 8 : v);
}

ProofRoute proof_route(uint64_t n, int fk20_capacity, bool eligible) {
    if (eligible && n <= (uint64_t)direct_proofs_max()) return {true, N_CELLS * (int)n};
    return {false, fk20_capacity};
}

const char* item_status_text(uint8_t code, bool cells, bool z) {
    if (code == ITEM_NON_CANONICAL && cells) return "Serialization(ScalarNotCanonical): a cell field element is >= the scalar modulus";
    if (code == ITEM_NON_CANONICAL) return "Serialization(ScalarNotCanonical): a blob field element is >= the BLS12-381 scalar modulus";
    if (code == ITEM_BAD_AUX && z) return "Serialization(ScalarNotCanonical): z is >= the BLS12-381 scalar modulus";
    if (code == ITEM_BAD_AUX) return "Serialization(G1PointInvalid): commitment is not a valid compressed G1 point in the prime-order subgroup";
    if (code == ITEM_BAD_DEGREE) return "ReedSolomon(PolynomialHasInvalidLength): recovered polynomial has degree >= 4096";
    return "Recovery: invalid cell indices";
}

int chunk_capacity() {
    const char* e = getenv("EKZG_CHUNK");
    int c = e ? atoi(e) : 1024;
    if (c < 1) c = 1;
    if (c > 4096) c = 4096;
    return c;
}

// ------------------------------------------------------------------------------------------------
Status Workspace::alloc(int cap, bool with_io, size_t msm_scratch_bytes) {
    capacity = cap;
    EKZG_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    EKZG_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    EKZG_CUDA(cudaStreamCreateWithFlags(&in_stream, cudaStreamNonBlocking));
    EKZG_CUDA(cudaStreamCreateWithFlags(&aux_stream, cudaStreamNonBlocking));
    EKZG_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    for (auto& e : piece_in) EKZG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (int i = 0; i < MAX_SUB; i++) {
        EKZG_CUDA(cudaEventCreateWithFlags(&sub_ready[i], cudaEventDisableTiming));
        EKZG_CUDA(cudaEventCreateWithFlags(&sub_out[i], cudaEventDisableTiming));
    }
    EKZG_CUDA(cudaMalloc(&d_coeffs, (size_t)cap * N_BLOB * sizeof(Fr)));
    EKZG_CUDA(cudaMalloc(&d_scalars, (size_t)cap * FK20_MSMS * FK20_POINTS * 32));
    EKZG_CUDA(cudaMalloc(&d_pts, (size_t)cap * 128 * sizeof(G1Jac)));
    EKZG_CUDA(cudaMalloc(&d_queue, g1_ntt_queue_words(cap) * sizeof(uint32_t)));
    EKZG_CUDA(cudaMalloc(&d_ntt_scratch, g1_ntt_scratch_bytes()));
    if (msm_scratch_bytes) EKZG_CUDA(cudaMalloc(&d_msm_scratch, msm_scratch_bytes));
    if (with_io) {
        EKZG_CUDA(cudaMalloc(&d_blobs, (size_t)cap * BYTES_PER_BLOB));
        EKZG_CUDA(cudaMalloc(&d_cells, (size_t)cap * N_EXT * 32));
        EKZG_CUDA(cudaMalloc(&d_proofs, (size_t)cap * N_CELLS * BYTES_PER_G1));
        EKZG_CUDA(cudaMalloc(&d_status, (size_t)cap * sizeof(uint32_t)));
        EKZG_CUDA(cudaMalloc(&d_c48, (size_t)cap * 48));
        EKZG_CUDA(cudaMalloc(&d_z32, (size_t)cap * 32));
        EKZG_CUDA(cudaMalloc(&d_out48, (size_t)cap * 48));
        EKZG_CUDA(cudaMalloc(&d_z, (size_t)cap * sizeof(Fr)));
        EKZG_CUDA(cudaMalloc(&d_aff, (size_t)cap * sizeof(G1Affine)));
        EKZG_CUDA(cudaMalloc(&d_status2, (size_t)cap * sizeof(uint32_t)));
        EKZG_CUDA(cudaMallocHost(&h_blobs, (size_t)cap * BYTES_PER_BLOB));
        EKZG_CUDA(cudaMallocHost(&h_cells, (size_t)cap * N_EXT * 32));
        EKZG_CUDA(cudaMallocHost(&h_proofs, (size_t)cap * N_CELLS * BYTES_PER_G1));
        EKZG_CUDA(cudaMallocHost(&h_status, (size_t)cap * sizeof(uint32_t)));
    }
    return Status::Ok();
}

Status Workspace::ensure_recover_buffers() {
    if (recover_ready) return Status::Ok();
    auto all = [&]() -> Status {
        EKZG_CUDA(cudaMalloc(&d_rcells, (size_t)capacity * N_CELLS * BYTES_PER_CELL));
        EKZG_CUDA(cudaMallocHost(&h_rcells, (size_t)capacity * N_CELLS * BYTES_PER_CELL));
        EKZG_CUDA(cudaMalloc(&d_slotmap, (size_t)capacity * 128 * sizeof(int16_t)));
        EKZG_CUDA(cudaMallocHost(&h_slotmap, (size_t)capacity * 128 * sizeof(int16_t)));
        EKZG_CUDA(cudaMalloc(&d_ze, (size_t)capacity * 128 * sizeof(Fr)));
        EKZG_CUDA(cudaMalloc(&d_czinv, (size_t)capacity * 128 * sizeof(Fr)));
        EKZG_CUDA(cudaMalloc(&d_cell_off, (size_t)capacity * sizeof(uint32_t)));
        EKZG_CUDA(cudaMallocHost(&h_cell_off, (size_t)capacity * sizeof(uint32_t)));
        return Status::Ok();
    };
    Status s = all();
    if (!s.ok) {   // all or none: a half-built set must never be seen by the next borrower of this workspace
        free_recover_buffers();
        cudaGetLastError();
        return s;
    }
    recover_ready = true;
    return Status::Ok();
}

void Workspace::free_recover_buffers() {
    cudaFree(d_rcells); cudaFreeHost(h_rcells); cudaFree(d_slotmap); cudaFreeHost(h_slotmap); cudaFree(d_ze); cudaFree(d_czinv);
    cudaFree(d_cell_off); cudaFreeHost(h_cell_off);
    d_rcells = nullptr; h_rcells = nullptr; d_slotmap = nullptr; h_slotmap = nullptr; d_ze = nullptr; d_czinv = nullptr;
    d_cell_off = nullptr; h_cell_off = nullptr;
}

Status Workspace::ensure_verify_buffers(int blobs) {
    if (verify_capacity >= blobs) return Status::Ok();
    free_verify_buffers();   // (idle: the workspace is borrowed by one call at a time, and its last user synchronised it)
    auto all = [&]() -> Status {
        EKZG_CUDA(cudaMalloc(&d_given_proofs, (size_t)blobs * PROOFS_PER_BLOB));
        EKZG_CUDA(cudaMalloc(&d_cell_mm, (size_t)blobs * (N_CELLS + 1)));
        EKZG_CUDA(cudaMallocHost(&h_cell_mm, (size_t)blobs * (N_CELLS + 1)));
        EKZG_CUDA(cudaMallocHost(&h_c48, (size_t)blobs * BYTES_PER_G1));
        return Status::Ok();
    };
    Status s = all();
    if (!s.ok) {   // all or none, as the recovery buffers
        free_verify_buffers();
        cudaGetLastError();
        return s;
    }
    d_blob_mm = d_cell_mm + (size_t)blobs * N_CELLS;
    h_blob_mm = h_cell_mm + (size_t)blobs * N_CELLS;
    verify_capacity = blobs;
    return Status::Ok();
}

void Workspace::free_verify_buffers() {
    cudaFree(d_given_proofs); cudaFree(d_cell_mm); cudaFreeHost(h_cell_mm); cudaFreeHost(h_c48);
    d_given_proofs = nullptr; d_cell_mm = nullptr; d_blob_mm = nullptr; h_cell_mm = nullptr; h_blob_mm = nullptr; h_c48 = nullptr;
    verify_capacity = 0;
}

void Workspace::synchronize() const {
    for (cudaStream_t s : {stream, copy_stream, in_stream, aux_stream}) cudaStreamSynchronize(s);
}

void Workspace::release() {
    free_recover_buffers();
    free_verify_buffers();
    cudaFree(d_c48); cudaFree(d_z32); cudaFree(d_out48); cudaFree(d_z); cudaFree(d_aff); cudaFree(d_status2);
    cudaFree(d_blobs); cudaFree(d_coeffs); cudaFree(d_cells); cudaFree(d_scalars); cudaFree(d_pts); cudaFree(d_queue); cudaFree(d_ntt_scratch); cudaFree(d_msm_scratch); cudaFree(d_proofs); cudaFree(d_status);
    cudaFreeHost(h_blobs); cudaFreeHost(h_cells); cudaFreeHost(h_proofs); cudaFreeHost(h_status);
    if (done) cudaEventDestroy(done);
    for (int i = 0; i < MAX_SUB; i++) {
        if (sub_ready[i]) cudaEventDestroy(sub_ready[i]);
        if (sub_out[i]) cudaEventDestroy(sub_out[i]);
    }
    for (auto& e : piece_in) if (e) cudaEventDestroy(e);
    if (aux_stream) cudaStreamDestroy(aux_stream);
    if (in_stream) cudaStreamDestroy(in_stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (stream) cudaStreamDestroy(stream);
}

// ------------------------------------------------------------------------------------------------
Status Context::bind_device() const {
    EKZG_CUDA(cudaSetDevice(device_));
    return Status::Ok();
}

Status Context::create(bool use_precomp, std::unique_ptr<Context>* out, int device, const SetupBytes* custom) {
    std::unique_ptr<Context> c(new Context());
    Status s = c->init(use_precomp, device, custom);
    if (!s.ok) return s;
    *out = std::move(c);
    return Status::Ok();
}

Context::~Context() {
    cudaSetDevice(device_);
    for (Workspace* w : pool_) { w->release(); delete w; }
    for (auto& q : co_) for (CoalesceStaging* st : q.free_staging) { st->release(); delete st; }
    for (void* p : allocs_) cudaFree(p);
    if (g2keys_) host::g2_keys_free(g2keys_);
}

template <class T>
static Status dev_alloc(std::vector<void*>& allocs, T** p, size_t count) {
    void* q = nullptr;
    EKZG_CUDA(cudaMalloc(&q, count * sizeof(T)));
    allocs.push_back(q);
    *p = reinterpret_cast<T*>(q);
    return Status::Ok();
}

// device memory the table sizing leaves free for workspaces and other tenants (default 16 GiB)
static size_t hbm_reserve_bytes() {
    const char* e = getenv("EKZG_HBM_RESERVE_GIB");
    const double gib = e ? atof(e) : 16.0;
    return (size_t)((gib < 1.0 ? 1.0 : gib) * 1073741824.0);
}

Status Context::init(bool use_precomp, int device, const SetupBytes* custom) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return Status::Error("no CUDA device: this backend has no CPU fallback");
    if (device >= 0) {                          // one member of a multi-device set (kzg_multi.cu)
        if (device >= ndev) return Status::Error("EKZG_DEVICES names device " + std::to_string(device) + " but only " + std::to_string(ndev) + " are visible");
        device_ = device;
        EKZG_CUDA(cudaSetDevice(device_));
    } else if (const char* e = getenv("EKZG_DEVICE")) {
        device_ = atoi(e);
        EKZG_CUDA(cudaSetDevice(device_));
    } else {
        EKZG_CUDA(cudaGetDevice(&device_));
    }
    cudaDeviceProp prop;
    EKZG_CUDA(cudaGetDeviceProperties(&prop, device_));
    if (prop.major < 10) return Status::Error(std::string("device '") + prop.name + "' is not sm_100-class; this library is built for sm_100a only");
    EKZG_CUDA(kernels_init());
    EKZG_CUDA(recover_kernels_init());

    // use_precomp = false (the reference's UsePrecomp::No, fixed_base_msm.rs:83-89): smallest tables.
    // use_precomp = true: the widest window whose per-window tables fit the free HBM with room for the batch
    // workspaces -- every extra bit removes additions from the MSM (w = 14: 19 per scalar, 114 GiB of tables).
    int w = 8;
    if (use_precomp) {
        if (const char* e = getenv("EKZG_FK20_WINDOW")) {
            w = atoi(e);
        } else {
            size_t free_b = 0, total_b = 0;
            EKZG_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const size_t reserve = hbm_reserve_bytes() + (size_t)4096 * (255 / 12 + 1) * ((size_t)1 << 11) * sizeof(G1Affine);  // workspaces + SRS tables
            for (int cand : {14, 13, 12, 10, 8}) {
                w = cand;
                const size_t need = (size_t)FK20_MSMS * FK20_POINTS * (255 / cand + 1) * ((size_t)1 << (cand - 1)) * sizeof(G1Affine);
                if (need + reserve <= free_b) break;
            }
        }
    }
    if (w < 4 || w > 16) return Status::Error("EKZG_FK20_WINDOW must be in [4, 16]");
    T_.fk20.set_window(w);
    // monomial SRS tables: w = 12 is 17.7 GiB for the 4096 points (21.5 additions per scalar), w = 13 is 30 GiB (20 additions)
    int ws = use_precomp ? 12 : 8;
    if (const char* e = getenv("EKZG_SRS_WINDOW")) {
        ws = atoi(e);
    } else if (use_precomp) {
        size_t free_b = 0, total_b = 0;
        EKZG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        auto table_bytes = [](size_t npoints, int wb) { return npoints * (size_t)(255 / wb + 1) * ((size_t)1 << (wb - 1)) * sizeof(G1Affine); };
        if (table_bytes((size_t)FK20_MSMS * FK20_POINTS, w) + table_bytes(4096, 13) + hbm_reserve_bytes() <= free_b) ws = 13;
    }
    if (ws < 4 || ws > 16) return Status::Error("EKZG_SRS_WINDOW must be in [4, 16]");
    T_.srs.set_window(ws);
    msm_scratch_bytes_ = std::max(fixed_msm_scratch_bytes(T_.fk20), fixed_msm_scratch_bytes(T_.srs));

    cudaStream_t st = 0;
    // twiddles
    Fr *tw4096, *tw4096_inv, *tw8192, *tw8192_inv, *tw128, *tw64_inv;
    EKZG_TRY(dev_alloc(allocs_, &tw4096, 2048));
    EKZG_TRY(dev_alloc(allocs_, &tw4096_inv, 2048));
    EKZG_TRY(dev_alloc(allocs_, &tw8192, 4096));
    EKZG_TRY(dev_alloc(allocs_, &tw8192_inv, 4096));
    EKZG_TRY(dev_alloc(allocs_, &tw128, 64));
    EKZG_TRY(dev_alloc(allocs_, &tw64_inv, 32));
    EKZG_CUDA(launch_powers(tw4096, fr_omega_4096().v, 2048, st));
    EKZG_CUDA(launch_powers(tw4096_inv, fr_omega_4096_inv().v, 2048, st));
    EKZG_CUDA(launch_powers(tw8192, fr_omega_8192().v, 4096, st));
    EKZG_CUDA(launch_powers(tw8192_inv, fr_omega_8192_inv().v, 4096, st));
    EKZG_CUDA(launch_powers(tw128, fr_omega_128().v, 64, st));
    EKZG_CUDA(launch_powers(tw64_inv, fr_omega_64_inv().v, 32, st));
    T_.tw4096 = tw4096; T_.tw4096_inv = tw4096_inv; T_.tw8192 = tw8192; T_.tw8192_inv = tw8192_inv;
    T_.tw128 = tw128; T_.tw64_inv = tw64_inv;
    Fr *sh_fwd, *sh_inv;
    EKZG_TRY(dev_alloc(allocs_, &sh_fwd, 8192));
    EKZG_TRY(dev_alloc(allocs_, &sh_inv, 8192));
    EKZG_CUDA(launch_powers(sh_fwd, fr_coset_gen().v, 8192, st, fr_inv_8192().v));
    EKZG_CUDA(launch_powers(sh_inv, fr_coset_gen_inv().v, 8192, st, fr_inv_8192().v));
    coset_shift_fwd_ = sh_fwd;
    coset_shift_inv_ = sh_inv;

    // trusted setup: the embedded ceremony output, or the caller's (TrustedSetup::from_json[_unchecked])
    const unsigned char* g1_bytes = nullptr;
    uint32_t n_g1 = 4096, n_pts = 0;
    bool check_subgroup = true;
    const char* what = "embedded trusted setup";
    if (custom) {
        what = "trusted setup";
        if (custom->g1_monomial.size() != (size_t)48 * 4096)
            return Status::Error("trusted setup: g1_monomial must hold 4096 points, got " + std::to_string(custom->g1_monomial.size() / 48));
        for (uint32_t i = 0; i < 4096; i++)   // the table fill divides by differences of these points: the identity has no place in a setup
            if (custom->g1_monomial[(size_t)48 * i] & 0x40) return Status::Error("trusted setup: g1_monomial[" + std::to_string(i) + "] is the point at infinity");
        std::string err;
        g2keys_ = host::g2_keys_from_compressed(custom->g2_monomial.data(), (int)(custom->g2_monomial.size() / 96), custom->subgroup_check, &err);
        if (!g2keys_) return Status::Error(err);
        g1_bytes = custom->g1_monomial.data();
        n_pts = 4096;                       // the Lagrange-basis points of the file are not used (the reference skips them as well)
        check_subgroup = custom->subgroup_check;
    } else {
        const unsigned char* ts = ekzg_trusted_setup_start;
        size_t ts_len = (size_t)(ekzg_trusted_setup_end - ekzg_trusted_setup_start);
        if (ts_len < 16 || memcmp(ts, "EKZGTS01", 8) != 0) return Status::Error("embedded trusted setup: bad magic");
        uint32_t n_g2;
        memcpy(&n_g1, ts + 8, 4);
        memcpy(&n_g2, ts + 12, 4);
        if (n_g1 != 4096 || n_g2 != 65 || ts_len != 16 + (size_t)48 * 2 * n_g1 + (size_t)96 * n_g2)
            return Status::Error("embedded trusted setup: unexpected size");
        g1_bytes = ts + 16;
        n_pts = 2 * n_g1;
    }
    uint8_t* d_bytes = nullptr;
    uint32_t* d_st = nullptr;
    EKZG_CUDA(cudaMalloc(&d_bytes, (size_t)48 * n_pts));
    EKZG_CUDA(cudaMalloc(&d_st, sizeof(uint32_t) * n_pts));
    EKZG_CUDA(cudaMemset(d_st, 0, sizeof(uint32_t) * n_pts));
    EKZG_CUDA(cudaMemcpy(d_bytes, g1_bytes, (size_t)48 * n_pts, cudaMemcpyHostToDevice));
    G1Affine* srs;
    EKZG_TRY(dev_alloc(allocs_, &srs, (size_t)n_pts));
    // decompress + on-curve + prime-order-subgroup check of every G1 point on the device: the same validation
    // blstrs' from_compressed gives the reference when it parses the ceremony JSON (crates/trusted_setup/src/lib.rs:112-115,
    // crates/serialization/src/lib.rs:69-81), so a corrupted or substituted setup cannot yield a context
    // (from_json_unchecked: decompression and the curve equation only)
    EKZG_CUDA(launch_g1_validate(d_bytes, srs, d_st, n_pts, check_subgroup, st));
    std::vector<uint32_t> hst(n_pts);
    EKZG_CUDA(cudaMemcpy(hst.data(), d_st, sizeof(uint32_t) * n_pts, cudaMemcpyDeviceToHost));
    cudaFree(d_bytes);
    cudaFree(d_st);
    for (uint32_t i = 0; i < n_pts; i++)
        if (hst[i]) return Status::Error(std::string(what) + ": G1 point " + std::to_string(i) + " is malformed, off the curve or outside the prime-order subgroup");
    T_.srs_g1 = srs;
    T_.srs_g1_lagrange = custom ? nullptr : srs + n_g1;

    // FK20 tables
    size_t nbases = (size_t)FK20_MSMS * FK20_POINTS * T_.fk20.nw;
    size_t nentries = nbases * T_.fk20.half;
    G1Affine* table;
    EKZG_TRY(dev_alloc(allocs_, &table, nentries));
    table_bytes_ = nentries * sizeof(G1Affine);
    G1Jac* scratch = nullptr;
    G1Affine* qaff = nullptr;
    EKZG_CUDA(cudaMalloc(&scratch, (size_t)128 * 64 * sizeof(G1Jac)));
    EKZG_CUDA(cudaMalloc(&qaff, nbases * sizeof(G1Affine)));
    T_.fk20.table = table;
    uint32_t* setup_queue = nullptr;
    void* setup_ntt_scratch = nullptr;
    EKZG_CUDA(cudaMalloc(&setup_queue, g1_ntt_queue_words(64) * sizeof(uint32_t)));
    EKZG_CUDA(cudaMalloc(&setup_ntt_scratch, g1_ntt_scratch_bytes()));
    EKZG_CUDA(launch_fk20_setup(T_.srs_g1, scratch, qaff, table, T_, setup_queue, setup_ntt_scratch, st));
    EKZG_CUDA(cudaDeviceSynchronize());
    cudaFree(setup_queue);
    cudaFree(setup_ntt_scratch);
    cudaFree(scratch);
    cudaFree(qaff);
    // monomial SRS tables (commitments, single-point proofs)
    size_t sbases = (size_t)n_g1 * T_.srs.nw;
    G1Affine* stable;
    EKZG_TRY(dev_alloc(allocs_, &stable, sbases * T_.srs.half));
    table_bytes_ += sbases * T_.srs.half * sizeof(G1Affine);
    EKZG_CUDA(cudaMalloc(&qaff, sbases * sizeof(G1Affine)));
    T_.srs.table = stable;
    EKZG_CUDA(launch_srs_table_setup(T_.srs_g1, (int)n_g1, qaff, stable, T_.srs, st));
    EKZG_CUDA(cudaDeviceSynchronize());
    cudaFree(qaff);
    return Status::Ok();
}

// Workspace capacities come in few sizes (powers of two from 32 up to the chunk capacity, then the chunk capacity itself), so
// callers with varying batch sizes -- the coalescer produces every size from 1 to the cap -- reuse each other's workspaces.
static int round_capacity(int n) {
    const int chunk = chunk_capacity();
    if (n >= chunk) return n;
    int c = 32;
    while (c < n) c <<= 1;
    return std::min(c, chunk);
}

Workspace* Context::acquire(int min_capacity, bool with_io) const {
    {
        std::lock_guard<std::mutex> g(pool_mu_);
        int best = -1;   // best fit: a one-blob call must not take the 1024-blob workspace from under a concurrent batch
        for (size_t i = 0; i < pool_.size(); i++) {
            Workspace* w = pool_[i];
            if (w->capacity >= min_capacity && (!with_io || w->d_blobs) && (best < 0 || w->capacity < pool_[best]->capacity)) best = (int)i;
        }
        if (best >= 0) {
            Workspace* w = pool_[best];
            pool_.erase(pool_.begin() + best);
            return w;
        }
    }
    const int cap = round_capacity(min_capacity);
    for (int attempt = 0; attempt < 2; attempt++) {
        Workspace* w = new Workspace();
        Status s = w->alloc(cap, with_io, msm_scratch_bytes_);
        if (s.ok) return w;
        w->release();
        delete w;
        cudaGetLastError();   // a failed cudaMalloc must not linger as this thread's "last error" into the next launch check
        if (attempt == 0 && !trim_pool(0)) break;   // out of memory: give the idle workspaces back to the driver and retry once
    }
    return nullptr;
}

// drops idle workspaces until at most `keep` are left; returns how many were released
size_t Context::trim_pool(size_t keep) const {
    std::vector<Workspace*> victims;
    {
        std::lock_guard<std::mutex> g(pool_mu_);
        while (pool_.size() > keep) {   // smallest first: the big ones are the expensive ones to rebuild
            size_t v = 0;
            for (size_t i = 1; i < pool_.size(); i++) if (pool_[i]->capacity < pool_[v]->capacity) v = i;
            victims.push_back(pool_[v]);
            pool_.erase(pool_.begin() + v);
        }
    }
    for (Workspace* w : victims) { w->release(); delete w; }
    return victims.size();
}

void Context::give_back(Workspace* ws, const Status& s) const {
    if (!s.ok) ws->synchronize();
    {
        std::lock_guard<std::mutex> g(pool_mu_);
        pool_.push_back(ws);
    }
    static const size_t max_idle = [] { const char* e = getenv("EKZG_POOL_MAX"); int v = e ? atoi(e) : 8; return (size_t)(v < 1 ? 1 : v); }();
    trim_pool(max_idle);
}

// a workspace whose buffers could not be completed (allocation failure) is destroyed, not pooled
void Context::discard(Workspace* ws) const {
    ws->release();
    delete ws;
    cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
void Context::set_profiling(bool on) const {
    profiling_ = on;
    if (!on) {
        for (auto& v : prof_events_) for (cudaEvent_t e : v) cudaEventDestroy(e);
        prof_events_.clear();
    }
}

int Context::collect_stage_times(double* ms) const {
    int n = 0;
    for (auto& v : prof_events_) {
        if (cudaEventSynchronize(v.back()) != cudaSuccess) continue;
        for (int s = 0; s < N_STAGES; s++) {
            float t = 0;
            if (cudaEventElapsedTime(&t, v[s], v[s + 1]) == cudaSuccess) ms[s] += t;
        }
        n++;
        for (cudaEvent_t e : v) cudaEventDestroy(e);
    }
    prof_events_.clear();
    return n;
}

// One or two blobs: every proof as its own 4096-point MSM over the SRS tables (see k_coset_quotients) -- 128 n "virtual blobs"
// through the commitment pipeline: quotients -> fixed-base MSM (64 partial sums each) -> tree sum -> compression.
Status Context::proofs_direct_device(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream) const {
    const int Bv = N_CELLS * n;
    if (Bv > ws.capacity) return Status::Error("workspace too small for the direct proof path");
    EKZG_CUDA(launch_coset_quotients(ws.d_coeffs, ws.d_scalars, T_, n, stream));
    return srs_msm_compress(ws, Bv, d_proofs, stream);
}

// fixed-base MSM (64 partial sums per item) -> tree sum -> compression
Status Context::srs_msm_compress(Workspace& ws, int B, uint8_t* d_out, cudaStream_t stream) const {
    EKZG_CUDA(launch_fixed_msm(ws.d_scalars, ws.d_pts, T_.srs, N_BLOB / FK20_POINTS, B, stream, 0, -1, ws.d_msm_scratch));
    EKZG_CUDA(launch_sum_positions(ws.d_pts, B, N_BLOB / FK20_POINTS, 2, stream));
    EKZG_CUDA(launch_g1_compress(ws.d_pts, d_out, 1, B, stream));
    return Status::Ok();
}

Status Context::commit_device(Workspace& ws, int n, uint8_t* d_out48, cudaStream_t stream) const {
    EKZG_CUDA(launch_coeffs_to_scalars(ws.d_coeffs, ws.d_scalars, n, stream));
    return srs_msm_compress(ws, n, d_out48, stream);
}

Status Context::fk20_msm(Workspace& ws, int n, int o, int c, cudaStream_t stream, std::vector<cudaEvent_t>* ev) const {
    EKZG_CUDA(launch_toeplitz_scalars(ws.d_coeffs, ws.d_scalars, T_, n, stream, o, c));
    if (ev) cudaEventRecord((*ev)[2], stream);
    EKZG_CUDA(launch_fixed_msm(ws.d_scalars, ws.d_pts, T_.fk20, FK20_MSMS, n, stream, o, c, ws.d_msm_scratch));
    if (ev) cudaEventRecord((*ev)[3], stream);
    return Status::Ok();
}

Status Context::fk20_ntt_compress(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream, std::vector<cudaEvent_t>* ev) const {
    EKZG_CUDA(launch_fk20_g1_ntts(ws.d_pts, n, ws.d_queue, ws.d_ntt_scratch, stream));
    if (ev) cudaEventRecord((*ev)[4], stream);
    EKZG_CUDA(launch_g1_compress(ws.d_pts, d_proofs, N_CELLS, n, stream));
    if (ev) cudaEventRecord((*ev)[5], stream);
    return Status::Ok();
}

Status Context::fk20_from_coeffs_device(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream, std::vector<cudaEvent_t>* ev) const {
    const ProofRoute route = proof_route(n, n, !ev);
    if (route.direct && route.capacity <= ws.capacity) return proofs_direct_device(ws, n, d_proofs, stream);
    EKZG_TRY(fk20_msm(ws, n, 0, -1, stream, ev));
    return fk20_ntt_compress(ws, n, d_proofs, stream, ev);
}

Status Context::fk20_device(Workspace& ws, int n, const uint8_t* d_blobs, uint8_t* d_cells, uint8_t* d_proofs, uint32_t* d_status,
                            cudaStream_t stream) const {
    if (n > ws.capacity) return Status::Error("workspace too small");
    EKZG_CUDA(cudaMemsetAsync(d_status, 0, sizeof(uint32_t) * n, stream));
    if (profiling_ && d_proofs) {
        std::vector<cudaEvent_t> v(N_STAGES + 1);
        for (auto& e : v) EKZG_CUDA(cudaEventCreate(&e));
        prof_events_.push_back(v);
        cudaEventRecord(v[0], stream);
    }
    EKZG_CUDA(launch_blob_to_coeffs_cells(d_blobs, ws.d_coeffs, d_cells, d_status, T_, n, d_cells != nullptr, stream));
    if (profiling_ && d_proofs) cudaEventRecord(prof_events_.back()[1], stream);
    if (d_proofs) EKZG_TRY(fk20_from_coeffs_device(ws, n, d_proofs, stream, profiling_ ? &prof_events_.back() : nullptr));
    return Status::Ok();
}

// true if the CUDA driver can DMA straight from/to this host range (cudaMallocHost / cudaHostRegister memory)
static bool host_range_is_pinned(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// items [o, o + cnt) of `item` bytes each of the chunk at `chunk` -> the same slots of `dev`, on `st`.  Pinned caller memory is
// DMA'd as it is; pageable memory is copied into the same slots of the pinned staging buffer `stage` in slices of 8 MiB (64
// blobs), each slice's H2D running while the host copies the next one.
static Status upload(uint8_t* dev, uint8_t* stage, const uint8_t* chunk, size_t item, int o, int cnt, bool src_pinned, cudaStream_t st) {
    const size_t off = (size_t)o * item;
    if (src_pinned) {
        EKZG_CUDA(cudaMemcpyAsync(dev + off, chunk + off, (size_t)cnt * item, cudaMemcpyHostToDevice, st));
        return Status::Ok();
    }
    const int slice = (int)std::max<size_t>(1, (size_t)64 * BYTES_PER_BLOB / item);
    for (int i = 0; i < cnt; i += slice) {
        const size_t at = off + (size_t)i * item, bytes = (size_t)std::min(slice, cnt - i) * item;
        memcpy(stage + at, chunk + at, bytes);
        EKZG_CUDA(cudaMemcpyAsync(dev + at, stage + at, bytes, cudaMemcpyHostToDevice, st));
    }
    return Status::Ok();
}

static Status upload_blobs(Workspace& ws, const uint8_t* chunk, int o, int cnt, bool src_pinned, cudaStream_t st) {
    return upload(ws.d_blobs, ws.h_blobs, chunk, BYTES_PER_BLOB, o, cnt, src_pinned, st);
}

// Blobs of the first FK20 piece of a chunk of cnt: its K1, K2 and K4 run while the rest of the chunk is still on the wire.  A
// quarter of the chunk (whole 32-blob groups) from 512 blobs up, else the whole chunk.
static int fk20_first_piece(int cnt) { return cnt >= 512 ? ((cnt / 4 + 31) & ~31) : cnt; }

// The batch scheduler behind every host-buffer prover entry point (replaces the reference's rayon fan-out,
// crates/maybe_rayon/src/multi_threaded.rs:9-39).  A chunk (<= EKZG_CHUNK blobs, default 1024) is cut into
// sub-blocks: sub-block s is copied in and run through K1 while s+1 is still on the wire; its cells go back to the
// host on a second stream as soon as K1 wrote them, i.e. during the ~100 ms the FK20 kernels (K2..K6, launched
// once for the whole chunk) need.  Caller buffers that are already pinned are used for the DMA directly; pageable
// ones go through the workspace's pinned staging, the host copies being hidden the same way.  Chunks alternate
// between two workspaces so the copies of chunk c+1 overlap the kernels of chunk c.
Status Context::compute_cells_and_kzg_proofs_batch(uint64_t n, const uint8_t* blobs, uint8_t* cells, uint8_t* proofs,
                                                   uint8_t* blob_status, bool want_proofs) const {
    if (n == 0) return Status::Ok();
    EKZG_TRY(bind_device());
    const int cap = (int)std::min<uint64_t>(n, (uint64_t)chunk_capacity());
    const uint64_t nchunks = (n + cap - 1) / cap;
    const ProofRoute route = proof_route(n, cap, want_proofs);   // direct: the latency path, see proofs_direct_device
    Workspace* W[2] = {acquire(route.capacity, true), nchunks > 1 ? acquire(cap, true) : nullptr};
    if (!W[0] || (nchunks > 1 && !W[1])) {
        const Status s = Status::Error("device/pinned memory allocation failed");
        for (Workspace* w : W) if (w) give_back(w, s);
        return s;
    }
    const bool in_pinned = host_range_is_pinned(blobs);
    const bool cells_pinned = cells && host_range_is_pinned(cells);
    const bool proofs_pinned = want_proofs && host_range_is_pinned(proofs);
    bool any_bad = false;
    Status result = Status::Ok();
    TraceClock tr("compute_cells_and_kzg_proofs_batch");
    // EKZG_TRACE: device timeline of the first chunk (timed events on the three streams)
    std::vector<std::pair<std::string, cudaEvent_t>> tl;
    auto stamp = [&](const char* what, int idx, cudaStream_t st) {
        if (!tr.on) return;
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        cudaEventRecord(e, st);
        tl.emplace_back(std::string(what) + (idx >= 0 ? " " + std::to_string(idx) : ""), e);
    };
    uint64_t pending_first[2] = {0, 0};
    int pending_cnt[2] = {0, 0}, pending_np[2] = {0, 0};
    int piece_off[2][Workspace::MAX_SUB], piece_len[2][Workspace::MAX_SUB];
    auto drain = [&](int slot) -> Status {
        Workspace& ws = *W[slot];
        if (!pending_cnt[slot]) return Status::Ok();
        const uint64_t first = pending_first[slot];
        const int cnt = pending_cnt[slot];
        if (cells) {
            for (int s = 0; s < pending_np[slot]; s++) {
                EKZG_CUDA(cudaEventSynchronize(ws.sub_out[s]));
                const int o = piece_off[slot][s], c = piece_len[slot][s];
                if (!cells_pinned) memcpy(cells + (first + o) * CELLS_PER_BLOB, ws.h_cells + (size_t)o * CELLS_PER_BLOB, (size_t)c * CELLS_PER_BLOB);
            }
        }
        tr.mark("cells of the chunk are in host memory");
        EKZG_CUDA(cudaEventSynchronize(ws.done));
        tr.mark("kernels + proofs D2H done");
        if (want_proofs && !proofs_pinned) memcpy(proofs + first * PROOFS_PER_BLOB, ws.h_proofs, (size_t)cnt * PROOFS_PER_BLOB);
        for (int i = 0; i < cnt; i++) {
            if (ws.h_status[i]) any_bad = true;
            if (blob_status) blob_status[first + i] = ws.h_status[i] ? ITEM_NON_CANONICAL : ITEM_OK;
        }
        pending_cnt[slot] = 0;
        return Status::Ok();
    };
    // One chunk.  Three streams: in_stream carries the blobs to the device piece by piece (50 GB/s: 1024 blobs in 2.6 ms);
    // ws.stream runs ALL kernels in order -- K1, K2, K4 of the first piece (a quarter of the chunk) as soon as that piece has
    // arrived, then K1, K2, K4 of the rest, then K5 (which wants the whole chunk for its parallelism) and K6; copy_stream takes
    // the cells of a piece home as soon as its K1 is done, i.e. underneath the ~90 ms of FK20 kernels.
    // (K1 must not run on a stream of its own next to K4: its 1024-thread, 128 KiB CTAs do not fit beside K4's resident CTAs and
    // starve until K4 ends -- measured: K1 of sub-block 5 waited 13 ms, profiles/r1_v4_e2e_timeline.txt.)
    auto submit = [&](int slot, uint64_t first, int cnt) -> Status {
        Workspace& ws = *W[slot];
        int np = 0;
        int* off = piece_off[slot];
        int* len = piece_len[slot];
        if (want_proofs) {
            const int q = fk20_first_piece(cnt);
            off[np] = 0; len[np++] = q;
            if (q < cnt) { off[np] = q; len[np++] = cnt - q; }
        } else {   // cells only: nothing but copies and K1, finer pieces keep both copy engines busy
            const int n_p = std::min(Workspace::MAX_SUB, (cnt + 127) / 128), per = (cnt + n_p - 1) / n_p;
            for (int o = 0; o < cnt; o += per) { off[np] = o; len[np++] = std::min(per, cnt - o); }
        }
        EKZG_CUDA(cudaStreamWaitEvent(ws.in_stream, ws.done, 0));   // (the previous chunk of this workspace has left the buffers)
        stamp("start", -1, ws.in_stream);
        EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * cnt, ws.stream));
        for (int s = 0; s < np; s++) {
            const int o = off[s], c = len[s];
            EKZG_TRY(upload_blobs(ws, blobs + first * BYTES_PER_BLOB, o, c, in_pinned, ws.in_stream));
            stamp("H2D done, piece", s, ws.in_stream);
            EKZG_CUDA(cudaEventRecord(ws.piece_in[s], ws.in_stream));
            EKZG_CUDA(cudaStreamWaitEvent(ws.stream, ws.piece_in[s], 0));
            EKZG_CUDA(launch_blob_to_coeffs_cells(ws.d_blobs + (size_t)o * BYTES_PER_BLOB, ws.d_coeffs + (size_t)o * N_BLOB,
                                                  cells ? ws.d_cells + (size_t)o * CELLS_PER_BLOB : nullptr, ws.d_status + o, T_, c, cells != nullptr, ws.stream));
            stamp("K1 done, piece", s, ws.stream);
            if (cells) {
                EKZG_CUDA(cudaEventRecord(ws.sub_ready[s], ws.stream));
                EKZG_CUDA(cudaStreamWaitEvent(ws.copy_stream, ws.sub_ready[s], 0));
                uint8_t* dst = cells_pinned ? cells + (first + o) * CELLS_PER_BLOB : ws.h_cells + (size_t)o * CELLS_PER_BLOB;
                EKZG_CUDA(cudaMemcpyAsync(dst, ws.d_cells + (size_t)o * CELLS_PER_BLOB, (size_t)c * CELLS_PER_BLOB, cudaMemcpyDeviceToHost, ws.copy_stream));
                EKZG_CUDA(cudaEventRecord(ws.sub_out[s], ws.copy_stream));
            }
            if (want_proofs && !route.direct) {
                EKZG_TRY(fk20_msm(ws, cnt, o, c, ws.stream, nullptr));
                stamp("K4 done, piece", s, ws.stream);
            }
        }
        if (want_proofs) {
            if (route.direct) {
                EKZG_TRY(proofs_direct_device(ws, cnt, ws.d_proofs, ws.stream));
                stamp("direct proofs done", -1, ws.stream);
            } else {
                EKZG_TRY(fk20_ntt_compress(ws, cnt, ws.d_proofs, ws.stream, nullptr));
            }
            EKZG_CUDA(cudaMemcpyAsync(proofs_pinned ? proofs + first * PROOFS_PER_BLOB : ws.h_proofs, ws.d_proofs, (size_t)cnt * PROOFS_PER_BLOB,
                                      cudaMemcpyDeviceToHost, ws.stream));
            stamp("K6 + proofs D2H done", -1, ws.stream);
        }
        EKZG_CUDA(cudaMemcpyAsync(ws.h_status, ws.d_status, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, ws.stream));
        EKZG_CUDA(cudaEventRecord(ws.done, ws.stream));
        pending_first[slot] = first;
        pending_cnt[slot] = cnt;
        pending_np[slot] = np;
        tr.mark("chunk enqueued");
        return Status::Ok();
    };
    for (uint64_t c = 0; c < nchunks && result.ok; c++) {
        const int slot = (int)(c & 1);
        result = drain(slot);
        if (!result.ok) break;
        const uint64_t first = c * cap;
        result = submit(slot, first, (int)std::min<uint64_t>(cap, n - first));
    }
    for (int slot = 0; slot < 2; slot++) {
        if (!W[slot]) continue;
        if (result.ok) result = drain(slot);
        give_back(W[slot], result);
    }
    if (tr.on && !tl.empty()) {
        cudaDeviceSynchronize();
        for (auto& pe : tl) {
            float ms = 0;
            cudaError_t ee = cudaEventElapsedTime(&ms, tl[0].second, pe.second);
            if (ee == cudaSuccess) fprintf(stderr, "[ekzg timeline] %8.3f ms  %s\n", ms, pe.first.c_str());
            else fprintf(stderr, "[ekzg timeline] %s: %s\n", pe.first.c_str(), cudaGetErrorString(ee));
        }
        for (auto& pe : tl) cudaEventDestroy(pe.second);
    }
    if (!result.ok) return result;
    if (any_bad) return Status::Error(item_status_text(ITEM_NON_CANONICAL, false, false));
    return Status::Ok();
}

// ------------------------------------------------------------------------------------------------
// Single-item entry points with coalescing of concurrent callers (see kzg_runtime.h).
//
// A batch is formed in a pinned staging block.  Every caller copies its own input into its slot of the block and, when the
// batch has run, copies its own results out to wherever its binding wants them (128 + 128 scattered pointers through the C
// ABI) -- so the host copies of a batch of n callers run on n threads, and the device DMAs straight from / into the block.
// The first caller of a batch is its leader: it lingers until nobody has joined for a moment (or, when two batches are
// already on the device, until one of them finishes -- more callers per batch cost nothing then), closes the batch, runs
// it through the batch entry point and wakes the members.  Callers arriving after the close start the next batch at once,
// so its staging overlaps the kernels of the batches in flight.
static int coalesce_capacity() {
    static const int v = [] {
        const char* e = getenv("EKZG_COALESCE_MAX");
        int c = e ? atoi(e) : 256;
        return c < 1 ? 1 : (c > 4096 ? 4096 : c);
    }();
    return std::min(v, chunk_capacity());
}

Status Context::CoalesceStaging::alloc(int cap, size_t in_bytes_per_item, bool with_proofs, bool with_index) {
    capacity = cap;
    in_stride = in_bytes_per_item;
    EKZG_CUDA(cudaMallocHost(&in, (size_t)cap * in_stride));
    EKZG_CUDA(cudaMallocHost(&cells, (size_t)cap * N_EXT * 32));
    if (with_proofs) EKZG_CUDA(cudaMallocHost(&proofs, (size_t)cap * N_CELLS * BYTES_PER_G1));
    status.assign(cap, 0);
    if (with_index) { counts.assign(cap, 0); indices.assign((size_t)cap * N_CELLS, 0); }
    return Status::Ok();
}
void Context::CoalesceStaging::release() {
    cudaFreeHost(in); cudaFreeHost(cells); cudaFreeHost(proofs);
    in = cells = proofs = nullptr;
}

// 128 cells or proofs of one blob, contiguous at `src`, out through the 128 separate pointers the C ABI hands over
static void scatter(const uint8_t* src, size_t item_bytes, uint8_t* const* dst) {
    for (int i = 0; i < N_CELLS; i++) memcpy(dst[i], src + (size_t)i * item_bytes, item_bytes);
}

Status Context::coalesce(int which, CoalesceReq& me) const {
    CoalesceQueue& Q = co_[which];
    const bool recover = which == CQ_RECOVER, want_proofs = which != CQ_CELLS;
    const int cap = coalesce_capacity();
    static const int linger_us = [] { const char* e = getenv("EKZG_COALESCE_LINGER_US"); return e ? atoi(e) : 300; }();
    constexpr int MAX_IN_FLIGHT = 2, MAX_STAGING = 6;
    std::unique_lock<std::mutex> lk(Q.mu);
    Q.callers++;
    struct Leave { CoalesceQueue& q; std::unique_lock<std::mutex>& l; ~Leave() { if (!l.owns_lock()) l.lock(); q.callers--; } } leave{Q, lk};
    // ---- join the batch being formed, or start one ----
    CoalesceBatch* Bt = nullptr;
    bool leader = false;
    for (;;) {
        Bt = Q.forming;
        if (Bt && !Bt->closed && Bt->n < Bt->st->capacity) break;
        // start a batch: needs a staging block
        CoalesceStaging* st = nullptr;
        if (!Q.free_staging.empty()) {
            st = Q.free_staging.back();
            Q.free_staging.pop_back();
        } else if (Q.n_staging < MAX_STAGING) {
            Q.n_staging++;
            lk.unlock();
            st = new CoalesceStaging();
            Status s = bind_device();
            if (s.ok) s = st->alloc(cap, recover ? (size_t)N_CELLS * BYTES_PER_CELL : (size_t)BYTES_PER_BLOB, want_proofs, recover);
            lk.lock();
            if (!s.ok) {
                st->release();
                delete st;
                cudaGetLastError();
                Q.n_staging--;
                return s;
            }
        } else {
            Q.cv.wait(lk);          // all blocks are busy: one comes back when its last member has copied out
            continue;
        }
        if (Q.forming && !Q.forming->closed && Q.forming->n < Q.forming->st->capacity) {   // somebody else started one meanwhile
            Q.free_staging.push_back(st);
            continue;
        }
        Bt = new CoalesceBatch();
        Bt->st = st;
        Q.forming = Bt;
        leader = true;
        break;
    }
    const int slot = Bt->n++;
    Bt->left++;
    CoalesceStaging& st = *Bt->st;
    lk.unlock();
    // ---- copy my input into my slot (all members do this at the same time) ----
    if (recover) {
        st.counts[slot] = me.count;
        // the batch entry point takes the cells of all items concatenated; a slot is 128 cells wide, so items are packed later by
        // the leader's index list only -- the cell bytes stay where they are and the batch call gets per-item offsets via counts
        memcpy(st.in + (size_t)slot * st.in_stride, me.in, (size_t)me.count * BYTES_PER_CELL);
        memcpy(&st.indices[(size_t)slot * N_CELLS], me.indices, (size_t)me.count * sizeof(uint64_t));
    } else {
        memcpy(st.in + (size_t)slot * st.in_stride, me.in, BYTES_PER_BLOB);
    }
    lk.lock();
    Bt->copied++;
    Q.cv_leader.notify_all();
    if (leader) {
        // ---- linger, close, run ----
        static const bool trace = getenv("EKZG_TRACE_COALESCE") != nullptr;
        const auto t_lead = std::chrono::steady_clock::now();
        const auto t_end = std::chrono::steady_clock::now() + std::chrono::microseconds(8 * (linger_us > 0 ? linger_us : 0));
        while (Bt->n < st.capacity) {
            if (Q.in_flight >= MAX_IN_FLIGHT) {          // the device is busy anyway: keep collecting until a batch finishes
                Q.cv_leader.wait_for(lk, std::chrono::microseconds(200));
                continue;
            }
            if (linger_us <= 0) break;
            if (Q.callers == 1 && Bt->n == 1) break;     // nobody else is in here: lingering would only add to a lone caller's latency
            const auto gap_end = std::min(t_end, std::chrono::steady_clock::now() + std::chrono::microseconds(linger_us));
            const int before = Bt->n;
            while (Bt->n == before && Q.cv_leader.wait_until(lk, gap_end) != std::cv_status::timeout) {}
            if (Bt->n == before || std::chrono::steady_clock::now() >= t_end) break;
        }
        Bt->closed = true;
        if (Q.forming == Bt) Q.forming = nullptr;
        while (Bt->copied < Bt->n) Q.cv_leader.wait(lk);
        const int n = Bt->n;
        const int flying = Q.in_flight++;
        const bool crowded = flying >= 1 || Q.callers > n;   // other batches on the device, or callers that did not make it into this one
        lk.unlock();
        const auto t_run = std::chrono::steady_clock::now();
        Status s = Status::Ok();
        try {
            std::fill(st.status.begin(), st.status.begin() + n, 0);
            // other batches are on the device already (or the next one is forming behind this one): this batch cannot have the
            // device to itself, so ask for the G1-NTT kernel with the least work (kzg_kernels.h) instead of the latency-mode ones
            set_k5_throughput_hint(crowded);
            if (recover) s = recover_impl(n, st.counts.data(), st.indices.data(), st.in, st.cells, st.proofs, st.status.data(), true);
            else s = compute_cells_and_kzg_proofs_batch(n, st.in, st.cells, want_proofs ? st.proofs : nullptr, st.status.data(), want_proofs);
        } catch (const std::exception& ex) {             // fail the batch, never the queue
            s = Status::Error(std::string("batch failed: ") + ex.what());
        }
        set_k5_throughput_hint(false);
        if (trace) {
            const auto t_done = std::chrono::steady_clock::now();
            fprintf(stderr, "[ekzg trace] coalesced batch of %d (queue %d, %d already on the device): formed in %.2f ms, ran %.2f ms\n", n, which, flying,
                    std::chrono::duration<double, std::milli>(t_run - t_lead).count(), std::chrono::duration<double, std::milli>(t_done - t_run).count());
        }
        lk.lock();
        Q.in_flight--;
        Bt->result = s;
        Bt->done = true;
        Q.cv.notify_all();
        Q.cv_leader.notify_all();
    } else {
        while (!Bt->done) Q.cv.wait(lk);
    }
    lk.unlock();
    // ---- copy my results out of my slot (again all members at once) ----
    Status mine = Status::Ok();
    bool any_flag = false;
    for (int i = 0; i < Bt->n && !any_flag; i++) any_flag = st.status[i] != 0;
    if (!Bt->result.ok && !any_flag) {
        mine = Bt->result;                                // the batch as a whole failed (CUDA error, allocation)
    } else if (st.status[slot]) {
        mine = Status::Error(item_status_text(st.status[slot], recover, false));   // this item is the invalid one; the others are served
    } else {
        const uint8_t* c = st.cells + (size_t)slot * CELLS_PER_BLOB;
        if (me.cells_scattered) scatter(c, BYTES_PER_CELL, me.cells_scattered);
        else memcpy(me.cells, c, CELLS_PER_BLOB);
        if (want_proofs) {
            const uint8_t* p = st.proofs + (size_t)slot * PROOFS_PER_BLOB;
            if (me.proofs_scattered) scatter(p, BYTES_PER_G1, me.proofs_scattered);
            else memcpy(me.proofs, p, PROOFS_PER_BLOB);
        }
    }
    lk.lock();
    if (--Bt->left == 0) {
        Q.free_staging.push_back(Bt->st);
        delete Bt;
        Q.cv.notify_all();
    }
    return mine;
}

static bool coalescing_off() {
    static const bool off = getenv("EKZG_NO_COALESCE") != nullptr;
    return off;
}

// One item as a batch of one, past the coalescer: run(cells, proofs) is the batch call, and outputs bound for 128 separate
// pointers go through temporary contiguous buffers.
template <class Run>
static Status run_uncoalesced(uint8_t* cells, uint8_t* proofs, uint8_t* const* cells_scattered, uint8_t* const* proofs_scattered, Run run) {
    std::vector<uint8_t> tc(cells_scattered ? CELLS_PER_BLOB : 0), tp(proofs_scattered ? PROOFS_PER_BLOB : 0);
    if (cells_scattered) cells = tc.data();
    if (proofs_scattered) proofs = tp.data();
    Status s = run(cells, proofs);
    if (!s.ok) return s;
    if (cells_scattered) scatter(cells, BYTES_PER_CELL, cells_scattered);
    if (proofs_scattered) scatter(proofs, BYTES_PER_G1, proofs_scattered);
    return s;
}

Status Context::compute_cells_and_kzg_proofs_one(const uint8_t* blob, uint8_t* cells, uint8_t* proofs, uint8_t* const* cells_scattered,
                                                 uint8_t* const* proofs_scattered, bool want_proofs) const {
    if (!want_proofs) { proofs = nullptr; proofs_scattered = nullptr; }
    if (coalescing_off())
        return run_uncoalesced(cells, proofs, cells_scattered, proofs_scattered, [&](uint8_t* c, uint8_t* p) {
            return compute_cells_and_kzg_proofs_batch(1, blob, c, p, nullptr, want_proofs);
        });
    CoalesceReq me;
    me.in = blob; me.cells = cells; me.proofs = proofs; me.cells_scattered = cells_scattered; me.proofs_scattered = proofs_scattered;
    return coalesce(want_proofs ? CQ_CELLS_PROOFS : CQ_CELLS, me);
}

Status Context::recover_cells_and_kzg_proofs_one(uint64_t count, const uint64_t* indices, const uint8_t* cells, uint8_t* out_cells,
                                                 uint8_t* out_proofs, uint8_t* const* cells_scattered, uint8_t* const* proofs_scattered) const {
    // index errors are decided here, in the reference's order (recovery.rs:90-146), so that a caller gets the exact error and a
    // malformed request never joins a shared batch
    bool bad = count < (uint64_t)N_CELLS / 2 || count > (uint64_t)N_CELLS;
    for (uint64_t k = 0; k < count && !bad; k++) bad = indices[k] >= (uint64_t)N_CELLS || (k && !(indices[k - 1] < indices[k]));
    if (bad || coalescing_off())
        return run_uncoalesced(out_cells, out_proofs, cells_scattered, proofs_scattered, [&](uint8_t* c, uint8_t* p) {
            return recover_cells_and_kzg_proofs_batch(1, &count, indices, cells, c, p, nullptr);
        });
    CoalesceReq me;
    me.in = cells; me.indices = indices; me.count = count; me.cells = out_cells; me.proofs = out_proofs;
    me.cells_scattered = cells_scattered; me.proofs_scattered = proofs_scattered;
    return coalesce(CQ_RECOVER, me);
}

// ------------------------------------------------------------------------------------------------
// Erasure recovery.
static int rev7(int x) {
    int r = 0;
    for (int b = 0; b < 7; b++) r |= ((x >> b) & 1) << (6 - b);
    return r;
}

// Host-side validation of n recovery items in the reference's order (recovery.rs:90-146): item i has counts[i] indices at
// indices + offset[i].  Marks every invalid item ITEM_BAD_INDICES in code[] and returns the error of the first one ("" if none).
static std::string check_recovery_indices(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint64_t* offset, uint8_t* code) {
    std::string first_err;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t* idx = indices + offset[i];
        const uint64_t c = counts[i];
        const char* err = nullptr;
        for (uint64_t k = 0; k < c && !err; k++)
            if (idx[k] >= (uint64_t)N_CELLS) err = "Recovery(CellIndexOutOfRange)";
        for (uint64_t k = 1; k < c && !err; k++)
            if (!(idx[k - 1] < idx[k])) err = "Recovery(CellIndicesNotUniquelyOrdered)";
        if (!err && c < (uint64_t)N_CELLS / 2) err = "Recovery(NotEnoughCellsToReconstruct)";
        if (!err && c > (uint64_t)N_CELLS) err = "Recovery(TooManyCellsReceived)";
        if (err) {
            code[i] = ITEM_BAD_INDICES;
            if (first_err.empty()) first_err = err;
        }
    }
    return first_err;
}

// The slot map of one item: sm[m] = rank of the given cell at bit-reversed domain position m, or -1.  An invalid item gets a
// harmless well-formed instance instead: all cells present (the caller points the device at 128 zero cells for it).
static void fill_slotmap(int16_t* sm, const uint64_t* idx, uint64_t count, bool invalid) {
    if (invalid) {
        for (int m = 0; m < N_CELLS; m++) sm[m] = (int16_t)m;
        return;
    }
    for (int m = 0; m < N_CELLS; m++) sm[m] = -1;
    for (uint64_t k = 0; k < count; k++) sm[rev7((int)idx[k])] = (int16_t)k;
}

// ItemStatus of a valid item from the status bits of the recovery kernels (nonzero)
static uint8_t recovery_device_code(uint32_t bits) { return (bits & 1) ? ITEM_NON_CANONICAL : ITEM_BAD_DEGREE; }

Status Context::recover_cells_and_kzg_proofs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells,
                                                   uint8_t* out_cells, uint8_t* out_proofs, uint8_t* item_status) const {
    return recover_impl(n, counts, indices, cells, out_cells, out_proofs, item_status, false);
}

Status Context::recover_impl(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_cells,
                             uint8_t* out_proofs, uint8_t* item_status, bool strided) const {
    if (n == 0) return Status::Ok();
    EKZG_TRY(bind_device());
    // host-side validation in the reference's order (recovery.rs:90-146); invalid items are skipped on the device
    std::vector<uint64_t> offset(n + 1, 0);
    for (uint64_t i = 0; i < n; i++) offset[i + 1] = strided ? (i + 1) * (uint64_t)N_CELLS : offset[i] + counts[i];
    std::vector<uint8_t> code(n, 0);
    std::string first_err = check_recovery_indices(n, counts, indices, offset.data(), code.data());
    const int cap = (int)std::min<uint64_t>(n, (uint64_t)chunk_capacity());
    Workspace* wsp = acquire(proof_route(n, cap, true).capacity, true);
    if (!wsp) return Status::Error("device/pinned memory allocation failed");
    Workspace& ws = *wsp;
    Status result = ws.ensure_recover_buffers();
    if (!result.ok) { discard(wsp); return result; }
    cudaStream_t st = ws.stream;
    const bool in_pinned = host_range_is_pinned(cells), cells_pinned = host_range_is_pinned(out_cells), proofs_pinned = host_range_is_pinned(out_proofs);
    TraceClock tr("recover_cells_and_kzg_proofs_batch");
    auto body = [&](uint64_t first, int cnt) -> Status {
        // slot maps (which input cell sits at which bit-reversed position) and the cells themselves: blob i's cells go
        // to slots 0..count-1 of its 128-slot row on the device, straight from the caller's memory when it is pinned
        for (int i = 0; i < cnt; i++) {
            int16_t* sm = ws.h_slotmap + (size_t)i * 128;
            const uint64_t g = first + i;
            uint8_t* d_row = ws.d_rcells + (size_t)i * N_CELLS * BYTES_PER_CELL;
            fill_slotmap(sm, indices + offset[g], counts[g], code[g] != 0);
            if (code[g]) {  // the harmless instance's cells: all zero
                EKZG_CUDA(cudaMemsetAsync(d_row, 0, (size_t)N_CELLS * BYTES_PER_CELL, st));
                continue;
            }
            const uint8_t* src = cells + offset[g] * BYTES_PER_CELL;
            const size_t bytes = (size_t)counts[g] * BYTES_PER_CELL;
            if (!in_pinned) {
                uint8_t* stage = ws.h_rcells + (size_t)i * N_CELLS * BYTES_PER_CELL;
                memcpy(stage, src, bytes);
                src = stage;
            }
            EKZG_CUDA(cudaMemcpyAsync(d_row, src, bytes, cudaMemcpyHostToDevice, st));
        }
        tr.mark("slot maps + enqueue H2D of the cells");
        EKZG_CUDA(cudaMemcpyAsync(ws.d_slotmap, ws.h_slotmap, (size_t)cnt * 128 * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * cnt, st));
        EKZG_CUDA(launch_recover_coeffs(ws.d_rcells, ws.d_slotmap, ws.d_ze, ws.d_czinv, reinterpret_cast<Fr*>(ws.d_scalars),
                                        reinterpret_cast<Fr*>(ws.d_cells), ws.d_coeffs, ws.d_status, T_, coset_shift_fwd_, coset_shift_inv_,
                                        fr_coset_gen_pow64().v, cnt, st));
        EKZG_CUDA(launch_coeffs_to_cells(ws.d_coeffs, ws.d_cells, T_, cnt, st));
        // the cells travel back on the copy stream while the FK20 kernels run
        EKZG_CUDA(cudaEventRecord(ws.sub_ready[0], st));
        EKZG_CUDA(cudaStreamWaitEvent(ws.copy_stream, ws.sub_ready[0], 0));
        EKZG_CUDA(cudaMemcpyAsync(cells_pinned ? out_cells + first * CELLS_PER_BLOB : ws.h_cells, ws.d_cells, (size_t)cnt * CELLS_PER_BLOB,
                                  cudaMemcpyDeviceToHost, ws.copy_stream));
        EKZG_CUDA(cudaEventRecord(ws.sub_out[0], ws.copy_stream));
        EKZG_TRY(fk20_from_coeffs_device(ws, cnt, ws.d_proofs, st));
        EKZG_CUDA(cudaMemcpyAsync(proofs_pinned ? out_proofs + first * PROOFS_PER_BLOB : ws.h_proofs, ws.d_proofs, (size_t)cnt * PROOFS_PER_BLOB,
                                  cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaMemcpyAsync(ws.h_status, ws.d_status, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaEventSynchronize(ws.sub_out[0]));
        if (!cells_pinned) memcpy(out_cells + first * CELLS_PER_BLOB, ws.h_cells, (size_t)cnt * CELLS_PER_BLOB);
        EKZG_CUDA(cudaStreamSynchronize(st));
        tr.mark("recovery kernels + FK20 + copies");
        if (!proofs_pinned) memcpy(out_proofs + first * PROOFS_PER_BLOB, ws.h_proofs, (size_t)cnt * PROOFS_PER_BLOB);
        for (int i = 0; i < cnt; i++) {
            const uint64_t g = first + i;
            if (!code[g] && ws.h_status[i]) {
                code[g] = recovery_device_code(ws.h_status[i]);
                if (first_err.empty()) first_err = item_status_text(code[g], true, false);
            }
        }
        return Status::Ok();
    };
    for (uint64_t first = 0; first < n && result.ok; first += cap) result = body(first, (int)std::min<uint64_t>(cap, n - first));
    give_back(wsp, result);
    if (item_status) memcpy(item_status, code.data(), n);
    if (!result.ok) return result;
    if (!first_err.empty()) return Status::Error(first_err);
    return Status::Ok();
}

// Blobs from their cells, without proofs: R0..R3 of the recovery, then only the first half of the extension (the blob).  With no
// FK20 behind them the kernels take about as long as the copies (up to 256 KiB of cells up, 128 KiB of blob down per item), so
// this path is a pipeline: chunks alternate over two workspaces as in compute_cells_and_kzg_proofs_batch, and a chunk is cut
// into pieces whose cells go up on in_stream, run through the kernels on `stream` and whose blobs go home on copy_stream, each
// piece a step behind the one before.  The cells go up as the caller packed them (k_recover_ntt_packed reads them through a
// per-blob offset table): one copy per run of valid items, with no re-layout on the host.
Status Context::recover_blobs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_blobs,
                                    uint8_t* item_status) const {
    if (n == 0) return Status::Ok();
    EKZG_TRY(bind_device());
    std::vector<uint64_t> offset(n + 1, 0);
    for (uint64_t i = 0; i < n; i++) offset[i + 1] = offset[i] + counts[i];
    std::vector<uint8_t> code(n, 0);
    std::string first_err = check_recovery_indices(n, counts, indices, offset.data(), code.data());
    const int cap = (int)std::min<uint64_t>(n, (uint64_t)chunk_capacity());
    const uint64_t nchunks = (n + cap - 1) / cap;
    Workspace* W[2] = {acquire(cap, true), nchunks > 1 ? acquire(cap, true) : nullptr};
    Status result = Status::Ok();
    if (!W[0] || (nchunks > 1 && !W[1])) result = Status::Error("device/pinned memory allocation failed");
    for (Workspace* w : W)
        if (w && result.ok) result = w->ensure_recover_buffers();
    if (!result.ok) {
        for (Workspace* w : W) if (w) give_back(w, result);
        return result;
    }
    const bool in_pinned = host_range_is_pinned(cells), out_pinned = host_range_is_pinned(out_blobs);
    TraceClock tr("recover_blobs_batch");
    uint64_t pending_first[2] = {0, 0};
    int pending_cnt[2] = {0, 0}, pending_np[2] = {0, 0};
    int piece_off[2][Workspace::MAX_SUB], piece_len[2][Workspace::MAX_SUB];
    auto drain = [&](int slot) -> Status {
        Workspace& ws = *W[slot];
        if (!pending_cnt[slot]) return Status::Ok();
        const uint64_t first = pending_first[slot];
        for (int s = 0; s < pending_np[slot]; s++) {
            EKZG_CUDA(cudaEventSynchronize(ws.sub_out[s]));
            const int o = piece_off[slot][s], c = piece_len[slot][s];
            if (!out_pinned) memcpy(out_blobs + (first + o) * BYTES_PER_BLOB, ws.h_blobs + (size_t)o * BYTES_PER_BLOB, (size_t)c * BYTES_PER_BLOB);
        }
        EKZG_CUDA(cudaEventSynchronize(ws.done));
        for (int i = 0; i < pending_cnt[slot]; i++)
            if (!code[first + i] && ws.h_status[i]) code[first + i] = recovery_device_code(ws.h_status[i]);
        pending_cnt[slot] = 0;
        return Status::Ok();
    };
    auto submit = [&](int slot, uint64_t first, int cnt) -> Status {
        Workspace& ws = *W[slot];
        const cudaStream_t st = ws.stream;
        int np = 0;
        int* off = piece_off[slot];
        int* len = piece_len[slot];
        const int n_p = std::min(Workspace::MAX_SUB, (cnt + 127) / 128), per = (cnt + n_p - 1) / n_p;
        for (int o = 0; o < cnt; o += per) { off[np] = o; len[np++] = std::min(per, cnt - o); }
        EKZG_CUDA(cudaStreamWaitEvent(ws.in_stream, ws.done, 0));   // (the previous chunk of this workspace has left the buffers)
        EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * cnt, st));
        // Valid items' cells are packed from cell 0 of d_rcells on; they fill at most 128 (cnt - invalid items) cells, so with an
        // invalid item in the chunk the last 128 cells of the chunk's rows are free: zeroed, they are the cells of every invalid item.
        const uint64_t zero_off = (uint64_t)(cnt - 1) * N_CELLS;
        if (std::any_of(code.begin() + first, code.begin() + first + cnt, [](uint8_t c) { return c != 0; }))
            EKZG_CUDA(cudaMemsetAsync(ws.d_rcells + zero_off * BYTES_PER_CELL, 0, (size_t)N_CELLS * BYTES_PER_CELL, ws.in_stream));
        uint64_t packed = 0;   // cells of the chunk's valid items so far
        for (int s = 0; s < np; s++) {
            const int o = off[s], c = len[s];
            for (int i = o; i < o + c;) {
                const uint64_t g = first + i;
                if (code[g]) {
                    fill_slotmap(ws.h_slotmap + (size_t)i * N_CELLS, nullptr, 0, true);
                    ws.h_cell_off[i++] = (uint32_t)zero_off;
                    continue;
                }
                int j = i;   // a run of valid items [i, j): their cells are contiguous in the caller's buffer and on the device
                for (; j < o + c && !code[first + j]; j++) {
                    fill_slotmap(ws.h_slotmap + (size_t)j * N_CELLS, indices + offset[first + j], counts[first + j], false);
                    ws.h_cell_off[j] = (uint32_t)(packed + offset[first + j] - offset[g]);
                }
                const uint64_t run = offset[first + j] - offset[g];
                EKZG_TRY(upload(ws.d_rcells + packed * BYTES_PER_CELL, ws.h_rcells + packed * BYTES_PER_CELL, cells + offset[g] * BYTES_PER_CELL,
                                BYTES_PER_CELL, 0, (int)run, in_pinned, ws.in_stream));
                packed += run;
                i = j;
            }
            EKZG_CUDA(cudaMemcpyAsync(ws.d_slotmap + (size_t)o * N_CELLS, ws.h_slotmap + (size_t)o * N_CELLS, (size_t)c * N_CELLS * sizeof(int16_t),
                                      cudaMemcpyHostToDevice, ws.in_stream));
            EKZG_CUDA(cudaMemcpyAsync(ws.d_cell_off + o, ws.h_cell_off + o, (size_t)c * sizeof(uint32_t), cudaMemcpyHostToDevice, ws.in_stream));
            EKZG_CUDA(cudaEventRecord(ws.piece_in[s], ws.in_stream));
            EKZG_CUDA(cudaStreamWaitEvent(st, ws.piece_in[s], 0));
            EKZG_CUDA(launch_recover_coeffs(ws.d_rcells, ws.d_slotmap + (size_t)o * N_CELLS, ws.d_ze + (size_t)o * N_CELLS, ws.d_czinv + (size_t)o * N_CELLS,
                                            reinterpret_cast<Fr*>(ws.d_scalars) + (size_t)o * N_EXT, reinterpret_cast<Fr*>(ws.d_cells) + (size_t)o * N_EXT,
                                            ws.d_coeffs + (size_t)o * N_BLOB, ws.d_status + o, T_, coset_shift_fwd_, coset_shift_inv_,
                                            fr_coset_gen_pow64().v, c, st, ws.d_cell_off + o));
            EKZG_CUDA(launch_coeffs_to_blob(ws.d_coeffs + (size_t)o * N_BLOB, ws.d_blobs + (size_t)o * BYTES_PER_BLOB, T_, c, st));
            EKZG_CUDA(cudaEventRecord(ws.sub_ready[s], st));
            EKZG_CUDA(cudaStreamWaitEvent(ws.copy_stream, ws.sub_ready[s], 0));
            uint8_t* dst = out_pinned ? out_blobs + (first + o) * BYTES_PER_BLOB : ws.h_blobs + (size_t)o * BYTES_PER_BLOB;
            EKZG_CUDA(cudaMemcpyAsync(dst, ws.d_blobs + (size_t)o * BYTES_PER_BLOB, (size_t)c * BYTES_PER_BLOB, cudaMemcpyDeviceToHost, ws.copy_stream));
            EKZG_CUDA(cudaEventRecord(ws.sub_out[s], ws.copy_stream));
        }
        EKZG_CUDA(cudaMemcpyAsync(ws.h_status, ws.d_status, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaStreamWaitEvent(st, ws.sub_out[np - 1], 0));   // `done` also covers the last blobs' D2H
        EKZG_CUDA(cudaEventRecord(ws.done, st));
        pending_first[slot] = first;
        pending_cnt[slot] = cnt;
        pending_np[slot] = np;
        tr.mark("chunk enqueued");
        return Status::Ok();
    };
    for (uint64_t c = 0; c < nchunks && result.ok; c++) {
        const int slot = (int)(c & 1);
        result = drain(slot);
        if (result.ok) result = submit(slot, c * cap, (int)std::min<uint64_t>(cap, n - c * cap));
    }
    for (int slot = 0; slot < 2; slot++) {
        if (!W[slot]) continue;
        if (result.ok) result = drain(slot);
        give_back(W[slot], result);
    }
    tr.mark("H2D + kernels + D2H of the chunks");
    if (item_status) memcpy(item_status, code.data(), n);
    if (!result.ok) return result;
    if (first_err.empty())   // no index errors: the first item the device flagged, as recover_impl reports it
        for (uint64_t i = 0; i < n && first_err.empty(); i++)
            if (code[i]) first_err = item_status_text(code[i], true, false);
    if (!first_err.empty()) return Status::Error(first_err);
    return Status::Ok();
}

// ------------------------------------------------------------------------------------------------
// EIP-4844 prover side.  One code path for the three functions; chunks of up to chunk_capacity() blobs.
Status Context::run_4844(Mode4844 mode, uint64_t n, const uint8_t* blobs, const uint8_t* aux_in, uint8_t* out48, uint8_t* out_y32,
                         uint8_t* item_status) const {
    if (n == 0) return Status::Ok();
    EKZG_TRY(bind_device());
    const int cap = (int)std::min<uint64_t>(n, (uint64_t)chunk_capacity());
    Workspace* wsp = acquire(cap, true);
    if (!wsp) return Status::Error("device/pinned memory allocation failed");
    Workspace& ws = *wsp;
    cudaStream_t st = ws.stream;
    bool bad_blob = false, bad_aux = false;
    Status result = Status::Ok();
    std::vector<uint32_t> hs(cap), hs2(cap);
    TraceClock tr(mode == Mode4844::Commit ? "blob_to_kzg_commitment_batch" : "compute_(blob_)kzg_proof_batch");
    const bool in_pinned = host_range_is_pinned(blobs);
    auto body = [&](uint64_t first, int cnt) -> Status {
        if (mode == Mode4844::BlobProof) {
            // commitment validation (decompress + subgroup check) is independent of the blob pipeline: side stream
            EKZG_CUDA(cudaMemsetAsync(ws.d_status2, 0, sizeof(uint32_t) * cnt, st));
            EKZG_CUDA(cudaMemcpyAsync(ws.d_c48, aux_in + first * 48, (size_t)cnt * 48, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaEventRecord(ws.sub_ready[0], st));
            EKZG_CUDA(cudaStreamWaitEvent(ws.copy_stream, ws.sub_ready[0], 0));
            EKZG_CUDA(launch_g1_validate(ws.d_c48, ws.d_aff, ws.d_status2, cnt, true, ws.copy_stream));
            EKZG_CUDA(cudaEventRecord(ws.sub_out[0], ws.copy_stream));
        }
        EKZG_TRY(upload_blobs(ws, blobs + first * BYTES_PER_BLOB, 0, cnt, in_pinned, st));
        tr.mark("stage + enqueue H2D of the blobs");
        EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * cnt, st));
        if (mode != Mode4844::BlobProof) EKZG_CUDA(cudaMemsetAsync(ws.d_status2, 0, sizeof(uint32_t) * cnt, st));
        EKZG_CUDA(launch_blob_to_coeffs_cells(ws.d_blobs, ws.d_coeffs, nullptr, ws.d_status, T_, cnt, false, st));
        if (mode == Mode4844::Commit) {
            EKZG_TRY(commit_device(ws, cnt, ws.d_out48, st));
        } else {
            if (mode == Mode4844::BlobProof && n <= (uint64_t)HOST_CHALLENGE_MAX) {
                // a handful of blobs: Fiat-Shamir challenges on the host (see host_blob_challenge), uploaded like user-supplied points
                std::vector<uint8_t> zb((size_t)cnt * 32);
                for (int i = 0; i < cnt; i++) host_blob_challenge(blobs + (first + i) * BYTES_PER_BLOB, aux_in + (first + i) * 48, &zb[(size_t)i * 32]);
                EKZG_CUDA(cudaMemcpyAsync(ws.d_z32, zb.data(), zb.size(), cudaMemcpyHostToDevice, st));
                EKZG_CUDA(cudaStreamSynchronize(st));   // zb is pageable and dies with this scope
                EKZG_CUDA(launch_scalars_from_be(ws.d_z32, ws.d_z, nullptr, cnt, st));
            } else if (mode == Mode4844::BlobProof) {
                EKZG_CUDA(launch_blob_challenge(ws.d_blobs, ws.d_c48, ws.d_z, cnt, st));
            } else {
                EKZG_CUDA(cudaMemcpyAsync(ws.d_z32, aux_in + first * 32, (size_t)cnt * 32, cudaMemcpyHostToDevice, st));
                EKZG_CUDA(launch_scalars_from_be(ws.d_z32, ws.d_z, ws.d_status2, cnt, st));
            }
            EKZG_CUDA(launch_quotient(ws.d_coeffs, ws.d_z, ws.d_scalars, mode == Mode4844::PointProof ? ws.d_z32 : nullptr, cnt, st));
            EKZG_TRY(srs_msm_compress(ws, cnt, ws.d_out48, st));
        }
        EKZG_CUDA(cudaMemcpyAsync(out48 + first * 48, ws.d_out48, (size_t)cnt * 48, cudaMemcpyDeviceToHost, st));
        if (mode == Mode4844::PointProof) EKZG_CUDA(cudaMemcpyAsync(out_y32 + first * 32, ws.d_z32, (size_t)cnt * 32, cudaMemcpyDeviceToHost, st));
        if (mode == Mode4844::BlobProof) EKZG_CUDA(cudaStreamWaitEvent(st, ws.sub_out[0], 0));
        EKZG_CUDA(cudaMemcpyAsync(hs.data(), ws.d_status, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaMemcpyAsync(hs2.data(), ws.d_status2, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaStreamSynchronize(st));
        tr.mark("H2D + kernels + D2H");
        for (int i = 0; i < cnt; i++) {
            const uint8_t code = hs[i] ? ITEM_NON_CANONICAL : (hs2[i] ? ITEM_BAD_AUX : ITEM_OK);
            if (code == ITEM_NON_CANONICAL) bad_blob = true;
            if (code == ITEM_BAD_AUX) bad_aux = true;
            if (item_status) item_status[first + i] = code;
        }
        return Status::Ok();
    };
    for (uint64_t first = 0; first < n && result.ok; first += cap) result = body(first, (int)std::min<uint64_t>(cap, n - first));
    give_back(wsp, result);
    if (!result.ok) return result;
    if (bad_blob) return Status::Error(item_status_text(ITEM_NON_CANONICAL, false, false));
    if (bad_aux) return Status::Error(item_status_text(ITEM_BAD_AUX, false, mode == Mode4844::PointProof));
    return Status::Ok();
}

Status Context::blob_to_kzg_commitment_batch(uint64_t n, const uint8_t* blobs, uint8_t* out48, uint8_t* item_status) const {
    return run_4844(Mode4844::Commit, n, blobs, nullptr, out48, nullptr, item_status);
}
Status Context::compute_blob_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments48, uint8_t* out48,
                                             uint8_t* item_status) const {
    return run_4844(Mode4844::BlobProof, n, blobs, commitments48, out48, nullptr, item_status);
}
Status Context::compute_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* z32, uint8_t* out_proof48, uint8_t* out_y32,
                                        uint8_t* item_status) const {
    return run_4844(Mode4844::PointProof, n, blobs, z32, out_proof48, out_y32, item_status);
}

// ------------------------------------------------------------------------------------------------
// The cell proofs of whole blobs, by recomputation: a blob has exactly one valid proof per cell, and the FK20 pipeline computes
// all 128 of them, so the check is a byte comparison -- no cells cross PCIe, no transcript hash, no randomness, and a verdict per
// cell.  Chunks and the two alternating workspaces as in compute_cells_and_kzg_proofs_batch; all kernels of a chunk on ws.stream.
Status Context::verify_blob_cell_proofs_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                              uint8_t* item_status, uint8_t* cell_status, bool* all_ok) const {
    *all_ok = n == 0;
    if (n == 0) return Status::Ok();
    EKZG_TRY(bind_device());
    const int cap = (int)std::min<uint64_t>(n, (uint64_t)chunk_capacity());
    const uint64_t nchunks = (n + cap - 1) / cap;
    const ProofRoute route = proof_route(n, cap, true);
    Workspace* W[2] = {acquire(route.capacity, true), nchunks > 1 ? acquire(cap, true) : nullptr};
    Status result = Status::Ok();
    if (!W[0] || (nchunks > 1 && !W[1])) result = Status::Error("device/pinned memory allocation failed");
    for (Workspace* w : W)
        if (w && result.ok) result = w->ensure_verify_buffers(cap);
    if (!result.ok) {
        for (Workspace* w : W) if (w) give_back(w, result);
        return result;
    }
    const bool blobs_pinned = host_range_is_pinned(blobs), c_pinned = host_range_is_pinned(commitments), p_pinned = host_range_is_pinned(proofs);
    std::vector<uint8_t> cell_mm((size_t)n * N_CELLS), blob_mm(n);
    TraceClock tr("verify_blob_cell_proofs_batch");
    uint64_t pending_first[2] = {0, 0};
    int pending_cnt[2] = {0, 0};
    auto drain = [&](int slot) -> Status {
        Workspace& ws = *W[slot];
        if (!pending_cnt[slot]) return Status::Ok();
        EKZG_CUDA(cudaEventSynchronize(ws.done));
        memcpy(&cell_mm[pending_first[slot] * N_CELLS], ws.h_cell_mm, (size_t)pending_cnt[slot] * N_CELLS);
        memcpy(&blob_mm[pending_first[slot]], ws.h_blob_mm, (size_t)pending_cnt[slot]);
        pending_cnt[slot] = 0;
        return Status::Ok();
    };
    auto submit = [&](int slot, uint64_t first, int cnt) -> Status {
        Workspace& ws = *W[slot];
        const cudaStream_t st = ws.stream;
        EKZG_CUDA(cudaStreamWaitEvent(ws.in_stream, ws.done, 0));
        EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * cnt, st));
        // the blobs in the prover's pieces: K1 (once: the coefficients both the proofs and the commitment are computed from), K2
        // and K4 of the first piece run while the rest is on the wire
        const int q = fk20_first_piece(cnt);
        const int off[2] = {0, q}, len[2] = {q, cnt - q};
        for (int s = 0; s < 2 && len[s]; s++) {
            EKZG_TRY(upload(ws.d_blobs, ws.h_blobs, blobs + first * BYTES_PER_BLOB, BYTES_PER_BLOB, off[s], len[s], blobs_pinned, ws.in_stream));
            EKZG_CUDA(cudaEventRecord(ws.piece_in[s], ws.in_stream));
            EKZG_CUDA(cudaStreamWaitEvent(st, ws.piece_in[s], 0));
            EKZG_CUDA(launch_blob_to_coeffs_cells(ws.d_blobs + (size_t)off[s] * BYTES_PER_BLOB, ws.d_coeffs + (size_t)off[s] * N_BLOB, nullptr,
                                                  ws.d_status + off[s], T_, len[s], false, st));
            if (!route.direct) EKZG_TRY(fk20_msm(ws, cnt, off[s], len[s], st, nullptr));
        }
        EKZG_TRY(upload(ws.d_given_proofs, ws.h_proofs, proofs + first * PROOFS_PER_BLOB, PROOFS_PER_BLOB, 0, cnt, p_pinned, ws.in_stream));
        EKZG_TRY(upload(ws.d_c48, ws.h_c48, commitments + first * BYTES_PER_G1, BYTES_PER_G1, 0, cnt, c_pinned, ws.in_stream));
        EKZG_CUDA(cudaEventRecord(ws.piece_in[2], ws.in_stream));   // (after the two pieces of blobs)
        if (route.direct) EKZG_TRY(proofs_direct_device(ws, cnt, ws.d_proofs, st));
        else EKZG_TRY(fk20_ntt_compress(ws, cnt, ws.d_proofs, st, nullptr));
        // The commitment reuses d_scalars and d_pts, which the proofs are done with once they are compressed (K6, or the direct
        // route's compression).  d_coeffs is still intact: K2 and the direct route's quotient kernel only read it.  On the direct
        // route the workspace holds 128 cnt "virtual blobs", far more than the cnt items of the commitment MSM.
        EKZG_TRY(commit_device(ws, cnt, ws.d_out48, st));
        EKZG_CUDA(cudaStreamWaitEvent(st, ws.piece_in[2], 0));   // the supplied proofs and commitments are on the device
        EKZG_CUDA(launch_compare_blob_proofs(ws.d_proofs, ws.d_given_proofs, ws.d_out48, ws.d_c48, ws.d_status, ws.d_cell_mm, ws.d_blob_mm, cnt, st));
        EKZG_CUDA(cudaMemcpyAsync(ws.h_cell_mm, ws.d_cell_mm, (size_t)cnt * N_CELLS, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaMemcpyAsync(ws.h_blob_mm, ws.d_blob_mm, (size_t)cnt, cudaMemcpyDeviceToHost, st));
        EKZG_CUDA(cudaEventRecord(ws.done, st));
        pending_first[slot] = first;
        pending_cnt[slot] = cnt;
        return Status::Ok();
    };
    for (uint64_t c = 0; c < nchunks && result.ok; c++) {
        const int slot = (int)(c & 1);
        result = drain(slot);
        if (result.ok) result = submit(slot, c * cap, (int)std::min<uint64_t>(cap, n - c * cap));
    }
    for (int slot = 0; slot < 2 && result.ok; slot++)
        if (W[slot]) result = drain(slot);
    tr.mark("H2D + kernels + D2H of the chunks");

    // Phase B, only where a comparison failed: is the differing encoding a valid point (verdict 1) or not (2)?  A byte-equal
    // encoding needs no check -- the library's own compression output is canonical and valid -- so an honest batch launches no
    // validation kernel.  Encodings of non-canonical blobs are skipped: those items are 2 whatever they hold.
    std::vector<uint8_t> enc;
    for (uint64_t i = 0; i < n && result.ok; i++) {
        if (blob_mm[i] & BLOB_MM_NON_CANONICAL) continue;
        if (blob_mm[i] & BLOB_MM_COMMITMENT) enc.insert(enc.end(), commitments + i * BYTES_PER_G1, commitments + (i + 1) * BYTES_PER_G1);
        if (blob_mm[i] & BLOB_MM_PROOF)
            for (int k = 0; k < N_CELLS; k++)
                if (cell_mm[i * N_CELLS + k]) {
                    const uint8_t* p = proofs + (i * N_CELLS + k) * BYTES_PER_G1;
                    enc.insert(enc.end(), p, p + BYTES_PER_G1);
                }
    }
    const size_t m = enc.size() / BYTES_PER_G1;
    tr.mark("phase B: gather");
    std::vector<uint32_t> invalid(m);
    if (m && result.ok) {
        uint8_t* d_enc = nullptr;
        G1Affine* d_aff = nullptr;
        uint32_t* d_st = nullptr;
        const cudaStream_t st = W[0]->stream;
        // stream-ordered allocations: cudaMalloc / cudaFree would wait for the work of every other caller on the device
        auto validate = [&]() -> Status {
            EKZG_CUDA(cudaMallocAsync(&d_enc, enc.size(), st));
            EKZG_CUDA(cudaMallocAsync(&d_aff, m * sizeof(G1Affine), st));
            EKZG_CUDA(cudaMallocAsync(&d_st, m * sizeof(uint32_t), st));
            EKZG_CUDA(cudaMemcpyAsync(d_enc, enc.data(), enc.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(launch_g1_validate(d_enc, d_aff, d_st, (int)m, true, st));
            EKZG_CUDA(cudaMemcpyAsync(invalid.data(), d_st, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            return Status::Ok();
        };
        result = validate();
        for (void* p : {(void*)d_enc, (void*)d_aff, (void*)d_st}) if (p) cudaFreeAsync(p, st);
        const cudaError_t e = cudaStreamSynchronize(st);   // (also when a step failed: the copies may still read `enc` / write `invalid`)
        if (result.ok && e != cudaSuccess) result = Status::Error(std::string("CUDA error: ") + cudaGetErrorString(e) + " in phase B");
        if (!result.ok) cudaGetLastError();
        tr.mark("phase B: validate");
    }
    for (Workspace* w : W) if (w) give_back(w, result);
    if (!result.ok) return result;

    // The verdicts.  Why comparing bytes decides what the reference verifier decides, opening by opening:
    //  - C = commit(p): the single-cell equation e(C - [I_k(tau)]_1, [1]_2) = e(pi, [tau^64 - h_k^64]_2) has exactly one solution
    //    pi (the G2 factor is not the identity, and pairing with it is injective on G1), and that solution is [q_k(tau)], the FK20
    //    output for cell k.  So cell verdict 0 <=> the reference accepts that opening, exactly.
    //  - C != commit(p): the reference could accept all 128 openings only if C opened to p at all 8192 points, i.e. C committed to
    //    p -- a break of KZG binding.  So the blob verdicts agree except on inputs nobody can produce.
    //  - Where the two differ: per opening, with C != commit(p), the reference can accept opening k (for example when C commits to
    //    p + c (X^64 - h_k^64), which agrees with p on coset k); this call reports the blob as failing and the cell by its proof.
    //  - The reference's batch check is itself probabilistic (error <= n / |Fr|); this one is deterministic.
    // cell_status therefore states a fact about the proof and the blob alone and does not depend on C.
    bool ok = true;
    size_t j = 0;   // walks `invalid` in the order phase B gathered the encodings
    for (uint64_t i = 0; i < n; i++) {
        uint8_t* cs = &cell_mm[i * N_CELLS];
        uint8_t v = VERDICT_OK;
        if (blob_mm[i] & BLOB_MM_NON_CANONICAL) {
            v = VERDICT_MALFORMED;   // (the kernel wrote 2 for every cell)
        } else {
            bool malformed = false, fails = false;
            if (blob_mm[i] & BLOB_MM_COMMITMENT) (invalid[j++] ? malformed : fails) = true;
            if (blob_mm[i] & BLOB_MM_PROOF)
                for (int k = 0; k < N_CELLS; k++)
                    if (cs[k]) {
                        cs[k] = invalid[j++] ? VERDICT_MALFORMED : VERDICT_FAILS;
                        (cs[k] == VERDICT_MALFORMED ? malformed : fails) = true;
                    }
            v = malformed ? VERDICT_MALFORMED : (fails ? VERDICT_FAILS : VERDICT_OK);
        }
        item_status[i] = v;
        ok = ok && v == VERDICT_OK;
    }
    // the gather loop and this one must visit the mismatches in the same order: if they ever disagree, fail rather than hand
    // out verdicts that belong to other encodings
    if (j != m) return Status::Error("verify_blob_cell_proofs_batch: phase B consumed " + std::to_string(j) + " of " + std::to_string(m) + " validations");
    if (cell_status) memcpy(cell_status, cell_mm.data(), cell_mm.size());
    *all_ok = ok;
    return Status::Ok();
}

}  // namespace ekzg
