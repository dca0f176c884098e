// extern "C" surface of libc_eth_kzg_b200.so (include/c_eth_kzg.h): pointer marshalling only, like the
// reference's bindings/c/src/*.rs.  Every function binds the context's device, so calls may come from
// any host thread (bindings/node calls from the libuv pool, SURVEY.md §8b "Threading").
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "../../include/c_eth_kzg.h"
#include "kzg_multi.h"
#include "host_pairing.h"

using ekzg::Status;
namespace ekzg { double probe_imad_wide_per_s(int reps); }   // kzg_probe.cu

struct DASContext {
    std::unique_ptr<ekzg::DeviceSet> set;   // one ekzg::Context per device of EKZG_DEVICES (default: the current device)
};

// Every entry point binds the device(s) of its context on the calling thread; the caller's own current device is put
// back on return, so the library has no side effect on the CUDA state of the host application.
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static CResult c_ok() { return CResult{Ok, nullptr}; }
static CResult c_err(const std::string& m) {
    char* p = (char*)malloc(m.size() + 1);
    if (p) memcpy(p, m.c_str(), m.size() + 1);
    return CResult{Err, p};
}
static CResult to_c(const Status& s) { return s.ok ? c_ok() : c_err(s.msg); }
static const ekzg::DeviceSet& ds(const DASContext* ctx) {
    if (!ctx) {  // the reference asserts (bindings/c/src/lib.rs: `assert!(!ctx.is_null())`) and aborts
        fprintf(stderr, "c_eth_kzg_b200: null DASContext\n");
        abort();
    }
    return *ctx->set;
}
static const ekzg::Context& cx(const DASContext* ctx) { return ds(ctx).primary(); }      // calls that use one device
static const ekzg::Context& next_cx(const DASContext* ctx) { return ds(ctx).next(); }    // single-item calls: round-robin

// The two stage hooks: one blob through K1, K2 and K4 (the kernels without scratch) on a borrowed workspace's stream, then
// tail(ws, stream), which returns its failing step or nullptr.  Synchronous.
template <class Tail>
static CResult debug_fk20_run(const DASContext* ctx, const uint8_t* blob, Tail tail) {
    using namespace ekzg;
    DeviceGuard guard;
    const Context& c = cx(ctx);
    Status s = c.bind_device();
    if (!s.ok) return c_err(s.msg);
    Workspace* ws = c.acquire(1, true);
    if (!ws) return c_err("allocation failed");
    cudaStream_t st = ws->stream;
    const DevTables& T = c.tables();
    auto run = [&]() -> const char* {
        if (cudaMemcpyAsync(ws->d_blobs, blob, BYTES_PER_BLOB, cudaMemcpyHostToDevice, st) != cudaSuccess) return "h2d";
        cudaMemsetAsync(ws->d_status, 0, 4, st);
        if (launch_blob_to_coeffs_cells(ws->d_blobs, ws->d_coeffs, ws->d_cells, ws->d_status, T, 1, true, st) != cudaSuccess) return "k1";
        if (launch_toeplitz_scalars(ws->d_coeffs, ws->d_scalars, T, 1, st) != cudaSuccess) return "k2";
        if (launch_fixed_msm(ws->d_scalars, ws->d_pts, T.fk20, FK20_MSMS, 1, st) != cudaSuccess) return "k4";
        if (const char* m = tail(*ws, st)) return m;
        const cudaError_t e = cudaStreamSynchronize(st);
        return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
    };
    const char* m = run();
    c.give_back(ws, m ? Status::Error(m) : Status::Ok());
    return m ? c_err(m) : c_ok();
}

extern "C" {

DASContext* eth_kzg_das_context_new(bool use_precomp) {
    DeviceGuard guard;
    std::unique_ptr<ekzg::DeviceSet> c;
    Status s = ekzg::DeviceSet::create(use_precomp, &c);
    if (!s.ok) {
        fprintf(stderr, "c_eth_kzg_b200: context creation failed: %s\n", s.msg.c_str());
        return nullptr;
    }
    DASContext* d = new DASContext();
    d->set = std::move(c);
    return d;
}

CResult eth_kzg_b200_das_context_new_from_json(const char* json, uint64_t json_len, bool subgroup_check, bool use_precomp, DASContext** out_ctx) {
    DeviceGuard guard;
    if (!out_ctx) return c_err("out_ctx is null");
    *out_ctx = nullptr;
    ekzg::SetupBytes setup;
    Status s = ekzg::parse_trusted_setup_json(json, (size_t)json_len, &setup);
    if (!s.ok) return to_c(s);
    setup.subgroup_check = subgroup_check;
    std::unique_ptr<ekzg::DeviceSet> c;
    s = ekzg::DeviceSet::create(use_precomp, &c, &setup);
    if (!s.ok) return to_c(s);
    DASContext* d = new DASContext();
    d->set = std::move(c);
    *out_ctx = d;
    return c_ok();
}

// Test hooks (host only, need no GPU): the JSON parser (returns the point counts) and the G2 decompression of the setup loader.
CResult eth_kzg_b200_debug_parse_trusted_setup_json(const char* json, uint64_t json_len, uint64_t* n_g1, uint64_t* n_g2, uint8_t* first_g1_48,
                                                    uint8_t* last_g2_96) {
    ekzg::SetupBytes setup;
    Status s = ekzg::parse_trusted_setup_json(json, (size_t)json_len, &setup);
    if (!s.ok) return to_c(s);
    *n_g1 = setup.g1_monomial.size() / 48;
    *n_g2 = setup.g2_monomial.size() / 96;
    if (first_g1_48 && *n_g1) memcpy(first_g1_48, setup.g1_monomial.data(), 48);
    if (last_g2_96 && *n_g2) memcpy(last_g2_96, setup.g2_monomial.data() + setup.g2_monomial.size() - 96, 96);
    return c_ok();
}
int eth_kzg_b200_debug_g2_decompress(const uint8_t* in96, uint64_t* out24) { return ekzg::host::g2_decompress_plain(in96, out24); }
CResult eth_kzg_b200_debug_g2_keys(const uint8_t* g2_65x96, int count, bool subgroup_check) {
    std::string err;
    ekzg::host::G2Keys* k = ekzg::host::g2_keys_from_compressed(g2_65x96, count, subgroup_check, &err);
    if (!k) return c_err(err);
    ekzg::host::g2_keys_free(k);
    return c_ok();
}

void eth_kzg_das_context_free(DASContext* ctx) {
    DeviceGuard guard;
    if (ctx) delete ctx;
}

void eth_kzg_free_error_message(char* c_message) {
    if (c_message) free(c_message);
}

uint64_t eth_kzg_constant_bytes_per_cell(void) { return ekzg::BYTES_PER_CELL; }
uint64_t eth_kzg_constant_bytes_per_proof(void) { return ekzg::BYTES_PER_G1; }
uint64_t eth_kzg_constant_cells_per_ext_blob(void) { return ekzg::N_CELLS; }

CResult eth_kzg_compute_cells_and_kzg_proofs(const DASContext* ctx, const uint8_t* blob, uint8_t** out_cells, uint8_t** out_proofs) {
    DeviceGuard guard;   // results go through the 128 + 128 pointers on the caller's own thread (pointer_utils.rs:53-62 write_to_2d_slice)
    return to_c(next_cx(ctx).compute_cells_and_kzg_proofs_one(blob, nullptr, nullptr, out_cells, out_proofs, true));
}

CResult eth_kzg_compute_cells(const DASContext* ctx, const uint8_t* blob, uint8_t** out_cells) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).compute_cells_and_kzg_proofs_one(blob, nullptr, nullptr, out_cells, nullptr, false));
}

CResult eth_kzg_b200_compute_cells_and_kzg_proofs_batch(const DASContext* ctx, uint64_t n, const uint8_t* blobs, uint8_t* out_cells,
                                                        uint8_t* out_proofs, uint8_t* blob_status) {
    DeviceGuard guard;
    return to_c(ds(ctx).compute_cells_and_kzg_proofs_batch(n, blobs, out_cells, out_proofs, blob_status, out_proofs != nullptr));
}

CResult eth_kzg_b200_compute_cells_and_kzg_proofs_device(const DASContext* ctx, uint64_t n, const void* d_blobs, void* d_cells,
                                                         void* d_proofs, void* d_status, void* cuda_stream) {
    DeviceGuard guard;
    if (n == 0) return c_ok();
    if (n > (1u << 20)) return c_err("batch too large");
    const ekzg::Context* owner = ds(ctx).size() == 1 ? &cx(ctx) : ds(ctx).owner_of(d_blobs);
    if (!owner) return c_err("the device buffers are not on a device of this context (EKZG_DEVICES)");
    const ekzg::Context& c = *owner;
    Status s = c.bind_device();
    if (!s.ok) return c_err(s.msg);
    ekzg::Workspace* ws = c.acquire(ekzg::proof_route(n, (int)n, d_proofs != nullptr).capacity, false);
    if (!ws) return c_err("device memory allocation failed");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    cudaStreamWaitEvent(st, ws->done, 0);  // the scratch buffers' previous user may have run on another stream
    s = c.fk20_device(*ws, (int)n, (const uint8_t*)d_blobs, (uint8_t*)d_cells, (uint8_t*)d_proofs, (uint32_t*)d_status, st);
    // the scratch buffers are reused by the next call on this context: order later work after this batch -- also when the
    // call failed half way, because the kernels enqueued before the failure still run
    cudaEventRecord(ws->done, st);
    cudaStreamWaitEvent(ws->stream, ws->done, 0);
    if (!s.ok) cudaGetLastError();
    c.give_back(ws, s);
    return to_c(s);
}

int eth_kzg_b200_context_device(const DASContext* ctx) { return cx(ctx).device(); }
int eth_kzg_b200_context_window(const DASContext* ctx) { return cx(ctx).tables().fk20.w; }
int eth_kzg_b200_context_srs_window(const DASContext* ctx) { return cx(ctx).tables().srs.w; }
uint64_t eth_kzg_b200_context_table_bytes(const DASContext* ctx) { return cx(ctx).table_bytes(); }
int eth_kzg_b200_context_device_count(const DASContext* ctx) { return (int)ds(ctx).size(); }
int eth_kzg_b200_context_device_at(const DASContext* ctx, int i) { return i >= 0 && (size_t)i < ds(ctx).size() ? ds(ctx).at(i).device() : -1; }
uint64_t eth_kzg_b200_kernel_launch_count(void) { return ekzg::g_kernel_launches.load(); }

// Measured issue rate of carry-chained IMAD.WIDE on the context's first device, in multiply-adds per second
// (the roofline denominator of the point-arithmetic kernels; ~30 ms).  0 on error.
double eth_kzg_b200_probe_imad_wide(const DASContext* ctx) {
    DeviceGuard guard;
    if (!cx(ctx).bind_device().ok) return 0;
    return ekzg::probe_imad_wide_per_s(3);
}

// Test hook (host only): the contiguous shard [lo, lo + cnt) that device i of `parts` gets from a batch of n items
void eth_kzg_b200_debug_shard_bounds(uint64_t n, uint64_t parts, uint64_t i, uint64_t* lo, uint64_t* cnt) {
    ekzg::DeviceSet::shard_bounds(n, (size_t)parts, (size_t)i, lo, cnt);
}

void eth_kzg_b200_set_profiling(const DASContext* ctx, bool on) { cx(ctx).set_profiling(on); }
int eth_kzg_b200_collect_stage_times(const DASContext* ctx, double* ms_out) {
    for (int i = 0; i < ekzg::Context::N_STAGES; i++) ms_out[i] = 0;
    return cx(ctx).collect_stage_times(ms_out);
}

// Stage dump of one blob for kernel-level parity tests: plain scalars [128][64][8 x u32 LE],
// MSM outputs (natural j order) and h commitments as compressed points.  Synchronous; test hook.
CResult eth_kzg_b200_debug_fk20_stages(const DASContext* ctx, const uint8_t* blob, uint32_t* out_scalars, uint8_t* out_msm, uint8_t* out_h) {
    using namespace ekzg;
    uint8_t tmp[128 * 48];
    CResult res = debug_fk20_run(ctx, blob, [&](Workspace& ws, cudaStream_t st) -> const char* {
        // (K4 leaves the scalars as they are)
        if (cudaMemcpyAsync(out_scalars, ws.d_scalars, 128 * 64 * 32, cudaMemcpyDeviceToHost, st) != cudaSuccess) return "d2h scalars";
        // MSM outputs sit at bit-reversed positions; compress all 128 then un-permute on the host
        if (launch_g1_compress(ws.d_pts, ws.d_proofs, 128, 1, st) != cudaSuccess) return "k6";
        if (cudaMemcpyAsync(tmp, ws.d_proofs, sizeof(tmp), cudaMemcpyDeviceToHost, st) != cudaSuccess) return "d2h msm";
        if (launch_g1_ntt_phases(ws.d_pts, 1, 0, 7, ws.d_queue, ws.d_ntt_scratch, st) != cudaSuccess) return "k5";
        if (launch_g1_compress(ws.d_pts, ws.d_proofs, 64, 1, st) != cudaSuccess) return "k6b";
        if (cudaMemcpyAsync(out_h, ws.d_proofs, 64 * 48, cudaMemcpyDeviceToHost, st) != cudaSuccess) return "d2h h";
        return nullptr;
    });
    if (res.status != Ok) return res;
    for (int j = 0; j < 128; j++) {
        int r = 0;
        for (int b = 0; b < 7; b++) r |= ((j >> b) & 1) << (6 - b);
        memcpy(out_msm + 48 * j, tmp + 48 * r, 48);
    }
    return c_ok();
}

// Test hook: the 128 points of one blob after the first `phases` G1-NTT phases (0 = the MSM outputs as K4 stored them), compressed,
// in storage order.  With EKZG_K5_R4_MAX >= 1 and an even `phases` the radix-4 kernel runs its first phases / 2 super-phases.
CResult eth_kzg_b200_debug_g1_ntt_prefix(const DASContext* ctx, const uint8_t* blob, int phases, uint8_t* out128x48) {
    using namespace ekzg;
    if (phases < 0 || phases > 14) return c_err("phases out of range");
    return debug_fk20_run(ctx, blob, [&](Workspace& ws, cudaStream_t st) -> const char* {
        if (phases > 0 && launch_g1_ntt_phases(ws.d_pts, 1, 0, phases, ws.d_queue, ws.d_ntt_scratch, st) != cudaSuccess) return "k5";
        if (launch_g1_compress(ws.d_pts, ws.d_proofs, 128, 1, st) != cudaSuccess) return "k6";
        if (cudaMemcpyAsync(out128x48, ws.d_proofs, 128 * 48, cudaMemcpyDeviceToHost, st) != cudaSuccess) return "d2h";
        return nullptr;
    });
}

// Test hook (host only, needs no GPU): prod e(P_i, Q_i) == 1 for affine G1 points given as 96 bytes each (x then y, plain
// little-endian 64-bit limbs; all-zero = identity) and G2 selectors 0 [1]_2, 1 [tau]_2, 2 [tau^64]_2, +3 for the negation.
int eth_kzg_b200_debug_pairing_check(int n, const uint8_t* g1_xy, const int* g2_sel) {
    std::vector<ekzg::host::PairingInput> in(n);
    for (int i = 0; i < n; i++) {
        memcpy(in[i].g1_x, g1_xy + 96 * i, 48);
        memcpy(in[i].g1_y, g1_xy + 96 * i + 48, 48);
        bool z = true;
        for (int b = 0; b < 96; b++) z = z && g1_xy[96 * i + b] == 0;
        in[i].g1_is_identity = z;
        in[i].g2 = (ekzg::host::G2Sel)g2_sel[i];
    }
    return ekzg::host::pairing_check(in.data(), n) ? 1 : 0;
}

// Test hook (host only): the pairing's shortcut routines against its general ones; 1 = they agree
int eth_kzg_b200_debug_pairing_selftest(void) { return ekzg::host::pairing_selftest() ? 1 : 0; }

CResult eth_kzg_blob_to_kzg_commitment(const DASContext* ctx, const uint8_t* blob, uint8_t* out) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).blob_to_kzg_commitment_batch(1, blob, out, nullptr));
}
CResult eth_kzg_compute_kzg_proof(const DASContext* ctx, const uint8_t* blob, const uint8_t* z, uint8_t* out_proof, uint8_t* out_y) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).compute_kzg_proof_batch(1, blob, z, out_proof, out_y, nullptr));
}
CResult eth_kzg_compute_blob_kzg_proof(const DASContext* ctx, const uint8_t* blob, const uint8_t* commitment, uint8_t* out_proof) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).compute_blob_kzg_proof_batch(1, blob, commitment, out_proof, nullptr));
}
CResult eth_kzg_b200_blob_to_kzg_commitment_batch(const DASContext* ctx, uint64_t n, const uint8_t* blobs, uint8_t* out, uint8_t* item_status) {
    DeviceGuard guard;
    return to_c(ds(ctx).blob_to_kzg_commitment_batch(n, blobs, out, item_status));
}
CResult eth_kzg_b200_compute_blob_kzg_proof_batch(const DASContext* ctx, uint64_t n, const uint8_t* blobs, const uint8_t* commitments,
                                                  uint8_t* out_proofs, uint8_t* item_status) {
    DeviceGuard guard;
    return to_c(ds(ctx).compute_blob_kzg_proof_batch(n, blobs, commitments, out_proofs, item_status));
}
CResult eth_kzg_recover_cells_and_proofs(const DASContext* ctx, uint64_t cells_length, const uint8_t* const* cells, uint64_t cell_indices_length,
                                         const uint64_t* cell_indices, uint8_t** out_cells, uint8_t** out_proofs) {
    DeviceGuard guard;
    const ekzg::Context& c = next_cx(ctx);
    if (cells_length != cell_indices_length)  // recovery.rs:95-100
        return c_err("Recovery(NumCellIndicesNotEqualToNumCells)");
    if (cells_length > 4096) return c_err("Recovery(TooManyCellsReceived)");
    std::vector<uint8_t> flat((size_t)cells_length * ekzg::BYTES_PER_CELL);
    for (uint64_t i = 0; i < cells_length; i++) memcpy(flat.data() + i * ekzg::BYTES_PER_CELL, cells[i], ekzg::BYTES_PER_CELL);
    uint64_t cnt = cells_length;
    return to_c(c.recover_cells_and_kzg_proofs_one(cnt, cell_indices, flat.data(), nullptr, nullptr, out_cells, out_proofs));
}
CResult eth_kzg_b200_recover_cells_and_kzg_proofs_batch(const DASContext* ctx, uint64_t n, const uint64_t* cell_counts, const uint64_t* cell_indices,
                                                        const uint8_t* cells, uint8_t* out_cells, uint8_t* out_proofs, uint8_t* item_status) {
    DeviceGuard guard;
    return to_c(ds(ctx).recover_cells_and_kzg_proofs_batch(n, cell_counts, cell_indices, cells, out_cells, out_proofs, item_status));
}

CResult eth_kzg_verify_cell_kzg_proof_batch(const DASContext* ctx, uint64_t commitments_length, const uint8_t* const* commitments,
                                            uint64_t cell_indices_length, const uint64_t* cell_indices, uint64_t cells_length,
                                            const uint8_t* const* cells, uint64_t proofs_length, const uint8_t* const* proofs, bool* verified) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_cell_kzg_proof_batch(commitments_length, commitments, cell_indices_length, cell_indices, cells_length, cells,
                                                    proofs_length, proofs, verified));
}
CResult eth_kzg_verify_kzg_proof(const DASContext* ctx, const uint8_t* commitment, const uint8_t* z, const uint8_t* y, const uint8_t* proof,
                                 bool* verified) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_kzg_proofs(0, 1, nullptr, &commitment, z, y, &proof, verified));
}
CResult eth_kzg_verify_blob_kzg_proof(const DASContext* ctx, const uint8_t* blob, const uint8_t* commitment, const uint8_t* proof, bool* verified) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_kzg_proofs(1, 1, &blob, &commitment, nullptr, nullptr, &proof, verified));
}
CResult eth_kzg_verify_blob_kzg_proof_batch(const DASContext* ctx, uint64_t blobs_length, const uint8_t* const* blobs, uint64_t commitments_length,
                                            const uint8_t* const* commitments, uint64_t proofs_length, const uint8_t* const* proofs,
                                            bool* verified) {
    if (!(blobs_length == commitments_length && blobs_length == proofs_length)) {  // eip4844/src/verifier.rs:86-95
        *verified = false;
        return c_err("Verifier(BatchVerificationInputsMustHaveSameLength)");
    }
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_kzg_proofs(1, blobs_length, blobs, commitments, nullptr, nullptr, proofs, verified));
}

CResult eth_kzg_b200_verify_cell_kzg_proof_batch_groups(const DASContext* ctx, uint64_t n, const uint8_t* const* commitments,
                                                        const uint64_t* cell_indices, const uint8_t* const* cells, const uint8_t* const* proofs,
                                                        uint64_t n_groups, const uint32_t* group_of, uint8_t* group_status, bool* all_ok) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_cell_kzg_proof_batch_groups(n, commitments, cell_indices, cells, proofs, n_groups, group_of, group_status,
                                                                all_ok));
}
CResult eth_kzg_b200_verify_blob_kzg_proof_batch_items(const DASContext* ctx, uint64_t n, const uint8_t* const* blobs,
                                                       const uint8_t* const* commitments, const uint8_t* const* proofs, uint8_t* item_status,
                                                       bool* all_ok) {
    DeviceGuard guard;
    return to_c(next_cx(ctx).verify_kzg_proofs(1, n, blobs, commitments, nullptr, nullptr, proofs, all_ok, item_status));
}

}  // extern "C"
