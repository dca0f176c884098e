// Host runtime: context (per-device tables), workspaces (per-call device + pinned staging buffers),
// and the batch pipeline that replaces the reference's maybe_rayon fan-out (crates/maybe_rayon) with
// a GPU batch scheduler: many blobs per kernel launch, copies overlapped with compute on two streams.
#pragma once
#include <cuda_runtime.h>
#include <condition_variable>
#include <deque>
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <vector>
#include "kzg_kernels.h"
#include "host_pairing.h"

namespace ekzg {

struct Status {
    bool ok = true;
    std::string msg;
    static Status Ok() { return Status(); }
    static Status Error(const std::string& m) { Status s; s.ok = false; s.msg = m; return s; }
};

#define EKZG_CUDA(expr)                                                                                         \
    do {                                                                                                        \
        cudaError_t e_ = (expr);                                                                                \
        if (e_ != cudaSuccess) return ::ekzg::Status::Error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #expr); \
    } while (0)
#define EKZG_TRY(expr) do { ::ekzg::Status s_ = (expr); if (!s_.ok) return s_; } while (0)

// Per-item status codes of the batch calls (item_status / blob_status of the C ABI: the values are fixed).
enum ItemStatus : uint8_t {
    ITEM_OK = 0,
    ITEM_NON_CANONICAL = 1,   // a blob or cell field element is >= the scalar modulus
    ITEM_BAD_AUX = 2,         // compute_blob_kzg_proof: invalid commitment; compute_kzg_proof: non-canonical z
    ITEM_BAD_INDICES = 3,     // recovery: cell indices out of range, not ascending, too few or too many
    ITEM_BAD_DEGREE = 4,      // recovery: the recovered polynomial has degree >= 4096
};
// Verdicts of the verifiers that answer per group of openings / per blob (group_status / item_status of the C ABI: the
// values are fixed).
enum Verdict : uint8_t {
    VERDICT_OK = 0,          // verifies (an empty group too)
    VERDICT_FAILS = 1,       // well-formed, does not verify
    VERDICT_MALFORMED = 2,   // holds an invalid point encoding / subgroup, a non-canonical scalar or a cell index >= 128
};
constexpr uint64_t MAX_VERIFY_GROUPS = 1u << 20;
// The error text of an item with status `code`: `cells` -- its inputs were cells (recovery), not a blob; `z` -- its second
// input was an evaluation point, not a commitment.
const char* item_status_text(uint8_t code, bool cells, bool z);

// A caller-supplied trusted setup with its points still in compressed form: what TrustedSetup::from_json /
// from_json_unchecked (crates/trusted_setup/src/lib.rs:112-127) hand to DASContext::new (crates/eip7594/src/lib.rs).
struct SetupBytes {
    std::vector<uint8_t> g1_monomial;   // 4096 x 48 bytes
    std::vector<uint8_t> g2_monomial;   // 65 x 96 bytes
    bool subgroup_check = true;         // from_json: true; from_json_unchecked: false (curve equation only)
};
// The consensus-specs JSON layout ({"g1_monomial": ["0x..", ..], "g1_lagrange": [..], "g2_monomial": [..]}); keys other than
// g1_monomial and g2_monomial are skipped, as serde does for the reference's TrustedSetupJSON (trusted_setup_json.cpp).
Status parse_trusted_setup_json(const char* json, size_t len, SetupBytes* out);

// Device + pinned buffers for one in-flight chunk of up to `capacity` blobs.
struct Workspace {
    int capacity = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;          // D2H of the cells while the FK20 kernels run on `stream`
    cudaStream_t in_stream = nullptr;            // H2D of the blobs, piece by piece, ahead of the kernels on `stream`
    cudaStream_t aux_stream = nullptr;           // fourth lane for the verifier's independent latency-bound chains
    cudaEvent_t done = nullptr;
    static constexpr int MAX_SUB = 16;           // pieces of a chunk for copy-in / K1 / copy-out pipelining
    cudaEvent_t piece_in[MAX_SUB] = {};          // blobs of piece s are on the device (recorded on `in_stream`)
    cudaEvent_t sub_ready[MAX_SUB] = {};         // K1 of piece s finished (recorded on `stream`)
    cudaEvent_t sub_out[MAX_SUB] = {};           // cells of piece s are in host memory (recorded on `copy_stream`)
    // device
    uint8_t* d_blobs = nullptr;
    Fr* d_coeffs = nullptr;
    uint8_t* d_cells = nullptr;
    uint32_t* d_scalars = nullptr;
    G1Jac* d_pts = nullptr;
    uint32_t* d_queue = nullptr;   // ticket counter + per-unit completion flags of K5
    void* d_ntt_scratch = nullptr; // K5: odd-multiples tables of the resident warps (g1_ntt_scratch_bytes())
    void* d_msm_scratch = nullptr; // K4a: per-window affine accumulators of the resident CTAs (fixed_msm_scratch_bytes())
    uint8_t* d_proofs = nullptr;
    uint32_t* d_status = nullptr;
    // small per-blob side buffers of the 4844 path
    uint8_t* d_c48 = nullptr;      // commitments in (48 B)
    uint8_t* d_z32 = nullptr;      // evaluation points in / y out (32 B)
    uint8_t* d_out48 = nullptr;    // commitment / proof out (48 B)
    Fr* d_z = nullptr;
    G1Affine* d_aff = nullptr;
    uint32_t* d_status2 = nullptr;
    // recovery inputs (allocated on first use)
    uint8_t* d_rcells = nullptr;   // [cap][128 slots][2048]
    uint8_t* h_rcells = nullptr;
    int16_t* d_slotmap = nullptr;  // [cap][128]
    int16_t* h_slotmap = nullptr;
    Fr* d_ze = nullptr;            // [cap][128]
    Fr* d_czinv = nullptr;
    uint32_t* d_cell_off = nullptr;   // [cap] recover_blobs_batch: first cell of blob i in the packed d_rcells
    uint32_t* h_cell_off = nullptr;
    bool recover_ready = false;    // all eight recovery buffers exist
    Status ensure_recover_buffers();
    void free_recover_buffers();
    // verify_blob_cell_proofs_batch (allocated on first use, for the blobs per chunk a call needs -- not the workspace capacity,
    // which on the direct route counts 128 "virtual blobs" per blob; the supplied commitments go to d_c48, pageable proofs are
    // staged in h_proofs)
    uint8_t* d_given_proofs = nullptr;   // [vcap][128][48]
    uint8_t* d_cell_mm = nullptr;        // [vcap][128] per-cell comparison bytes, then d_blob_mm
    uint8_t* d_blob_mm = nullptr;        // [vcap] per-blob BLOB_MM_* bits
    uint8_t* h_cell_mm = nullptr;        // pinned, the same layout
    uint8_t* h_blob_mm = nullptr;
    uint8_t* h_c48 = nullptr;            // pinned staging of pageable commitments
    int verify_capacity = 0;             // vcap: blobs the buffers hold (0: none allocated)
    Status ensure_verify_buffers(int blobs);   // (re)allocates when fewer than `blobs` (<= capacity) fit
    void free_verify_buffers();
    // pinned host staging (the ABI hands us scattered caller buffers)
    uint8_t* h_blobs = nullptr;
    uint8_t* h_cells = nullptr;
    uint8_t* h_proofs = nullptr;
    uint32_t* h_status = nullptr;
    Status alloc(int cap, bool with_io, size_t msm_scratch_bytes);
    void synchronize() const;   // waits for the work queued on all four streams
    void release();
};

// Proof route of an n-blob call.  Up to EKZG_DIRECT_MAX blobs (default 1, 0 = off) take the DIRECT route (128 SRS MSMs per
// blob instead of FK20) when `eligible` (the call computes proofs and is not timed per FK20 stage).
struct ProofRoute {
    bool direct;
    int capacity;   // workspace capacity the call needs: 128 "virtual blobs" per blob on the direct route, else `fk20_capacity`
};
ProofRoute proof_route(uint64_t n, int fk20_capacity, bool eligible);

class Context {
public:
    // device < 0: the calling thread's current device (or EKZG_DEVICE)
    // custom == nullptr: the embedded mainnet ceremony output
    static Status create(bool use_precomp, std::unique_ptr<Context>* out, int device = -1, const SetupBytes* custom = nullptr);
    ~Context();

    int device() const { return device_; }
    const DevTables& tables() const { return T_; }
    uint64_t table_bytes() const { return table_bytes_; }
    const host::G2Keys* g2_keys() const { return g2keys_; }

    // Everything on device, asynchronous on `stream`; scratch comes from `ws` (capacity: proof_route(n, n, d_proofs).capacity).
    Status fk20_device(Workspace& ws, int n, const uint8_t* d_blobs, uint8_t* d_cells, uint8_t* d_proofs, uint32_t* d_status,
                       cudaStream_t stream) const;

    // Host buffers, contiguous; chunks the batch through two workspaces.
    Status compute_cells_and_kzg_proofs_batch(uint64_t n, const uint8_t* blobs, uint8_t* cells, uint8_t* proofs,
                                              uint8_t* blob_status, bool want_proofs) const;

    // One blob, as the reference's ABI hands them over (bindings/c/src/lib.rs:226-262), from any number of host threads at
    // once: concurrent callers are coalesced into batches (leader/follower: the first caller to find no batch in flight runs
    // one for everything queued, callers arriving meanwhile form the next).  This is what replaces the reference's per-call
    // rayon fan-out (crates/eip7594/src/prover.rs:117-148 over maybe_rayon): a lone blob fills 1 of the 32 lanes of every K5
    // work unit, 32 coalesced blobs cost the same time.  cells: 128*2048 B, proofs: 128*48 B or nullptr (compute_cells).
    // Outputs either contiguous (cells / proofs) or, as the C ABI hands them over, through 128 separate pointers each
    // (cells_scattered / proofs_scattered; bindings/c/src/pointer_utils.rs:53-62) -- the caller's own thread writes them.
    Status compute_cells_and_kzg_proofs_one(const uint8_t* blob, uint8_t* cells, uint8_t* proofs, uint8_t* const* cells_scattered,
                                            uint8_t* const* proofs_scattered, bool want_proofs) const;
    // the same for eth_kzg_recover_cells_and_proofs: `count` cells (contiguous) at `indices`
    Status recover_cells_and_kzg_proofs_one(uint64_t count, const uint64_t* indices, const uint8_t* cells, uint8_t* out_cells,
                                            uint8_t* out_proofs, uint8_t* const* cells_scattered, uint8_t* const* proofs_scattered) const;

    // EIP-4844 prover side (crates/eip4844/src/prover.rs:17-88), batched.  Host buffers, contiguous.
    // item_status[i]: ItemStatus 0, 1 or 2.
    Status blob_to_kzg_commitment_batch(uint64_t n, const uint8_t* blobs, uint8_t* out48, uint8_t* item_status) const;
    Status compute_blob_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments48, uint8_t* out48,
                                        uint8_t* item_status) const;
    Status compute_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* z32, uint8_t* out_proof48, uint8_t* out_y32,
                                   uint8_t* item_status) const;

    // Erasure recovery (crates/eip7594/src/prover.rs:156-171, recovery.rs:22-146), batched: blob i provides counts[i]
    // cells; indices and cells of all blobs are concatenated.  item_status: ItemStatus 0, 1, 3 or 4.
    // out_* contiguous per blob (128*2048 B, 128*48 B).
    Status recover_cells_and_kzg_proofs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells,
                                              uint8_t* out_cells, uint8_t* out_proofs, uint8_t* item_status) const;
    // The same recovery without proofs: out_blobs n x 131072 B, cells 0..63 of what the call above returns for the valid items.
    // Inputs, validation order, item_status and error texts as there; the blobs of invalid items are unspecified.
    Status recover_blobs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_blobs,
                               uint8_t* item_status) const;

    // Verifiers.  Err = malformed input, Ok + *verified = false = the proof does not check (bindings/c/src/lib.rs:272-280).
    Status verify_cell_kzg_proof_batch(uint64_t n_commitments, const uint8_t* const* commitments, uint64_t n_indices,
                                       const uint64_t* cell_indices, uint64_t n_cells, const uint8_t* const* cells, uint64_t n_proofs,
                                       const uint8_t* const* proofs, bool* verified) const;
    // The same check with a Verdict per caller-defined group of openings: group_of[n] < n_groups, group_status[n_groups].
    // *all_ok = every group is VERDICT_OK.  Err only for a group id >= n_groups or n_groups > MAX_VERIFY_GROUPS.
    Status verify_cell_kzg_proof_batch_groups(uint64_t n, const uint8_t* const* commitments, const uint64_t* cell_indices,
                                              const uint8_t* const* cells, const uint8_t* const* proofs, uint64_t n_groups,
                                              const uint32_t* group_of, uint8_t* group_status, bool* all_ok) const;
    // mode 0: verify_kzg_proof items (commitment, z, y, proof); mode 1: verify_blob_kzg_proof(_batch) items (blob, commitment, proof).
    // item_status (mode 1 only, optional): a Verdict per item instead of Err for malformed items; *verified = all are VERDICT_OK.
    Status verify_kzg_proofs(int mode, uint64_t n, const uint8_t* const* blobs, const uint8_t* const* commitments, const uint8_t* z32,
                             const uint8_t* y32, const uint8_t* const* proofs, bool* verified, uint8_t* item_status = nullptr) const;
    // The cell proofs of whole blobs (an EIP-7594 blob transaction): recomputes each blob's commitment and 128 proofs and compares
    // bytes.  Host buffers, contiguous: blobs n x 131072 B, commitments n x 48 B, proofs n x 128 x 48 B.  item_status[n]: a Verdict
    // per blob; cell_status[n][128] (optional): 0 the proof of cell k, 1 a valid point but not that proof, 2 not a valid encoding or
    // a non-canonical blob.  *all_ok = every item is VERDICT_OK.  Err only for allocation / CUDA failures.
    Status verify_blob_cell_proofs_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                         uint8_t* item_status, uint8_t* cell_status, bool* all_ok) const;

    // workspace pool (calls are re-entrant: concurrent callers each borrow their own workspaces)
    Workspace* acquire(int min_capacity, bool with_io) const;
    // `s`: the outcome of the call that borrowed `ws`.  After a failure the work queued before it may still be running: the
    // workspace's streams are synchronised before it is pooled, so the next borrower finds its buffers idle.
    void give_back(Workspace* ws, const Status& s) const;
    void discard(Workspace* ws) const;             // destroy instead of pooling (its buffers are incomplete)
    size_t trim_pool(size_t keep) const;           // release idle workspaces beyond `keep`

    Status bind_device() const;

    // Optional per-stage timing of fk20_device with CUDA events on the launching stream (bench.py's
    // live roofline figures).  Stages: 0 K1 blob->coeffs/cells, 1 K2 toeplitz scalars, 2 K4 MSM,
    // 3 K5 G1 NTTs, 4 K6 compress.  Not thread-safe: enable only from a single-threaded benchmark.
    static constexpr int N_STAGES = 5;
    void set_profiling(bool on) const;
    // accumulates finished batches into ms[N_STAGES], returns the number of batches accumulated
    int collect_stage_times(double* ms) const;

private:
    enum class Mode4844 { Commit, BlobProof, PointProof };
    Status run_4844(Mode4844 mode, uint64_t n, const uint8_t* blobs, const uint8_t* aux_in, uint8_t* out48, uint8_t* out_y32,
                    uint8_t* item_status) const;
    Context() = default;
    // both cell verifiers: n openings, lengths and (plain call) indices already checked; `groups` == nullptr: the plain call
    struct GroupVerdicts {
        const uint32_t* group_of;
        uint64_t n_groups;
        uint8_t* status;
    };
    Status verify_cells(uint64_t n, const uint8_t* const* commitments, const uint64_t* cell_indices, const uint8_t* const* cells,
                        const uint8_t* const* proofs, const GroupVerdicts* groups, bool* verified) const;
    // proofs of n blobs from ws.d_coeffs, asynchronous on `stream`: by the direct route when proof_route() picks it
    // (never with stage_events), else FK20 = fk20_msm of all n blobs, then fk20_ntt_compress
    Status fk20_from_coeffs_device(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream,
                                   std::vector<cudaEvent_t>* stage_events = nullptr) const;
    Status proofs_direct_device(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream) const;   // needs ws.capacity >= 128 n
    // commitments of n blobs from ws.d_coeffs into d_out48 (n x 48 B), asynchronous on `stream`; uses ws.d_scalars and ws.d_pts
    Status commit_device(Workspace& ws, int n, uint8_t* d_out48, cudaStream_t stream) const;
    // B 4096-point MSMs over the SRS tables from the scalars in ws.d_scalars ([4096][B] plain), compressed into d_out (B x 48 B)
    Status srs_msm_compress(Workspace& ws, int B, uint8_t* d_out, cudaStream_t stream) const;
    // K2 + K4 of blobs [o, o + c) of an n-blob batch (c < 0: to the end), then K5 + K6 of all n; stage events 2..5 as in fk20_device
    Status fk20_msm(Workspace& ws, int n, int o, int c, cudaStream_t stream, std::vector<cudaEvent_t>* stage_events) const;
    Status fk20_ntt_compress(Workspace& ws, int n, uint8_t* d_proofs, cudaStream_t stream, std::vector<cudaEvent_t>* stage_events) const;
    // Leader/follower coalescing of concurrent single-item callers into shared batches (see compute_cells_and_kzg_proofs_one).
    struct CoalesceReq {
        // compute: blob -> cells (+ proofs);   recover: count cells at `indices` -> cells + proofs
        const uint8_t* in = nullptr;        // blob (131072 B) / the given cells, contiguous (count * 2048 B)
        const uint64_t* indices = nullptr;  // recover only
        uint64_t count = 0;                 // recover only
        uint8_t* cells = nullptr;           // 128 * 2048 B out, contiguous ...
        uint8_t* proofs = nullptr;          // 128 * 48 B out
        uint8_t* const* cells_scattered = nullptr;   // ... or through 128 pointers each
        uint8_t* const* proofs_scattered = nullptr;
    };
    // pinned host block a coalesced batch is formed in: slot i holds member i's input, later its outputs
    struct CoalesceStaging {
        int capacity = 0;
        size_t in_stride = 0;
        uint8_t* in = nullptr;
        uint8_t* cells = nullptr;
        uint8_t* proofs = nullptr;
        std::vector<uint8_t> status;
        std::vector<uint64_t> counts, indices;   // recover: per slot, indices 128 wide
        Status alloc(int cap, size_t in_bytes_per_item, bool with_proofs, bool with_index);
        void release();
    };
    struct CoalesceBatch {
        CoalesceStaging* st = nullptr;
        int n = 0;          // members that joined
        int copied = 0;     // members whose input is in the block
        int left = 0;       // members that have not copied their results out yet
        bool closed = false, done = false;
        Status result = Status::Ok();
    };
    struct CoalesceQueue {
        std::mutex mu;
        std::condition_variable cv;         // members: "my batch is done"; starters: "a staging block is free"
        std::condition_variable cv_leader;  // leader: "somebody joined / finished copying in / a batch left the device"
        CoalesceBatch* forming = nullptr;
        int in_flight = 0;                  // batches handed to the device and not finished
        int callers = 0;                    // threads inside coalesce() on this queue (a lone caller does not linger)
        int n_staging = 0;
        std::vector<CoalesceStaging*> free_staging;
    };
    enum { CQ_CELLS = 0, CQ_CELLS_PROOFS = 1, CQ_RECOVER = 2 };
    mutable CoalesceQueue co_[3];
    Status coalesce(int which, CoalesceReq& me) const;
    // strided: item i's indices at indices + 128 i and its cells at cells + 128 i * 2048 (the coalescer's staging slots)
    Status recover_impl(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_cells, uint8_t* out_proofs,
                        uint8_t* item_status, bool strided) const;
    Status init(bool use_precomp, int device, const SetupBytes* custom);
    host::G2Keys* g2keys_ = nullptr;   // G2 side of a caller-supplied setup (nullptr: the embedded ceremony's constants)
    int device_ = 0;
    DevTables T_{};
    std::vector<void*> allocs_;
    uint64_t table_bytes_ = 0;
    size_t msm_scratch_bytes_ = 0;
    const Fr* coset_shift_fwd_ = nullptr;   // 7^i / 8192
    const Fr* coset_shift_inv_ = nullptr;   // 7^-i / 8192
    mutable bool profiling_ = false;
    mutable std::vector<std::vector<cudaEvent_t>> prof_events_;  // one vector of N_STAGES+1 events per batch
    mutable std::mutex pool_mu_;
    mutable std::vector<Workspace*> pool_;
};

int chunk_capacity();
// z = SHA-256("FSBLOBVERIFY_V1_" || u128_be(4096) || blob || commitment) mod r as 32 canonical big-endian bytes
// (crates/eip4844/src/verifier.rs:155-196) on the HOST: for a handful of blobs the x86 SHA extensions (0.1 ms per blob) beat the
// device kernel, where one thread walks the 2049 compressions of a blob (~4 ms whatever the count).
void host_blob_challenge(const uint8_t* blob, const uint8_t* commitment48, uint8_t z_be[32]);
constexpr int HOST_CHALLENGE_MAX = 16;   // blobs per call up to which the challenges are hashed on the host

// EKZG_TRACE=1: wall-clock marks of the host-side phases on stderr (the reference's optional `tracing` feature,
// crates/eip7594/Cargo.toml, plays this role there)
struct TraceClock {
    bool on;
    const char* what;
    double t0;
    static double now();
    explicit TraceClock(const char* w);
    void mark(const char* phase);
};

}  // namespace ekzg
