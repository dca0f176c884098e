// One DASContext over several GPUs of one box.
//
// The reference fans ONE call out over every core of the machine (crates/maybe_rayon/src/multi_threaded.rs:9-39, call
// sites crates/cryptography/kzg_multi_open/src/fk20/batch_toeplitz.rs:95-117 and crates/eip7594/src/prover.rs:117-148).
// The counterpart one level up: a DeviceSet owns one Context (tables, workspace pool, coalescing queues) per device
// named in EKZG_DEVICES ("all" or a comma list of ordinals; unset = the calling thread's current device only, so a
// process-per-GPU launcher such as torchrun keeps one device per rank).  A batch call is cut into contiguous shards,
// one per device, each driven by its own host thread through that device's three-stream pipeline; results are DMA'd
// straight into the caller's buffers (no gather step, no collective: blobs are independent -- SURVEY.md §8e).
// Single-item calls are dealt round-robin to the devices' coalescing queues.
#pragma once
#include <atomic>
#include <functional>
#include "kzg_runtime.h"

namespace ekzg {

class DeviceSet {
public:
    static Status create(bool use_precomp, std::unique_ptr<DeviceSet>* out, const SetupBytes* custom = nullptr);

    size_t size() const { return ctx_.size(); }
    const Context& primary() const { return *ctx_[0]; }
    const Context& at(size_t i) const { return *ctx_[i]; }
    // next device for a single-item call (round-robin; every device has its own coalescing queues)
    const Context& next() const { return *ctx_[ctx_.size() == 1 ? 0 : rr_.fetch_add(1, std::memory_order_relaxed) % ctx_.size()]; }
    // the member whose device owns this device pointer (nullptr if none does)
    const Context* owner_of(const void* device_ptr) const;

    // shard i of a batch of n items over `parts` devices: whole blob groups of the G1-NTT kernels (32 items, or 8 where a device's
    // share is at most 80 items: the cooperative latency-mode kernel), sizes differing by at most one group
    static void shard_bounds(uint64_t n, size_t parts, size_t i, uint64_t* lo, uint64_t* cnt);

    // Runs fn(context, first item, item count) once per non-empty shard, shard 0 on the calling thread and the others on
    // threads of their own; returns the first failure in shard order.
    Status fan_out(uint64_t n, const std::function<Status(const Context&, uint64_t, uint64_t)>& fn) const;
    // fan_out over items whose cells and indices are concatenated (counts[i] of item i): fn also gets the offset of the shard's
    // first cell
    Status fan_out_cells(uint64_t n, const uint64_t* counts, const std::function<Status(const Context&, uint64_t, uint64_t, uint64_t)>& fn) const;

    Status compute_cells_and_kzg_proofs_batch(uint64_t n, const uint8_t* blobs, uint8_t* cells, uint8_t* proofs, uint8_t* blob_status,
                                              bool want_proofs) const;
    Status blob_to_kzg_commitment_batch(uint64_t n, const uint8_t* blobs, uint8_t* out48, uint8_t* item_status) const;
    Status compute_blob_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments48, uint8_t* out48,
                                        uint8_t* item_status) const;
    Status recover_cells_and_kzg_proofs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells,
                                              uint8_t* out_cells, uint8_t* out_proofs, uint8_t* item_status) const;
    Status recover_blobs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_blobs,
                               uint8_t* item_status) const;
    Status verify_blob_cell_proofs_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                         uint8_t* item_status, uint8_t* cell_status, bool* all_ok) const;

    uint64_t table_bytes() const;

private:
    DeviceSet() = default;
    std::vector<std::unique_ptr<Context>> ctx_;
    mutable std::atomic<uint32_t> rr_{0};
};

}  // namespace ekzg
