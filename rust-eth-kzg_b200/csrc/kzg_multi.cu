// One DASContext over several GPUs (see kzg_multi.h).
#include "kzg_multi.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

namespace ekzg {

static Status parse_devices(std::vector<int>* out) {
    const char* e = getenv("EKZG_DEVICES");
    out->clear();
    if (!e || !*e) {
        out->push_back(-1);   // the calling thread's current device (or EKZG_DEVICE), as before
        return Status::Ok();
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return Status::Error("no CUDA device: this backend has no CPU fallback");
    }
    if (!strcmp(e, "all")) {
        for (int d = 0; d < ndev; d++) out->push_back(d);
        return Status::Ok();
    }
    for (const char* p = e; *p;) {
        char* end = nullptr;
        const long d = strtol(p, &end, 10);
        if (end == p || d < 0 || d >= ndev) return Status::Error(std::string("EKZG_DEVICES: bad device list '") + e + "' (" + std::to_string(ndev) + " devices visible)");
        // (an ordinal may appear twice: two member contexts then share that device, each with its own tables and queues --
        //  how the sharding path is exercised on a one-GPU box, tests/test_gpu_multi.py)
        out->push_back((int)d);
        p = end;
        if (*p == ',') p++;
        else if (*p) return Status::Error(std::string("EKZG_DEVICES: bad device list '") + e + "'");
    }
    if (out->empty()) return Status::Error("EKZG_DEVICES is empty");
    return Status::Ok();
}

Status DeviceSet::create(bool use_precomp, std::unique_ptr<DeviceSet>* out, const SetupBytes* custom) {
    std::vector<int> devs;
    Status s = parse_devices(&devs);
    if (!s.ok) return s;
    std::unique_ptr<DeviceSet> set(new DeviceSet());
    set->ctx_.resize(devs.size());
    // the tables of every device are built concurrently (2 s each for the widest layout), one host thread per device
    std::vector<Status> st(devs.size());
    std::vector<std::thread> th;
    for (size_t i = 1; i < devs.size(); i++)
        th.emplace_back([&, i] { st[i] = Context::create(use_precomp, &set->ctx_[i], devs[i], custom); });
    st[0] = Context::create(use_precomp, &set->ctx_[0], devs[0], custom);
    for (auto& t : th) t.join();
    for (size_t i = 0; i < devs.size(); i++)
        if (!st[i].ok) return Status::Error("device " + std::to_string(devs[i]) + ": " + st[i].msg);
    if (getenv("EKZG_TRACE")) {
        for (auto& c : set->ctx_)
            fprintf(stderr, "[ekzg trace] context on device %d: FK20 window %d bits, SRS window %d bits, %.1f GiB of tables\n", c->device(),
                    c->tables().fk20.w, c->tables().srs.w, c->table_bytes() / 1073741824.0);
    }
    *out = std::move(set);
    return Status::Ok();
}

const Context* DeviceSet::owner_of(const void* device_ptr) const {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, device_ptr) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return nullptr;
    for (auto& c : ctx_)
        if (c->device() == a.device) return c.get();
    return nullptr;
}

void DeviceSet::shard_bounds(uint64_t n, size_t parts, size_t i, uint64_t* lo, uint64_t* cnt) {
    // whole blob groups of the G1-NTT kernels: 32 blobs per warp, or 8 where a device's share is small enough for the cooperative
    // latency-mode kernel (four lanes per field element, up to 80 blobs) -- 64 blobs on eight devices are eight shards of 8, not two of 32
    const uint64_t gw = (n + parts - 1) / parts <= 80 ? 8 : 32;
    const uint64_t groups = (n + gw - 1) / gw;
    const uint64_t g0 = groups * i / parts, g1 = groups * (i + 1) / parts;
    const uint64_t a = std::min<uint64_t>(n, g0 * gw), b = std::min<uint64_t>(n, g1 * gw);
    *lo = a;
    *cnt = b - a;
}

Status DeviceSet::fan_out(uint64_t n, const std::function<Status(const Context&, uint64_t, uint64_t)>& fn) const {
    const size_t D = ctx_.size();
    if (D == 1 || n <= 8) return fn(*ctx_[0], 0, n);
    std::vector<Status> st(D);
    std::vector<std::thread> th;
    uint64_t lo0 = 0, cnt0 = 0;
    shard_bounds(n, D, 0, &lo0, &cnt0);
    for (size_t i = 1; i < D; i++) {
        uint64_t lo, cnt;
        shard_bounds(n, D, i, &lo, &cnt);
        if (!cnt) continue;
        th.emplace_back([&, i, lo, cnt] {
            try {
                st[i] = fn(*ctx_[i], lo, cnt);
            } catch (const std::exception& ex) {
                st[i] = Status::Error(std::string("shard failed: ") + ex.what());
            }
        });
    }
    if (cnt0) st[0] = fn(*ctx_[0], lo0, cnt0);
    for (auto& t : th) t.join();
    for (size_t i = 0; i < D; i++)
        if (!st[i].ok) return st[i];
    return Status::Ok();
}

Status DeviceSet::compute_cells_and_kzg_proofs_batch(uint64_t n, const uint8_t* blobs, uint8_t* cells, uint8_t* proofs, uint8_t* blob_status,
                                                     bool want_proofs) const {
    return fan_out(n, [&](const Context& c, uint64_t lo, uint64_t cnt) {
        return c.compute_cells_and_kzg_proofs_batch(cnt, blobs + lo * BYTES_PER_BLOB, cells ? cells + lo * CELLS_PER_BLOB : nullptr,
                                                    proofs ? proofs + lo * PROOFS_PER_BLOB : nullptr, blob_status ? blob_status + lo : nullptr, want_proofs);
    });
}

Status DeviceSet::blob_to_kzg_commitment_batch(uint64_t n, const uint8_t* blobs, uint8_t* out48, uint8_t* item_status) const {
    return fan_out(n, [&](const Context& c, uint64_t lo, uint64_t cnt) {
        return c.blob_to_kzg_commitment_batch(cnt, blobs + lo * BYTES_PER_BLOB, out48 + lo * 48, item_status ? item_status + lo : nullptr);
    });
}

Status DeviceSet::compute_blob_kzg_proof_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments48, uint8_t* out48,
                                               uint8_t* item_status) const {
    return fan_out(n, [&](const Context& c, uint64_t lo, uint64_t cnt) {
        return c.compute_blob_kzg_proof_batch(cnt, blobs + lo * BYTES_PER_BLOB, commitments48 + lo * 48, out48 + lo * 48,
                                              item_status ? item_status + lo : nullptr);
    });
}

Status DeviceSet::fan_out_cells(uint64_t n, const uint64_t* counts,
                                const std::function<Status(const Context&, uint64_t, uint64_t, uint64_t)>& fn) const {
    if (ctx_.size() == 1 || n <= 8) return fn(*ctx_[0], 0, n, 0);
    std::vector<uint64_t> offset(n + 1, 0);   // blob i's cells and indices start at offset[i] in the concatenated inputs
    for (uint64_t i = 0; i < n; i++) offset[i + 1] = offset[i] + counts[i];
    return fan_out(n, [&](const Context& c, uint64_t lo, uint64_t cnt) { return fn(c, lo, cnt, offset[lo]); });
}

Status DeviceSet::recover_cells_and_kzg_proofs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells,
                                                     uint8_t* out_cells, uint8_t* out_proofs, uint8_t* item_status) const {
    return fan_out_cells(n, counts, [&](const Context& c, uint64_t lo, uint64_t cnt, uint64_t cell0) {
        return c.recover_cells_and_kzg_proofs_batch(cnt, counts + lo, indices + cell0, cells + cell0 * BYTES_PER_CELL,
                                                    out_cells + lo * CELLS_PER_BLOB, out_proofs + lo * PROOFS_PER_BLOB,
                                                    item_status ? item_status + lo : nullptr);
    });
}

Status DeviceSet::recover_blobs_batch(uint64_t n, const uint64_t* counts, const uint64_t* indices, const uint8_t* cells, uint8_t* out_blobs,
                                      uint8_t* item_status) const {
    return fan_out_cells(n, counts, [&](const Context& c, uint64_t lo, uint64_t cnt, uint64_t cell0) {
        return c.recover_blobs_batch(cnt, counts + lo, indices + cell0, cells + cell0 * BYTES_PER_CELL, out_blobs + lo * BYTES_PER_BLOB,
                                     item_status ? item_status + lo : nullptr);
    });
}

Status DeviceSet::verify_blob_cell_proofs_batch(uint64_t n, const uint8_t* blobs, const uint8_t* commitments, const uint8_t* proofs,
                                                uint8_t* item_status, uint8_t* cell_status, bool* all_ok) const {
    *all_ok = false;
    EKZG_TRY(fan_out(n, [&](const Context& c, uint64_t lo, uint64_t cnt) {
        bool shard_ok = false;   // unused: each shard's verdict covers only its items; the batch verdict is formed from item_status below
        return c.verify_blob_cell_proofs_batch(cnt, blobs + lo * BYTES_PER_BLOB, commitments + lo * BYTES_PER_G1, proofs + lo * PROOFS_PER_BLOB,
                                               item_status + lo, cell_status ? cell_status + lo * N_CELLS : nullptr, &shard_ok);
    }));
    *all_ok = std::all_of(item_status, item_status + n, [](uint8_t s) { return s == VERDICT_OK; });
    return Status::Ok();
}

uint64_t DeviceSet::table_bytes() const {
    uint64_t t = 0;
    for (auto& c : ctx_) t += c->table_bytes();
    return t;
}

}  // namespace ekzg
