// Host orchestration of the verifiers (see kzg_kernels_verify.cu for the device side, host_pairing.cpp for the pairing).
//   reference: crates/eip7594/src/verifier.rs:49-164 (dedup + validation + dispatch),
//              kzg_multi_open/src/fk20/verifier.rs:129-328, crates/eip4844/src/verifier.rs:19-260.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <map>
#include <string>
#include "host_pairing.h"
#include "host_sha256.h"
#include <array>
#include <future>
#include <system_error>
#include <thread>
#include <unordered_map>
#include "kzg_runtime.h"
#include "sha256.cuh"

namespace ekzg {

namespace {

// stream-ordered scratch that frees itself
struct Scratch {
    cudaStream_t st;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t s) : st(s) {}
    ~Scratch() { for (void* p : ptrs) cudaFreeAsync(p, st); }
    template <class T>
    Status get(T** out, size_t count) {
        void* p = nullptr;
        EKZG_CUDA(cudaMallocAsync(&p, (count ? count : 1) * sizeof(T), st));
        ptrs.push_back(p);
        *out = reinterpret_cast<T*>(p);
        return Status::Ok();
    }
};

void be64(uint8_t* o, uint64_t v) { for (int i = 0; i < 8; i++) o[i] = (uint8_t)(v >> (56 - 8 * i)); }

bool run_pairing(const uint32_t* w /*2 x PAIRING_INPUT_WORDS*/, host::G2Sel q0, host::G2Sel q1, const host::G2Keys* keys) {
    host::PairingInputJac in[2];
    for (int i = 0; i < 2; i++) {
        const uint32_t* o = w + PAIRING_INPUT_WORDS * i;
        for (int l = 0; l < 6; l++) {
            in[i].x[l] = (uint64_t)o[2 * l] | ((uint64_t)o[2 * l + 1] << 32);
            in[i].y[l] = (uint64_t)o[12 + 2 * l] | ((uint64_t)o[12 + 2 * l + 1] << 32);
            in[i].z[l] = (uint64_t)o[24 + 2 * l] | ((uint64_t)o[24 + 2 * l + 1] << 32);
        }
        in[i].g1_is_identity = o[36] != 0;
    }
    in[0].g2 = q0;
    in[1].g2 = q1;
    return host::pairing_check_jac(in, 2, keys);
}

// fn(i) for every i < count, spread over up to hardware_concurrency() threads, this one included (pairing_check_jac is
// re-entrant: its shared tables are built once, under a once_flag, and only read afterwards)
template <class F>
void parallel_for(size_t count, F fn) {
    const size_t workers = std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), count);
    std::atomic<size_t> next{0};
    auto work = [&]() {
        for (size_t i; (i = next.fetch_add(1)) < count;) fn(i);
    };
    std::vector<std::thread> pool;
    for (size_t w = 1; w < workers; w++) {
        try {
            pool.emplace_back(work);
        } catch (const std::system_error&) {   // no more threads to be had: the ones running share the rest
            break;
        }
    }
    work();
    for (std::thread& t : pool) t.join();
}

}  // namespace

// ------------------------------------------------------------------------------------------------
Status Context::verify_cell_kzg_proof_batch(uint64_t n_commitments, const uint8_t* const* commitments, uint64_t n_indices,
                                            const uint64_t* cell_indices, uint64_t n_cells, const uint8_t* const* cells, uint64_t n_proofs,
                                            const uint8_t* const* proofs, bool* verified) const {
    *verified = false;
    // validation (verifier.rs:123-164)
    if (!(n_commitments == n_indices && n_commitments == n_cells && n_commitments == n_proofs))
        return Status::Error("Verifier(BatchVerificationInputsMustHaveSameLength)");
    for (uint64_t i = 0; i < n_indices; i++)
        if (cell_indices[i] >= (uint64_t)N_CELLS) return Status::Error("Verifier(CellIndexOutOfRange)");
    return verify_cells(n_cells, commitments, cell_indices, cells, proofs, nullptr, verified);
}

Status Context::verify_cell_kzg_proof_batch_groups(uint64_t n, const uint8_t* const* commitments, const uint64_t* cell_indices,
                                                   const uint8_t* const* cells, const uint8_t* const* proofs, uint64_t n_groups,
                                                   const uint32_t* group_of, uint8_t* group_status, bool* all_ok) const {
    *all_ok = false;
    if (n_groups > MAX_VERIFY_GROUPS) return Status::Error("too many groups: n_groups above 2^20");
    for (uint64_t k = 0; k < n; k++)
        if (group_of[k] >= n_groups) return Status::Error("group id out of range: group_of[" + std::to_string(k) + "] >= n_groups");
    std::fill(group_status, group_status + n_groups, (uint8_t)VERDICT_OK);
    const GroupVerdicts groups{group_of, n_groups, group_status};
    return verify_cells(n, commitments, cell_indices, cells, proofs, &groups, all_ok);
}

Status Context::verify_cells(uint64_t n, const uint8_t* const* commitments, const uint64_t* cell_indices, const uint8_t* const* cells,
                             const uint8_t* const* proofs, const GroupVerdicts* groups, bool* verified) const {
    *verified = false;
    TraceClock tr(groups ? "verify_cell_kzg_proof_batch_groups" : "verify_cell_kzg_proof_batch");
    // deduplicate_with_indices (verifier.rs:49-65): first occurrence order is part of the transcript
    std::vector<const uint8_t*> uniq;
    std::vector<uint32_t> rows(n);
    {
        std::unordered_map<std::string, uint32_t> seen;
        seen.reserve(256);
        const uint8_t* last_ptr = nullptr;
        uint32_t last_row = 0;
        for (uint64_t i = 0; i < n; i++) {
            // callers repeat one commitment per cell of a blob (often the very same pointer): skip the lookup then
            if (last_ptr && (commitments[i] == last_ptr || memcmp(commitments[i], last_ptr, 48) == 0)) { rows[i] = last_row; continue; }
            std::string key(reinterpret_cast<const char*>(commitments[i]), 48);
            last_ptr = commitments[i];
            auto it = seen.find(key);
            if (it == seen.end()) {
                it = seen.emplace(key, (uint32_t)uniq.size()).first;
                uniq.push_back(commitments[i]);
            }
            rows[i] = last_row = it->second;
        }
    }
    const int N = (int)n, M = (int)uniq.size();
    if (N == 0) { *verified = true; return Status::Ok(); }
    EKZG_TRY(bind_device());

    // pack inputs
    // the ABI hands us one pointer per item (pointer_utils.rs:25-44); when the items happen to be laid out back to
    // back (the usual case for a caller holding a flat buffer) the gather copy of the 2 KiB cells is skipped
    bool cells_contig = true;
    for (int k = 1; k < N && cells_contig; k++) cells_contig = cells[k] == cells[0] + (size_t)k * BYTES_PER_CELL;
    std::vector<uint8_t> hc((size_t)M * 48), hp((size_t)N * 48), hcells_store(cells_contig ? 0 : (size_t)N * BYTES_PER_CELL);
    std::vector<uint32_t> hcol(N);
    for (int i = 0; i < M; i++) memcpy(&hc[(size_t)i * 48], uniq[i], 48);
    for (int k = 0; k < N; k++) {
        memcpy(&hp[(size_t)k * 48], proofs[k], 48);
        if (!cells_contig) memcpy(&hcells_store[(size_t)k * BYTES_PER_CELL], cells[k], BYTES_PER_CELL);
        // (an index >= 128 reaches the device only from the grouped call, which flags it there and masks the opening)
        hcol[k] = (uint32_t)std::min<uint64_t>(cell_indices[k], N_CELLS);
    }
    const uint8_t* hcells = cells_contig ? cells[0] : hcells_store.data();
    tr.mark("dedup + pack");
    // Fiat-Shamir transcript (fk20/verifier.rs:269-328): ONE sequential SHA-256 chain over every input byte (34.6 MB for
    // 128 x 128 cells, 21 ms with the x86 SHA extensions).  It only needs host data, so it starts now on a helper thread
    // while this thread stages the copies (the 33 MB of cells are pageable caller memory: a synchronous 3 ms) and the device
    // validates the points.  The grouped call hashes exactly these bytes, malformed items included.
    auto hash_transcript = [&]() {
        std::array<uint8_t, 32> out;
        host::Sha256Stream h;
        uint8_t head[16 + 32];
        memcpy(head, "RCKZGCBATCH__V1_", 16);
        be64(head + 16, N_BLOB); be64(head + 24, CELL_ELEMS); be64(head + 32, (uint64_t)M); be64(head + 40, (uint64_t)N);
        h.update(head, sizeof head);
        h.update(hc.data(), hc.size());
        for (int k = 0; k < N; k++) {
            uint8_t idx[16];
            be64(idx, rows[k]); be64(idx + 8, cell_indices[k]);
            h.update(idx, 16);
            h.update(&hcells[(size_t)k * BYTES_PER_CELL], BYTES_PER_CELL);
            h.update(&hp[(size_t)k * 48], 48);
        }
        h.final(out.data());
        return out;
    };
    std::future<std::array<uint8_t, 32>> hash_task;
    try {
        hash_task = std::async(std::launch::async, hash_transcript);
    } catch (const std::exception&) {   // no thread to be had: hash on this one, when the value is needed
        hash_task = std::async(std::launch::deferred, hash_transcript);
    }
    Workspace* wsp = acquire(1, true);
    if (!wsp) { hash_task.wait(); return Status::Error("allocation failed"); }
    cudaStream_t st = wsp->stream;
    Status result = Status::Ok();
    uint32_t pin[2 * PAIRING_INPUT_WORDS];
    std::vector<uint32_t> stc(M), stp(N), flag(groups ? N : 0);
    uint32_t cell_status = 0;
    {
        Scratch S(st);
        auto run = [&]() -> Status {
            uint8_t *d_c, *d_p, *d_cells, *d_hash;
            uint32_t *d_col, *d_row, *d_stc, *d_stp, *d_cellst, *d_s1, *d_s2, *d_w, *d_i, *d_out, *d_cellbad = nullptr, *d_flag = nullptr;
            G1Affine *a_c, *a_p;
            Fr *d_rpow, *d_interp;
            G1Jac *d_mul, *d_mul_b, *d_mul_c, *d_mul_d, *d_part, *d_part_b, *d_part_d, *d_sums, *d_colsum;
            EKZG_TRY(S.get(&d_colsum, 2 * N_CELLS));
            EKZG_TRY(S.get(&d_c, (size_t)M * 48)); EKZG_TRY(S.get(&d_p, (size_t)N * 48)); EKZG_TRY(S.get(&d_cells, (size_t)N * BYTES_PER_CELL));
            EKZG_TRY(S.get(&d_hash, 32)); EKZG_TRY(S.get(&d_col, N)); EKZG_TRY(S.get(&d_row, N)); EKZG_TRY(S.get(&d_stc, M)); EKZG_TRY(S.get(&d_stp, N));
            EKZG_TRY(S.get(&d_cellst, 1)); EKZG_TRY(S.get(&d_s1, (size_t)N * 8)); EKZG_TRY(S.get(&d_s2, (size_t)N * 8)); EKZG_TRY(S.get(&d_w, (size_t)M * 8));
            EKZG_TRY(S.get(&d_i, 64 * 8)); EKZG_TRY(S.get(&d_out, 2 * PAIRING_INPUT_WORDS)); EKZG_TRY(S.get(&a_c, M)); EKZG_TRY(S.get(&a_p, N)); EKZG_TRY(S.get(&d_rpow, N));
            EKZG_TRY(S.get(&d_interp, (size_t)N * 64)); EKZG_TRY(S.get(&d_mul, std::max(N, 128))); EKZG_TRY(S.get(&d_mul_b, std::max(M, 128))); EKZG_TRY(S.get(&d_mul_c, 128)); EKZG_TRY(S.get(&d_part, 148)); EKZG_TRY(S.get(&d_part_b, 148)); EKZG_TRY(S.get(&d_mul_d, std::max(N, 128))); EKZG_TRY(S.get(&d_part_d, 148)); EKZG_TRY(S.get(&d_sums, 4));
            if (groups) { EKZG_TRY(S.get(&d_cellbad, N)); EKZG_TRY(S.get(&d_flag, N)); }
            EKZG_CUDA(cudaMemcpyAsync(d_c, hc.data(), hc.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_p, hp.data(), hp.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_cells, hcells, (size_t)N * BYTES_PER_CELL, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_col, hcol.data(), sizeof(uint32_t) * N, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_row, rows.data(), sizeof(uint32_t) * N, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemsetAsync(d_cellst, 0, 4, st));
            // point validation runs while the host hashes the transcript: decompression here; the subgroup checks (twice the
            // work, and nothing downstream needs their result before the final read-back) on a side stream, where for a small
            // call they run beside the scalar multiplications instead of in front of them
            cudaStream_t sb = wsp->copy_stream, sc = wsp->in_stream, sd = wsp->aux_stream;
            EKZG_CUDA(launch_g1_validate(d_p, a_p, d_stp, N, false, st));
            EKZG_CUDA(launch_g1_validate(d_c, a_c, d_stc, M, false, st));
            EKZG_CUDA(cudaEventRecord(wsp->sub_ready[1], st));
            EKZG_CUDA(cudaStreamWaitEvent(sc, wsp->sub_ready[1], 0));
            EKZG_CUDA(launch_g1_subgroup(a_p, d_stp, N, a_c, d_stc, M, sc));
            if (groups) {   // the grouped call masks malformed openings, which needs every status before the first sum
                EKZG_CUDA(launch_cell_canonical(d_cells, d_cellbad, N, sc));
                EKZG_CUDA(cudaEventRecord(wsp->sub_out[3], sc));
            }
            tr.mark("alloc + enqueue copies/validation");
            const std::array<uint8_t, 32> hash_arr = hash_task.get();
            const uint8_t* hash = hash_arr.data();
            tr.mark("waiting for the transcript sha256");
            EKZG_CUDA(cudaMemcpyAsync(d_hash, hash, 32, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(launch_powers_from_hash(d_hash, d_rpow, N, st));
            if (groups) {
                EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[3], 0));
                EKZG_CUDA(launch_mask_openings(d_rpow, d_stp, d_stc, d_row, d_col, d_cellbad, a_p, a_c, d_flag, N, M, st));
            }
            EKZG_CUDA(launch_cell_verify_scalars(d_rpow, d_col, d_s1, d_s2, T_, N, st));
            // Independent, latency-bound chains follow (a handful of CTAs each: one 255-bit scalar multiplication takes ~3 ms
            // whatever the count): they run side by side on the workspace's four streams.
            EKZG_CUDA(cudaEventRecord(wsp->sub_ready[0], st));
            EKZG_CUDA(cudaStreamWaitEvent(sb, wsp->sub_ready[0], 0));
            EKZG_CUDA(cudaStreamWaitEvent(sc, wsp->sub_ready[0], 0));
            // (A)  P = sum rho_k pi_k ; W = sum rho_k h_k^64 pi_k  (verifier.rs:188-213)
            static const bool force_columns = getenv("EKZG_VERIFY_COLUMN_SUMS") != nullptr;
            // EKZG_VERIFY_MSM=bucket | ladder: the bucket-method MSM (K7, kzg_kernels_msm.cu) for both sums, or never; default: by size
            const char* msm_env = getenv("EKZG_VERIFY_MSM");
            const bool bucket = !force_columns && (msm_env ? msm_env[0] == 'b' : (N >= MSM_BUCKET_MIN && N <= 32768));
            const bool ladders = !bucket && !force_columns && N <= 32768;
            if (bucket) {
                uint8_t* d_msm;
                EKZG_TRY(S.get(&d_msm, msm_bucket_scratch_bytes(N, 2)));
                EKZG_CUDA(launch_msm_bucket(a_p, d_s1, d_s2, N, &d_sums[0], &d_sums[1], d_msm, st));
            } else if (ladders) {
                // two passes of N scalar multiplications at the same time (the machine holds both; 16384 points are 512 warps)
                EKZG_CUDA(cudaStreamWaitEvent(sd, wsp->sub_ready[0], 0));
                EKZG_CUDA(launch_scalar_mul(a_p, d_s1, d_mul, N, st));
                EKZG_CUDA(launch_sum_points(d_mul, N, d_part, &d_sums[0], st));
                EKZG_CUDA(launch_scalar_mul(a_p, d_s2, d_mul_d, N, sd));
                EKZG_CUDA(launch_sum_points(d_mul_d, N, d_part_d, &d_sums[1], sd));
                EKZG_CUDA(cudaEventRecord(wsp->sub_out[2], sd));
                EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[2], 0));
            } else {
                // large batches are throughput-bound: ONE pass of N scalar multiplications, then per-column sums and 128
                // multiplications by fixed roots of unity (kzg_kernels_verify.cu: k_column_sums)
                EKZG_CUDA(launch_scalar_mul(a_p, d_s1, d_mul, N, st));
                EKZG_CUDA(launch_column_sums(d_mul, d_col, d_colsum, d_colsum + N_CELLS, N, st));
                EKZG_CUDA(launch_sum_points(d_colsum, N_CELLS, d_part, &d_sums[0], st));
                EKZG_CUDA(launch_sum_points(d_colsum + N_CELLS, N_CELLS, d_part, &d_sums[1], st));
            }
            // (B, on sb)  Cs = sum w_i C_i
            EKZG_CUDA(launch_commitment_weights(d_rpow, d_row, d_w, N, M, sb));
            EKZG_CUDA(launch_scalar_mul(a_c, d_w, d_mul_b, M, sb));
            EKZG_CUDA(launch_sum_points(d_mul_b, M, d_part_b, &d_sums[2], sb));
            EKZG_CUDA(cudaEventRecord(wsp->sub_out[0], sb));
            // (C, on sc)  Ic = commit(sum rho_k I_k): 64 coefficients on the first 64 monomial SRS points = group 0 of the
            // fixed-base SRS tables (natural position 0 of a 128-slot row)
            EKZG_CUDA(launch_cell_interp(d_cells, d_col, d_rpow, d_interp, d_cellst, T_, N, sc));
            EKZG_CUDA(launch_interp_column_sum(d_interp, d_i, N, sc));
            EKZG_CUDA(launch_fixed_msm(d_i, d_mul_c, T_.srs, 1, 1, sc));
            EKZG_CUDA(cudaMemcpyAsync(&d_sums[3], d_mul_c, sizeof(G1Jac), cudaMemcpyDeviceToDevice, sc));
            EKZG_CUDA(cudaEventRecord(wsp->sub_out[1], sc));
            EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[0], 0));
            EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[1], 0));
            // pairing inputs: (P, [tau^64]_2), (Cs - Ic + W, -[1]_2)
            EKZG_CUDA(launch_pairing_inputs(&d_sums[0], &d_sums[2], &d_sums[3], &d_sums[1], d_out, st));
            EKZG_CUDA(cudaMemcpyAsync(pin, d_out, sizeof pin, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(stc.data(), d_stc, sizeof(uint32_t) * M, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(stp.data(), d_stp, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(&cell_status, d_cellst, 4, cudaMemcpyDeviceToHost, st));
            if (groups) EKZG_CUDA(cudaMemcpyAsync(flag.data(), d_flag, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaStreamSynchronize(st));
            tr.mark("device work after the hash");
            if (!groups) return Status::Ok();

            // ---- verdicts per group ----
            uint8_t* gs = groups->status;
            for (int k = 0; k < N; k++)
                if (flag[k]) gs[groups->group_of[k]] = VERDICT_MALFORMED;
            // Phase A: the masked aggregate, i.e. the equation of the plain call over the well-formed openings.  It holds in
            // the honest case, and then so does every group without a malformed opening: nothing more runs.
            if (run_pairing(pin, host::G2Sel::Tau64, host::G2Sel::NegGen, g2keys_)) {
                tr.mark("pairing");
                return Status::Ok();
            }
            // Phase B: the same equation restricted to each group g that holds no malformed opening, with the same rho_k:
            //   e(sum_{k in g} rho_k pi_k, [tau^64]_2) * e(sum_{k in g} rho_k (C_row(k) + h_k^64 pi_k) - [sum_{k in g} rho_k I_k(tau)]_1, -[1]_2) == 1.
            // Soundness: r is the transcript hash of ALL inputs, so it is fixed before any group is formed, and rho_k = r^k
            // for the group's openings.  If one opening of g is false, the group's check is a nonzero polynomial identity in
            // r of degree < n that holds at the random r with probability <= n / |Fr|: the bound of the batch check itself.
            // Only the groups to check are laid out: CSR order of their openings (a counting sort by group).
            std::vector<uint32_t> count(groups->n_groups, 0), live, off(1, 0), order, small, large;
            for (int k = 0; k < N; k++)
                if (gs[groups->group_of[k]] != VERDICT_MALFORMED) count[groups->group_of[k]]++;
            for (uint64_t g = 0; g < groups->n_groups; g++)
                if (count[g]) {
                    (count[g] > 256 ? large : small).push_back((uint32_t)live.size());   // a CTA for a large group, a warp for a small one
                    live.push_back((uint32_t)g);
                    off.push_back(off.back() + count[g]);
                    count[g] = off[off.size() - 2];   // now the group's write cursor
                }
            const int G = (int)live.size();
            if (G == 0) return Status::Ok();
            order.resize(off.back());
            for (int k = 0; k < N; k++)
                if (gs[groups->group_of[k]] != VERDICT_MALFORMED) order[count[groups->group_of[k]]++] = (uint32_t)k;
            small.insert(small.end(), large.begin(), large.end());
            uint32_t *d_order, *d_off, *d_teams, *d_gi, *d_gpin;
            G1Affine* a_cg;
            G1Jac *d_mul_e, *d_gsum, *d_gI;
            EKZG_TRY(S.get(&d_order, order.size())); EKZG_TRY(S.get(&d_off, off.size())); EKZG_TRY(S.get(&d_teams, small.size()));
            EKZG_TRY(S.get(&d_gi, (size_t)64 * G * 8)); EKZG_TRY(S.get(&d_gpin, (size_t)2 * PAIRING_INPUT_WORDS * G));
            EKZG_TRY(S.get(&a_cg, N)); EKZG_TRY(S.get(&d_mul_e, N)); EKZG_TRY(S.get(&d_gsum, (size_t)3 * G)); EKZG_TRY(S.get(&d_gI, G));
            EKZG_CUDA(cudaMemcpyAsync(d_order, order.data(), sizeof(uint32_t) * order.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_off, off.data(), sizeof(uint32_t) * off.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_teams, small.data(), sizeof(uint32_t) * small.size(), cudaMemcpyHostToDevice, st));
            // per-opening products rho_k pi_k (d_mul), rho_k h_k^64 pi_k (d_mul_d), rho_k C_row(k) (d_mul_e): what the route above
            // did not leave behind, as three ladders side by side
            EKZG_CUDA(cudaEventRecord(wsp->sub_ready[2], st));
            EKZG_CUDA(cudaStreamWaitEvent(sb, wsp->sub_ready[2], 0));
            EKZG_CUDA(cudaStreamWaitEvent(sd, wsp->sub_ready[2], 0));
            if (bucket) EKZG_CUDA(launch_scalar_mul(a_p, d_s1, d_mul, N, st));
            if (!ladders) EKZG_CUDA(launch_scalar_mul(a_p, d_s2, d_mul_d, N, sd));
            EKZG_CUDA(cudaEventRecord(wsp->sub_out[4], sd));
            EKZG_CUDA(launch_gather_points(a_c, d_row, a_cg, N, sb));
            EKZG_CUDA(launch_scalar_mul(a_cg, d_s1, d_mul_e, N, sb));
            EKZG_CUDA(cudaEventRecord(wsp->sub_out[5], sb));
            EKZG_CUDA(launch_group_interp_sums(d_interp, d_order, d_off, d_gi, G, st));
            EKZG_CUDA(launch_fixed_msm(d_gi, d_gI, T_.srs, 1, G, st));
            EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[4], 0));
            EKZG_CUDA(cudaStreamWaitEvent(st, wsp->sub_out[5], 0));
            const int n_small = (int)(small.size() - large.size());
            EKZG_CUDA(launch_group_point_sums(d_mul, d_mul_d, d_mul_e, d_order, d_off, d_teams, n_small, d_teams + n_small, (int)large.size(),
                                              d_gsum, G, st));
            // (P_g, Cs_g - I_g + W_g), as the aggregate's k_pairing_inputs
            EKZG_CUDA(launch_pairing_inputs_n(d_gsum, d_gsum + 2 * G, d_gI, d_gsum + G, true, d_gpin, G, st));
            std::vector<uint32_t> gpin((size_t)2 * PAIRING_INPUT_WORDS * G);
            EKZG_CUDA(cudaMemcpyAsync(gpin.data(), d_gpin, sizeof(uint32_t) * gpin.size(), cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaStreamSynchronize(st));
            tr.mark("per-group sums");
            parallel_for(G, [&](size_t j) {
                if (!run_pairing(&gpin[2 * PAIRING_INPUT_WORDS * j], host::G2Sel::Tau64, host::G2Sel::NegGen, g2keys_)) gs[live[j]] = VERDICT_FAILS;
            });
            tr.mark("per-group pairings");
            return Status::Ok();
        };
        result = run();
        if (!result.ok) wsp->synchronize();   // S frees in the order of `st` alone: the side streams' work must be over first
    }
    give_back(wsp, result);
    if (!result.ok) return result;
    if (groups) {
        *verified = std::all_of(groups->status, groups->status + groups->n_groups, [](uint8_t v) { return v == VERDICT_OK; });
        return Status::Ok();
    }
    // deserialisation errors in the reference's order: commitments, proofs, cells (verifier.rs:96-98)
    for (uint32_t v : stc) if (v) return Status::Error("Serialization(G1PointInvalid): commitment");
    for (uint32_t v : stp) if (v) return Status::Error("Serialization(G1PointInvalid): proof");
    if (cell_status) return Status::Error("Serialization(ScalarNotCanonical): cell");
    *verified = run_pairing(pin, host::G2Sel::Tau64, host::G2Sel::NegGen, g2keys_);
    tr.mark("pairing");
    return Status::Ok();
}

// ------------------------------------------------------------------------------------------------
// EIP-4844 verifiers.  mode 0: (commitment, z, y, proof) given; mode 1: blobs given, z and y derived on the device.
Status Context::verify_kzg_proofs(int mode, uint64_t n, const uint8_t* const* blobs, const uint8_t* const* commitments, const uint8_t* z32,
                                  const uint8_t* y32, const uint8_t* const* proofs, bool* verified, uint8_t* item_status) const {
    *verified = false;
    if (n == 0) { *verified = true; return Status::Ok(); }
    const bool items = mode == 1 && item_status;
    if (n > (1u << 24)) return Status::Error("batch too large");   // (the per-item side buffers are sized by N; the blobs go in chunks)
    EKZG_TRY(bind_device());
    const int N = (int)n;
    std::vector<uint8_t> hc((size_t)N * 48), hp((size_t)N * 48);
    for (int i = 0; i < N; i++) { memcpy(&hc[(size_t)i * 48], commitments[i], 48); memcpy(&hp[(size_t)i * 48], proofs[i], 48); }
    // mode 1: the blobs pass through the workspace in chunks (only their challenge z and evaluation y are kept), so that a
    // large batch neither allocates nor retains a workspace of its own size (the reference accepts any length)
    const int chunk = mode == 1 ? std::min(N, chunk_capacity()) : 1;
    Workspace* wsp = acquire(chunk, true);
    if (!wsp) return Status::Error("allocation failed");
    Workspace& ws = *wsp;
    cudaStream_t st = ws.stream;
    Status result = Status::Ok();
    uint32_t pin[2 * PAIRING_INPUT_WORDS];
    std::vector<uint32_t> stc(N), stp(N), stb(N, 0), stz(N, 0), sty(N, 0), flag(items ? N : 0);
    {
        Scratch S(st);
        auto run = [&]() -> Status {
            uint8_t *d_c, *d_p, *d_zb, *d_yb, *d_hash;
            uint32_t *d_stc, *d_stp, *d_stz, *d_sty, *d_out, *d_stb = nullptr, *d_flag = nullptr;
            G1Affine *a_c, *a_p;
            Fr *d_z, *d_y, *d_rpow;
            G1Jac *d_prod, *d_part, *d_part2, *d_sums;
            G1Affine* d_pairs;
            uint32_t* d_psc;
            EKZG_TRY(S.get(&d_c, (size_t)N * 48)); EKZG_TRY(S.get(&d_p, (size_t)N * 48)); EKZG_TRY(S.get(&d_zb, (size_t)N * 32)); EKZG_TRY(S.get(&d_yb, (size_t)N * 32));
            EKZG_TRY(S.get(&d_hash, 32)); EKZG_TRY(S.get(&d_stc, N)); EKZG_TRY(S.get(&d_stp, N)); EKZG_TRY(S.get(&d_stz, N)); EKZG_TRY(S.get(&d_sty, N));
            EKZG_TRY(S.get(&d_out, 2 * PAIRING_INPUT_WORDS)); EKZG_TRY(S.get(&a_c, N)); EKZG_TRY(S.get(&a_p, N)); EKZG_TRY(S.get(&d_z, N)); EKZG_TRY(S.get(&d_y, N));
            EKZG_TRY(S.get(&d_rpow, N)); EKZG_TRY(S.get(&d_prod, (size_t)4 * N)); EKZG_TRY(S.get(&d_pairs, (size_t)4 * N)); EKZG_TRY(S.get(&d_psc, (size_t)32 * N));
            EKZG_TRY(S.get(&d_part, 148)); EKZG_TRY(S.get(&d_part2, 148)); EKZG_TRY(S.get(&d_sums, 2));
            if (items) { EKZG_TRY(S.get(&d_stb, N)); EKZG_TRY(S.get(&d_flag, N)); }
            EKZG_CUDA(cudaMemcpyAsync(d_c, hc.data(), hc.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemcpyAsync(d_p, hp.data(), hp.size(), cudaMemcpyHostToDevice, st));
            EKZG_CUDA(cudaMemsetAsync(d_stz, 0, sizeof(uint32_t) * N, st));
            EKZG_CUDA(cudaMemsetAsync(d_sty, 0, sizeof(uint32_t) * N, st));
            // decompression here, the subgroup checks beside the rest on a side stream (see verify_cell_kzg_proof_batch)
            EKZG_CUDA(launch_g1_validate(d_c, a_c, d_stc, N, false, st));
            EKZG_CUDA(launch_g1_validate(d_p, a_p, d_stp, N, false, st));
            EKZG_CUDA(cudaEventRecord(ws.sub_ready[1], st));
            EKZG_CUDA(cudaStreamWaitEvent(ws.copy_stream, ws.sub_ready[1], 0));
            EKZG_CUDA(launch_g1_subgroup(a_c, d_stc, N, a_p, d_stp, N, ws.copy_stream));
            EKZG_CUDA(cudaEventRecord(ws.sub_out[0], ws.copy_stream));
            std::vector<uint8_t> zb((size_t)N * 32), yb((size_t)N * 32);
            if (mode == 0) {
                EKZG_CUDA(cudaMemcpyAsync(d_zb, z32, (size_t)N * 32, cudaMemcpyHostToDevice, st));
                EKZG_CUDA(cudaMemcpyAsync(d_yb, y32, (size_t)N * 32, cudaMemcpyHostToDevice, st));
                EKZG_CUDA(launch_scalars_from_be(d_zb, d_z, d_stz, N, st));
                EKZG_CUDA(launch_scalars_from_be(d_yb, d_y, d_sty, N, st));
            } else {
                for (int o = 0; o < N; o += chunk) {
                    const int c = std::min(chunk, N - o);
                    if (o) EKZG_CUDA(cudaStreamSynchronize(st));   // the staging buffer is reused
                    for (int i = 0; i < c; i++) memcpy(ws.h_blobs + (size_t)i * BYTES_PER_BLOB, blobs[o + i], BYTES_PER_BLOB);
                    EKZG_CUDA(cudaMemcpyAsync(ws.d_blobs, ws.h_blobs, (size_t)c * BYTES_PER_BLOB, cudaMemcpyHostToDevice, st));
                    EKZG_CUDA(cudaMemsetAsync(ws.d_status, 0, sizeof(uint32_t) * c, st));
                    EKZG_CUDA(launch_blob_to_coeffs_cells(ws.d_blobs, ws.d_coeffs, nullptr, ws.d_status, T_, c, false, st));
                    if (items) EKZG_CUDA(cudaMemcpyAsync(d_stb + o, ws.d_status, sizeof(uint32_t) * c, cudaMemcpyDeviceToDevice, st));
                    if (N <= HOST_CHALLENGE_MAX) {   // a handful of blobs: challenges on the host (kzg_runtime.h), as canonical bytes
                        std::vector<uint8_t> zh((size_t)c * 32);
                        for (int i = 0; i < c; i++) host_blob_challenge(blobs[o + i], &hc[(size_t)(o + i) * 48], &zh[(size_t)i * 32]);
                        EKZG_CUDA(cudaMemcpyAsync(d_zb + (size_t)o * 32, zh.data(), zh.size(), cudaMemcpyHostToDevice, st));
                        EKZG_CUDA(cudaStreamSynchronize(st));
                        EKZG_CUDA(launch_scalars_from_be(d_zb + (size_t)o * 32, d_z + o, nullptr, c, st));
                    } else {
                        EKZG_CUDA(launch_blob_challenge(ws.d_blobs, d_c + (size_t)o * 48, d_z + o, c, st));
                    }
                    EKZG_CUDA(launch_poly_eval(ws.d_coeffs, d_z + o, d_y + o, d_yb + (size_t)o * 32, c, st));
                    EKZG_CUDA(cudaMemcpyAsync(stb.data() + o, ws.d_status, sizeof(uint32_t) * c, cudaMemcpyDeviceToHost, st));
                }
            }
            uint8_t hash[32] = {0};
            if (N > 1) {
                // r = H("RCKZGBATCH___V1_" || u64(4096) || u64(n) || (C, z, y, pi)*)  (eip4844/src/verifier.rs:202-260)
                if (mode == 1) {
                    EKZG_CUDA(launch_fr_to_be(d_z, d_zb, N, st));
                    EKZG_CUDA(cudaMemcpyAsync(zb.data(), d_zb, zb.size(), cudaMemcpyDeviceToHost, st));
                    EKZG_CUDA(cudaMemcpyAsync(yb.data(), d_yb, yb.size(), cudaMemcpyDeviceToHost, st));
                    EKZG_CUDA(cudaStreamSynchronize(st));
                } else {
                    memcpy(zb.data(), z32, zb.size());
                    memcpy(yb.data(), y32, yb.size());
                }
                host::Sha256Stream h;
                uint8_t head[32];
                memcpy(head, "RCKZGBATCH___V1_", 16);
                be64(head + 16, N_BLOB); be64(head + 24, (uint64_t)N);
                h.update(head, 32);
                for (int i = 0; i < N; i++) {
                    h.update(&hc[(size_t)i * 48], 48);
                    h.update(&zb[(size_t)i * 32], 32);
                    h.update(&yb[(size_t)i * 32], 32);
                    h.update(&hp[(size_t)i * 48], 48);
                }
                h.final(hash);
            }
            // N == 1: the only power used is r^0 = 1, whatever the digest
            EKZG_CUDA(cudaMemcpyAsync(d_hash, hash, 32, cudaMemcpyHostToDevice, st));
            EKZG_CUDA(launch_powers_from_hash(d_hash, d_rpow, N, st));
            if (items) {   // malformed items add nothing to the sums below; the others keep their powers
                EKZG_CUDA(cudaStreamWaitEvent(st, ws.sub_out[0], 0));
                EKZG_CUDA(launch_mask_items(d_rpow, d_stb, d_stc, d_stp, a_c, a_p, d_flag, N, st));
            }
            // the 4 N independent products r^i C_i, (-r^i y_i) G, (r^i z_i) pi_i | r^i pi_i in one pass, then the two sums
            EKZG_CUDA(launch_kzg_verify_pairs(a_c, a_p, d_z, d_y, d_rpow, d_pairs, d_psc, N, st));
            EKZG_CUDA(launch_scalar_mul(d_pairs, d_psc, d_prod, 4 * N, st));
            EKZG_CUDA(launch_sum_points(d_prod + (size_t)3 * N, N, d_part, &d_sums[0], st));
            EKZG_CUDA(launch_sum_points(d_prod, 3 * N, d_part2, &d_sums[1], st));
            EKZG_CUDA(launch_pairing_inputs(&d_sums[0], &d_sums[1], nullptr, nullptr, d_out, st));
            EKZG_CUDA(cudaStreamWaitEvent(st, ws.sub_out[0], 0));   // the subgroup verdicts
            EKZG_CUDA(cudaMemcpyAsync(pin, d_out, sizeof pin, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(stc.data(), d_stc, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(stp.data(), d_stp, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(stz.data(), d_stz, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaMemcpyAsync(sty.data(), d_sty, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            if (items) EKZG_CUDA(cudaMemcpyAsync(flag.data(), d_flag, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaStreamSynchronize(st));
            if (!items) return Status::Ok();
            // verdicts per item: phase A, the masked aggregate, holds in the honest case; else phase B checks every
            // well-formed item on its own, e(r^i pi_i, [tau]_2) * e(r^i (C_i - y_i G + z_i pi_i), -[1]_2) == 1, with the
            // products the aggregate was formed from (r^i != 0 scales both sides alike)
            for (int i = 0; i < N; i++) item_status[i] = flag[i] ? VERDICT_MALFORMED : VERDICT_OK;
            if (run_pairing(pin, host::G2Sel::Tau, host::G2Sel::NegGen, g2keys_)) return Status::Ok();
            uint32_t* d_ipin;
            EKZG_TRY(S.get(&d_ipin, (size_t)2 * PAIRING_INPUT_WORDS * N));
            EKZG_CUDA(launch_pairing_inputs_n(d_prod + (size_t)3 * N, d_prod, d_prod + N, d_prod + (size_t)2 * N, false, d_ipin, N, st));
            std::vector<uint32_t> ipin((size_t)2 * PAIRING_INPUT_WORDS * N);
            EKZG_CUDA(cudaMemcpyAsync(ipin.data(), d_ipin, sizeof(uint32_t) * ipin.size(), cudaMemcpyDeviceToHost, st));
            EKZG_CUDA(cudaStreamSynchronize(st));
            parallel_for(N, [&](size_t i) {
                if (!flag[i] && !run_pairing(&ipin[2 * PAIRING_INPUT_WORDS * i], host::G2Sel::Tau, host::G2Sel::NegGen, g2keys_))
                    item_status[i] = VERDICT_FAILS;
            });
            return Status::Ok();
        };
        result = run();
        if (!result.ok) ws.synchronize();     // (see verify_cell_kzg_proof_batch)
    }
    give_back(wsp, result);
    if (!result.ok) return result;
    if (items) {
        *verified = std::all_of(item_status, item_status + N, [](uint8_t v) { return v == VERDICT_OK; });
        return Status::Ok();
    }
    for (uint32_t v : stb) if (v) return Status::Error("Serialization(ScalarNotCanonical): blob");
    for (uint32_t v : stc) if (v) return Status::Error("Serialization(G1PointInvalid): commitment");
    for (uint32_t v : stp) if (v) return Status::Error("Serialization(G1PointInvalid): proof");
    for (uint32_t v : stz) if (v) return Status::Error("Serialization(ScalarNotCanonical): z");
    for (uint32_t v : sty) if (v) return Status::Error("Serialization(ScalarNotCanonical): y");
    *verified = run_pairing(pin, host::G2Sel::Tau, host::G2Sel::NegGen, g2keys_);
    return Status::Ok();
}

}  // namespace ekzg
