// Whole-shard transcript driver: ShardProver::prove_shard_with_data (crates/hypercube/src/prover/shard.rs:650-792; GPU twin
// sp1-gpu/crates/shard_prover/src/prover.rs:618-763) composed from the phase entry points of this library:
// observe public values -> jagged commit of the main traces -> observe commitment and chip table shapes -> LogUp-GKR ->
// sample alpha, gamma -> zerocheck -> jagged evaluation proof at the zerocheck point.
#include "ctx.cuh"
#include "challenger.cuh"
#include "hostfield.hpp"
#include "machine.cuh"
#include "pcs.cuh"
#include <cstring>
#include <memory>
#include <string>
#include <vector>

extern "C" {

// Proof words: [5][len_0..len_4] then the sections
//   0 main commitment (8) | 1 LogUp-GKR proof (sp1b200_logup_gkr words) | 2 zerocheck proof + opened values (sp1b200_zerocheck words) |
//   3 evaluation proof (sp1b200_jagged_prove words) | 4 public values
// = the fields of ShardProof (crates/hypercube/src/verifier/proof.rs:47-61); chip degrees are the heights the caller passed.
// h_replay_witnesses (grind_mode == 1): {gkr witness, batch grinding witness, pow witness}.
sp1b200_err sp1b200_prove_shard(sp1b200_ctx* ctx, const sp1b200_machine* m, sp1b200_jagged_round* prep_round, const uint32_t* main_dense_any,
                                const uint64_t* h_heights, const char* const* chip_names, const uint32_t* h_pv, uint32_t n_pv,
                                const uint32_t* h_replay_witnesses, uint32_t* h_chal, uint32_t* h_proof, uint64_t cap, uint64_t* h_words) { SP1_DEVICE_GUARD(ctx);
    using hf::E4;
    const size_t nch = m->chips.size();
    const uint32_t mlr = ctx->params.max_log_row_count;
    PhaseTimer t_all(ctx, "shard.total");
    HostChallenger ch;
    SP1_TRY(ch.init(ctx, h_chal));
    ch.observe_n(h_pv, n_pv);
    // main commit
    std::vector<uint64_t> rows(nch), cols(nch);
    for (size_t k = 0; k < nch; k++) { rows[k] = h_heights[k]; cols[k] = m->chips[k].main_w; }
    uint32_t commit[8];
    sp1b200_jagged_round* main_round = nullptr;
    {
        PhaseTimer t(ctx, "shard.commit");
        SP1_TRY(sp1b200_jagged_commit(ctx, main_dense_any, (uint32_t)nch, rows.data(), cols.data(), 1, commit, &main_round));
        t.stop();
    }
    struct Guard { sp1b200_ctx* c; sp1b200_jagged_round* r; ~Guard() { sp1b200_jagged_round_free(c, r); } } guard{ctx, main_round};
    ch.observe_n(commit, 8);
    ch.observe(hf::to_monty(nch));
    for (size_t k = 0; k < nch; k++) {
        ch.observe(hf::to_monty(h_heights[k]));
        const size_t len = strlen(chip_names[k]);
        ch.observe(hf::to_monty(len));
        for (size_t i = 0; i < len; i++) ch.observe(hf::to_monty((uint8_t)chip_names[k][i]));
    }
    // chip column pointers inside the dense buffers
    std::vector<const uint32_t*> d_main(nch, nullptr), d_prep(nch, nullptr);
    {
        uint64_t off = 0, poff = 0; size_t pt = 0;
        for (size_t k = 0; k < nch; k++) {
            d_main[k] = main_round->d_dense + off;
            off += h_heights[k] * m->chips[k].main_w;
            if (m->chips[k].prep_w) {
                if (!prep_round || pt + 2 >= prep_round->row_counts.size() + 0 || prep_round->col_counts[pt] != m->chips[k].prep_w)
                    return sp1b200_set_error("prove_shard: preprocessed round does not match the machine at chip %zu", k);
                if (prep_round->row_counts[pt] != h_heights[k])
                    return sp1b200_set_error("prove_shard: chip %zu: preprocessed height %llu != main height %llu", k,
                                             (unsigned long long)prep_round->row_counts[pt], (unsigned long long)h_heights[k]);
                d_prep[k] = prep_round->d_dense + poff;
                poff += prep_round->row_counts[pt] * prep_round->col_counts[pt];
                pt++;
            }
        }
    }
    uint32_t st[34];
    ch.store(st);
    // per-context scratch for the phase outputs, allocated once and reused by every shard proven on this context (uninitialised:
    // zero-filling 3 x 64 MiB per shard would cost more than some of the phases)
    const uint64_t scratch_cap = (uint64_t)1 << 24;
    if (!ctx->shard_scratch) ctx->shard_scratch.reset(new uint32_t[3 * scratch_cap]);
    uint32_t* gkr = ctx->shard_scratch.get();
    uint64_t n_gkr = 0;
    SP1_TRY(sp1b200_logup_gkr(ctx, m, h_heights, d_main.data(), d_prep.data(), h_replay_witnesses, st, gkr, scratch_cap, &n_gkr));
    // tail of the gkr words: point (mlr ext) | per chip {main, prep openings} | witness
    size_t total_w = 0;
    for (auto& c : m->chips) total_w += c.main_w + c.prep_w;
    if (n_gkr < 1 + 4 * total_w + 4 * (uint64_t)mlr)
        return sp1b200_set_error("prove_shard: LogUp-GKR section has %llu words, fewer than its point + openings + witness tail", (unsigned long long)n_gkr);
    const uint32_t* tail = gkr + n_gkr - 1 - 4 * total_w - 4 * mlr;
    const uint32_t* gkr_point = tail;
    const uint32_t* openings = tail + 4 * mlr;
    ch.load(st);
    E4 alpha, gamma;
    ch.sample_ext(alpha.c); ch.sample_ext(gamma.c);
    std::vector<uint32_t> claims(nch * 4);
    {
        const uint32_t* o = openings;
        for (size_t k = 0; k < nch; k++) {
            E4 acc, g = gamma;
            for (uint32_t j = 0; j < m->chips[k].main_w + m->chips[k].prep_w; j++, o += 4) { acc = acc + E4::load(o) * g; g = g * gamma; }
            acc.store(&claims[4 * k]);
        }
    }
    ch.store(st);
    uint32_t* zc = gkr + scratch_cap;
    uint64_t n_zc = 0;
    SP1_TRY(sp1b200_zerocheck(ctx, m, h_heights, d_main.data(), d_prep.data(), h_pv, n_pv, gkr_point, alpha.c, gamma.c, claims.data(), st, zc,
                              scratch_cap, &n_zc));
    // zerocheck words: [mlr] { [5] coeffs(20) } x mlr | claimed_sum 4 | point 4 mlr | eval 4 | per chip {prep evals, main evals}
    if (n_zc != 1 + (uint64_t)mlr * 21 + 4 + 4 * (uint64_t)mlr + 4 + 4 * total_w || zc[0] != mlr)
        return sp1b200_set_error("prove_shard: zerocheck section has %llu words, layout expects %llu", (unsigned long long)n_zc,
                                 (unsigned long long)(1 + (uint64_t)mlr * 21 + 4 + 4 * (uint64_t)mlr + 4 + 4 * total_w));
    const uint32_t* zpoint = zc + 1 + (size_t)mlr * 21 + 4;
    const uint32_t* zopen = zpoint + 4 * mlr + 4;
    std::vector<uint32_t> jclaims;
    {
        std::vector<uint32_t> pc, mc;
        const uint32_t* o = zopen;
        for (size_t k = 0; k < nch; k++) {
            pc.insert(pc.end(), o, o + 4 * m->chips[k].prep_w); o += 4 * m->chips[k].prep_w;
            mc.insert(mc.end(), o, o + 4 * m->chips[k].main_w); o += 4 * m->chips[k].main_w;
        }
        if (prep_round) jclaims.insert(jclaims.end(), pc.begin(), pc.end());
        jclaims.insert(jclaims.end(), mc.begin(), mc.end());
    }
    std::vector<sp1b200_jagged_round*> rounds;
    if (prep_round) rounds.push_back(prep_round);
    rounds.push_back(main_round);
    uint32_t* ev = gkr + 2 * scratch_cap;
    uint64_t n_ev = 0;
    SP1_TRY(sp1b200_jagged_prove(ctx, rounds.data(), (uint32_t)rounds.size(), zpoint, jclaims.data(), h_replay_witnesses ? h_replay_witnesses + 1 : nullptr,
                                 st, ev, scratch_cap, &n_ev));
    const uint64_t total = 6 + 8 + n_gkr + n_zc + n_ev + n_pv;
    t_all.stop();
    if (h_words) *h_words = total;
    // the caller's challenger is advanced only together with a delivered proof: on a capacity error h_chal is untouched and
    // *h_words holds the size to retry with
    if (h_proof && total > cap) return sp1b200_set_error("prove_shard: proof needs %llu words, capacity %llu", (unsigned long long)total, (unsigned long long)cap);
    memcpy(h_chal, st, sizeof(st));
    if (h_proof) {
        uint32_t* o = h_proof;
        const uint32_t hdr[6] = {5, 8, (uint32_t)n_gkr, (uint32_t)n_zc, (uint32_t)n_ev, n_pv};
        memcpy(o, hdr, 24); o += 6;
        memcpy(o, commit, 32); o += 8;
        memcpy(o, gkr, n_gkr * 4); o += n_gkr;
        memcpy(o, zc, n_zc * 4); o += n_zc;
        memcpy(o, ev, n_ev * 4); o += n_ev;
        memcpy(o, h_pv, n_pv * 4);
    }
    return nullptr;
}

// AirProver::setup_and_prove_shard (shard.rs:56-68): setup = commit the preprocessed traces, observe the verifying key
// (MachineVerifyingKey::observe_into, verifier/config.rs:97-112: commitment, then the program-dependent words), prove.
sp1b200_err sp1b200_setup_and_prove_shard(sp1b200_ctx* ctx, const sp1b200_machine* m, const uint32_t* prep_dense_any, uint32_t n_prep,
                                          const uint64_t* h_prep_rows, const uint64_t* h_prep_cols, const uint32_t* h_vk_tail, uint32_t n_vk_tail,
                                          const uint32_t* main_dense_any, const uint64_t* h_heights, const char* const* chip_names,
                                          const uint32_t* h_pv, uint32_t n_pv, const uint32_t* h_replay_witnesses, uint32_t* h_chal,
                                          uint32_t* h_prep_commit8, sp1b200_jagged_round** prep_round_out, uint32_t* h_proof, uint64_t cap,
                                          uint64_t* h_words) { SP1_DEVICE_GUARD(ctx);
    if (!prep_round_out) return sp1b200_set_error("setup_and_prove_shard: prep_round_out is NULL");
    *prep_round_out = nullptr;
    uint32_t commit[8] = {0};
    sp1b200_jagged_round* prep = nullptr;
    if (n_prep) SP1_TRY(sp1b200_jagged_commit(ctx, prep_dense_any, n_prep, h_prep_rows, h_prep_cols, 1, commit, &prep));
    HostChallenger ch;
    sp1b200_err e = ch.init(ctx, h_chal);
    if (!e) {
        ch.observe_n(commit, 8);
        ch.observe_n(h_vk_tail, n_vk_tail);
        uint32_t st[34];
        ch.store(st);
        e = sp1b200_prove_shard(ctx, m, prep, main_dense_any, h_heights, chip_names, h_pv, n_pv, h_replay_witnesses, st, h_proof, cap, h_words);
        if (!e) memcpy(h_chal, st, sizeof(st));
    }
    if (e) { sp1b200_jagged_round_free(ctx, prep); return e; }
    if (h_prep_commit8) memcpy(h_prep_commit8, commit, 32);
    *prep_round_out = prep;
    return nullptr;
}
}
