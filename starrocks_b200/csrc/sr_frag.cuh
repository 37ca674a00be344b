// sr_frag.cuh -- the fused pipeline fragment: scan -> filter -> [hash-join probe]* -> aggregate
// in ONE pass over the fact columns.  This is the hot kernel of the SSB Q4.1 / Q1.1 configs.
//
// What it fuses (reference call stack, SURVEY.md section 3.3-3.5):
//   OlapChunkSource::_read_chunk_from_storage filter step   scan/olap_chunk_source.cpp:676-722
//   HashJoinProbeOperator::push_chunk/pull_chunk x N        hashjoin/hash_join_probe_operator.cpp:55-96
//     -> JoinHashMap::probe (lookup_init + _probe_from_ht + _probe_output/_build_output)
//   AggregateBlockingSinkOperator::push_chunk               aggregate/aggregate_blocking_sink_operator.cpp:101-138
//
// B200 design (HBM-bound integer/gather work, no tensor cores):
//  * persistent CTAs (grid = SMs x resident CTAs).  The main loop streams the scan-predicate
//    columns and the FIRST join's key column: each thread owns groups of 4 consecutive rows, so a
//    tile column is one 128-bit ld.global.nc.L1::no_allocate per thread and group;
//  * selection-vector cascade: rows that survive stage k are appended (warp ballot + popc) to a
//    per-warp queue in shared memory; as soon as a queue holds 32 rows the warp runs stage k+1
//    for 32 rows at once (one row per lane).  Later stages therefore always execute with full
//    warps, their column loads are issued for 32 rows together, and the dependent-load chain of
//    a tile is one DRAM round trip instead of one per join;
//  * late materialisation: a column is only loaded for rows still alive, so DRAM sectors of later
//    columns are skipped when all 8 rows of a 32-byte sector were filtered out;
//  * every range-mapped join is tested against its 1-bit-per-key bitmap; the bitmaps of the
//    earliest joins are copied into shared memory once per CTA, the others are read through
//    L1/L2 (SSB dimension bitmaps are 25-375 KB and stay L2 resident);
//  * the build row index (first[]) and payload columns are only fetched for rows that survive all
//    joins; the group-by / SUM update of the final queue goes to shared-memory accumulators when
//    the table is small, flushed once per CTA;
//  * join order: pass rates measured on a sample of the first batch (adaptive), most selective
//    first, smaller table first on a tie -- inner joins commute, the result is order independent.
#pragma once

#include "sr_agg.cuh"

#include "sr_frag_kernel.cuh"
#include "sr_frag_pass.cuh"

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
struct sr_fragment {
    sr_ctx* ctx = nullptr;
    std::vector<sr_pred> preds;
    std::vector<sr_expr> exprs;
    int32_t num_joins = 0;
    sr_frag_join joins[SR_MAX_FRAG_JOINS];
    sr_agg* agg = nullptr;
    bool compiled = false;
    VReg reg; // fact + payload values
    std::vector<int32_t> value_src;         // per value: -1 fact, j = payload of (ordered) join j
    std::vector<const BuildCol*> value_col; // payload column for src >= 0
    srd::FragDev host;
    DevBuf dev, counters;
    Staged staged;
    size_t smem_bytes = 0;
    int32_t queue_word_off = 0;
    bool smem_agg = false;
    int grid = 0;
    int order[SR_MAX_FRAG_JOINS];
    double pass_rate[SR_MAX_FRAG_JOINS];
    double pred_rate = 1.0;
    // selective mode (sr_frag_pass.cuh): streaming pass -> gather passes -> final pass
    int force_mode = 0; // 0 = choose from the sampled pass rates, 1 = fused cascade kernel, 2 = selection-vector passes
    bool selective = false;
    bool expand = false; // some INNER join has duplicate build keys: selection-vector passes + k_frag_gather_agg_expand
    srd::PassDev pass;
    std::vector<int> gather_joins; // probe positions that get a pass of their own
    DevBuf sel[2], pass_counters;
    double est_rate = 1.0; // sampled fraction of the fact rows that reaches the aggregate
    size_t stream_smem = 0;
    int stream_grid = 0;
    int final_grid = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool timed_push = false;
    ~sr_fragment() {
        for (int e = 0; e < 4; e++)
            if (ev[e]) cudaEventDestroy(ev[e]);
    }
};

struct FragTypeCtx {
    sr_fragment* f;
};

// slot type: fact chunk first, then payload columns of the joins
static int32_t frag_slot_type(void* user, int32_t slot) {
    sr_fragment* f = ((FragTypeCtx*)user)->f;
    const int k = f->staged.find(slot);
    if (k >= 0) return f->staged.cols[k].type;
    for (int j = 0; j < f->num_joins; j++)
        for (int p = 0; p < f->joins[j].num_payload; p++)
            if (f->joins[j].payload_build_slots[p] == slot) {
                const BuildCol* bc = f->joins[j].join->find_col(slot);
                return bc ? bc->type : 0;
            }
    return 0;
}
static bool frag_slot_nullable(void* user, int32_t slot) {
    sr_fragment* f = ((FragTypeCtx*)user)->f;
    const int k = f->staged.find(slot);
    if (k >= 0) return f->staged.cols[k].nulls != nullptr;
    for (int j = 0; j < f->num_joins; j++)
        for (int p = 0; p < f->joins[j].num_payload; p++)
            if (f->joins[j].payload_build_slots[p] == slot) {
                const BuildCol* bc = f->joins[j].join->find_col(slot);
                return bc && bc->nullable;
            }
    return false;
}

static int32_t frag_bind_vtab(sr_fragment* f, VTab* vt) {
    sr_ctx* ctx = f->ctx;
    vt->n = (int32_t)f->reg.slots.size();
    for (size_t k = 0; k < f->reg.slots.size(); k++) {
        if (f->value_src[k] < 0) {
            const int c = f->staged.find(f->reg.slots[k]);
            if (c < 0) return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "fact chunk misses slot %d", f->reg.slots[k]);
            if (f->staged.cols[c].type != f->reg.types[k]) return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "fact slot %d changed type", f->reg.slots[k]);
            vt->v[k].data = f->staged.cols[c].data;
            vt->v[k].nulls = f->staged.cols[c].nulls;
            vt->v[k].type = f->staged.cols[c].type;
            vt->v[k].src = -1;
        } else {
            const BuildCol* bc = f->value_col[k];
            vt->v[k].data = bc->data.p;
            vt->v[k].nulls = bc->nullable ? (const uint8_t*)bc->nulls.p : nullptr;
            vt->v[k].type = bc->type;
            vt->v[k].src = f->value_src[k];
        }
    }
    vt_mark_plain32(vt);
    return SR_OK;
}

static int32_t frag_compile(sr_fragment* f) {
    sr_ctx* ctx = f->ctx;
    FragTypeCtx tc{f};
    srd::FragDev& h = f->host;
    memset(&h, 0, sizeof(h));
    f->reg = VReg();
    if (f->preds.size() > 8 || f->exprs.size() > 4) return sr_fail(ctx, SR_ERR_NOT_SUPPORTED, "too many scan conjuncts for the fused fragment");
    for (size_t k = 0; k < f->preds.size(); k++) SR_TRY(compile_pred(ctx, &f->preds[k], &f->reg, frag_slot_type, &tc, &h.preds[k]));
    for (size_t k = 0; k < f->exprs.size(); k++) {
        SR_TRY(compile_expr(ctx, &f->exprs[k], &f->reg, frag_slot_type, &tc, &h.exprs[k]));
        if (h.exprs[k].result_is_double) return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "filter expression %zu is not boolean", k);
    }
    h.num_preds = (int32_t)f->preds.size();
    h.num_exprs = (int32_t)f->exprs.size();
    h.num_joins = f->num_joins;
    // join keys (identity order for now; reordered after sampling)
    for (int j = 0; j < f->num_joins; j++) {
        sr_join* jn = f->joins[j].join;
        const int c = f->staged.find(f->joins[j].probe_key_slot);
        if (c < 0) return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "fact chunk misses probe key slot %d", f->joins[j].probe_key_slot);
        if (srd::is_float_class(f->staged.cols[c].type) || f->staged.cols[c].width > 8)
            return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "probe key slot %d has a non-integer type", f->joins[j].probe_key_slot);
        if (f->staged.cols[c].width != srd::type_width(jn->desc.key_types[0]))
            return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "probe key slot %d width differs from the join's key type", f->joins[j].probe_key_slot);
        const int id = f->reg.add(f->joins[j].probe_key_slot, f->staged.cols[c].type);
        if (id >= SR_MAX_VALUES) return sr_fail(ctx, SR_ERR_NOT_SUPPORTED, "too many distinct columns");
        h.joins[j].key_value_id = id;
        h.joins[j].j = jn->dev();
        h.joins[j].smem_off = -1;
        h.joins[j].use_bitmap = jn->method != SR_JOIN_METHOD_LINEAR_CHAINED ? 1 : 0;
        h.joins[j].bitmap_words = (int32_t)((std::max<int64_t>(jn->bucket_size, 1) + 31) / 32);
        // one-to-many INNER join: the final pass walks the build chain of every surviving row
        h.joins[j].expand = (jn->has_dup && jn->desc.join_type == SR_JOIN_INNER) ? 1 : 0;
        h.joins[j].need_head = h.joins[j].expand;
        h.joins[j].idx32 = (h.joins[j].use_bitmap && jn->min_value >= INT32_MIN && jn->max_value <= INT32_MAX && jn->max_value >= jn->min_value) ? 1 : 0;
        f->order[j] = j;
    }
    // aggregate (its expressions may reference fact slots and payload slots)
    SR_TRY(agg_compile(f->agg, frag_slot_type, frag_slot_nullable, &tc));
    // the fragment and its aggregate share one value table: rebuild the aggregate's value ids on top
    // of the fragment registry
    {
        VReg merged = f->reg;
        std::vector<int> remap(f->agg->reg.slots.size());
        for (size_t k = 0; k < f->agg->reg.slots.size(); k++) {
            remap[k] = merged.add(f->agg->reg.slots[k], f->agg->reg.types[k]);
            if (remap[k] >= SR_MAX_VALUES) return sr_fail(ctx, SR_ERR_NOT_SUPPORTED, "too many distinct columns");
        }
        srd::AggDev& ah = f->agg->host;
        for (int k = 0; k < ah.num_keys; k++) ah.key_value_id[k] = remap[ah.key_value_id[k]];
        for (int q = 0; q < ah.num_fns; q++)
            for (int k = 0; k < ah.fns[q].input.num_nodes; k++)
                if (ah.fns[q].input.nodes[k].op == srd::C_LOAD_I || ah.fns[q].input.nodes[k].op == srd::C_LOAD_D)
                    ah.fns[q].input.nodes[k].arg = remap[ah.fns[q].input.nodes[k].arg];
        f->agg->reg = merged;
        f->reg = merged;
        SR_TRY(agg_upload(f->agg));
    }
    // classify values: fact column or payload of join j
    f->value_src.assign(f->reg.slots.size(), -1);
    f->value_col.assign(f->reg.slots.size(), nullptr);
    for (size_t k = 0; k < f->reg.slots.size(); k++) {
        if (f->staged.find(f->reg.slots[k]) >= 0) continue;
        bool found = false;
        for (int j = 0; j < f->num_joins && !found; j++)
            for (int p = 0; p < f->joins[j].num_payload && !found; p++)
                if (f->joins[j].payload_build_slots[p] == f->reg.slots[k]) {
                    f->value_src[k] = j;
                    f->value_col[k] = f->joins[j].join->find_col(f->reg.slots[k]);
                    h.joins[j].need_head = 1;
                    found = true;
                }
        if (!found) return sr_fail(ctx, SR_ERR_INVALID_ARGUMENT, "slot %d is neither a fact column nor a join payload", f->reg.slots[k]);
    }
    SR_TRY(f->counters.reserve(ctx, 256));
    SR_CUDA(ctx, cudaMemsetAsync(f->counters.p, 0, 256, ctx->stream));
    h.rows_passed = f->counters.as<unsigned long long>();
    return SR_OK;
}

// sample pass rates, order the joins, assign shared-memory bitmaps, upload, pick the grid
static int32_t frag_plan(sr_fragment* f, const VTab& vt, int64_t n) {
    sr_ctx* ctx = f->ctx;
    srd::FragDev& h = f->host;
    SR_TRY(f->dev.reserve(ctx, sizeof(srd::FragDev)));
    SR_CUDA(ctx, cudaMemcpyAsync(f->dev.p, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    const int64_t sample = std::min<int64_t>(n, 1 << 16);
    unsigned long long counts[24] = {0}; // [0, 6): joins, [6]: all conjuncts, [16 + p]: conjuncts 0..p
    static_assert(SR_MAX_FRAG_JOINS + 1 <= 16, "sample counter layout");
    counts[SR_MAX_FRAG_JOINS] = (unsigned long long)sample;
    for (int p = 0; p < 8; p++) counts[16 + p] = (unsigned long long)sample;
    if (sample > 0 && (f->num_joins > 0 || h.num_preds > 0 || h.num_exprs > 0)) {
        unsigned long long* dcounts = f->counters.as<unsigned long long>() + 8;
        SR_CUDA(ctx, cudaMemsetAsync(dcounts, 0, sizeof(counts), ctx->stream));
        srd::k_frag_sample<<<grid_for(sample, 256), 256, 0, ctx->stream>>>((const srd::FragDev*)f->dev.p, vt, sample, dcounts);
        SR_LAUNCH_CHECK(ctx);
        SR_CUDA(ctx, cudaMemcpyAsync(counts, dcounts, sizeof(counts), cudaMemcpyDeviceToHost, ctx->stream));
        SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    for (int j = 0; j < f->num_joins; j++) f->pass_rate[j] = sample > 0 ? (double)counts[j] / (double)sample : 1.0;
    f->pred_rate = sample > 0 ? (double)counts[SR_MAX_FRAG_JOINS] / (double)sample : 1.0;
    std::vector<int> ord(f->num_joins);
    for (int j = 0; j < f->num_joins; j++) ord[j] = j;
    // most selective first; pass rates within 15 % of each other count as a tie -> smaller table first
    // (the first join sees every row: its bitmap should fit shared memory)
    std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) {
        const double pa = f->pass_rate[a], pb = f->pass_rate[b];
        if (std::abs(pa - pb) > 0.15 * std::max(pa, pb)) return pa < pb;
        return h.joins[a].bitmap_words < h.joins[b].bitmap_words;
    });
    srd::FragJoinDev reordered[SR_MAX_FRAG_JOINS];
    std::vector<int> inv(f->num_joins);
    for (int q = 0; q < f->num_joins; q++) {
        reordered[q] = h.joins[ord[q]];
        inv[ord[q]] = q;
        f->order[q] = ord[q];
    }
    for (int q = 0; q < f->num_joins; q++) h.joins[q] = reordered[q];
    for (size_t k = 0; k < f->value_src.size(); k++)
        if (f->value_src[k] >= 0) f->value_src[k] = inv[f->value_src[k]];
    // stream the second join's key together with the first when most of its 64-byte DRAM bursts would
    // be touched anyway: 1 - (1 - p)^16 >= 0.74 for p >= 0.08
    h.eager1 = (f->num_joins >= 2 && f->pass_rate[ord[0]] >= 0.08) ? 1 : 0;
    // ---- mode: when few rows reach the aggregate, run selection-vector passes instead of the cascade ----
    double total_rate = f->pred_rate;
    for (int q = 0; q < f->num_joins; q++) total_rate *= f->pass_rate[ord[q]];
    f->est_rate = total_rate;
    f->selective = f->expand || f->force_mode == 2 || (f->force_mode == 0 && total_rate < 0.25 && n >= (1 << 16));
    if (f->selective) {
        // joins whose key column is streamed: the first one, and the second when >= 8 % of the rows reach it
        int ns = f->num_joins > 0 ? 1 : 0;
        if (f->num_joins > 1 && f->pred_rate * f->pass_rate[ord[0]] >= 0.08) ns = 2;
        // trailing joins that filter (almost) nothing are tested inline by the final pass
        int ff = f->num_joins;
        while (ff > ns && f->pass_rate[ord[ff - 1]] >= 0.9) ff--;
        memset(&f->pass, 0, sizeof(f->pass));
        f->pass.num_stream_joins = ns;
        f->pass.final_first_join = ff;
        // a streamed join whose build row the final pass looks up (payload) hands its int32 key over through the
        // selection vector: one random fact-sector read less per surviving row
        f->pass.carry_join = -1;
        f->pass.carry_value_id = -1;
        for (int q = 0; q < ns; q++) {
            const int id = h.joins[q].key_value_id;
            const int32_t kt = f->reg.types[id];
            if (h.joins[q].need_head && srd::type_width(kt) == 4 && !srd::is_float_class(kt) && id < 127) {
                f->pass.carry_join = (int8_t)q;
                f->pass.carry_value_id = (int8_t)id;
                break;
            }
        }
        // the streaming pass in "tests" form (k_frag_stream_tests): every scan conjunct must reduce to an int32 range
        // and every streamed column must be int32-class; otherwise the generic streaming kernel runs
        {
            bool ok = h.num_exprs == 0 && h.num_preds + ns > 0 && h.num_preds + ns <= SR_MAX_STREAM_TESTS;
            int nt = 0;
            auto int32_class = [&](int id) { return srd::type_width(f->reg.types[id]) == 4 && !srd::is_float_class(f->reg.types[id]); };
            for (int p = 0; p < h.num_preds && ok; p++) {
                const srd::CPred& cp = h.preds[p];
                long long lo = INT32_MIN, hi = INT32_MAX;
                switch (cp.op) {
                case SR_PRED_EQ: lo = hi = cp.ilo; break;
                case SR_PRED_LT: hi = cp.ilo - 1; break;
                case SR_PRED_LE: hi = cp.ilo; break;
                case SR_PRED_GT: lo = cp.ilo + 1; break;
                case SR_PRED_GE: lo = cp.ilo; break;
                case SR_PRED_BETWEEN: lo = cp.ilo; hi = cp.ihi; break;
                default: ok = false; break;
                }
                lo = std::max<long long>(lo, INT32_MIN);
                hi = std::min<long long>(hi, INT32_MAX);
                if (cp.is_double || !int32_class(cp.value_id) || lo > hi) ok = false;
                if (!ok) break;
                srd::StreamTest& st = f->pass.tests[nt++];
                st.kind = 0;
                st.value_id = cp.value_id;
                st.join = -1;
                st.lo = (uint32_t)(int32_t)lo;
                st.span = (uint32_t)(hi - lo);
            }
            for (int q = 0; q < ns && ok; q++) {
                if (!int32_class(h.joins[q].key_value_id)) {
                    ok = false;
                    break;
                }
                srd::StreamTest& st = f->pass.tests[nt++];
                st.kind = 1;
                st.value_id = h.joins[q].key_value_id;
                st.join = q;
                st.lo = st.span = 0;
            }
            f->pass.num_tests = ok ? nt : 0;
            // the second test's column is streamed with vector loads as well when >= 8 % of the rows reach it
            // (most of its 64-byte DRAM bursts would be touched anyway, and the loads do not wait for test 0)
            double reach1 = 1.0;
            if (ok && nt > 1) reach1 = f->pass.tests[0].kind == 0 ? (double)counts[16] / (double)std::max<int64_t>(sample, 1) : f->pred_rate * f->pass_rate[ord[0]];
            f->pass.num_vec = (ok && nt > 1 && reach1 >= 0.08) ? 2 : 1;
        }
        f->gather_joins.clear();
        for (int q = ns; q < ff; q++) f->gather_joins.push_back(q);
        // streaming pass shared memory: bitmaps of the streamed joins only
        size_t sw = 0;
        const size_t sbudget = (100 * 1024) / 4;
        for (int q = 0; q < f->num_joins; q++) {
            srd::FragJoinDev& fj = h.joins[q];
            fj.smem_off = -1;
            if (q < ns && fj.use_bitmap && sw + (size_t)fj.bitmap_words + 1 <= sbudget) {
                fj.smem_off = (int32_t)sw;
                sw += ((size_t)fj.bitmap_words + 1 + 3) & ~(size_t)3; // + one zero guard word (stream_test_reg kind 1)
            }
        }
        f->stream_smem = sw * 4;
        f->smem_agg = f->agg->smem_bytes > 0;
        f->smem_bytes = f->agg->smem_bytes;
        f->queue_word_off = 0;
        SR_CUDA(ctx, cudaMemcpyAsync(f->dev.p, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
        SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        int per_sm = 0;
        SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_frag_stream<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(f->stream_smem, 16)));
        SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_frag_stream<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(f->stream_smem, 16)));
        SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_frag_stream_tests<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(f->stream_smem, 16)));
        SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_frag_stream_tests<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(f->stream_smem, 16)));
        SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, srd::k_frag_stream<false>, srd::STREAM_BLOCK, f->stream_smem));
        if (per_sm < 1) return sr_fail(ctx, SR_ERR_CUDA, "streaming pass does not fit on an SM (smem %zu)", f->stream_smem);
        f->stream_grid = per_sm * ctx->num_sms;
        // gather passes: exactly one wave of resident CTAs (grid-stride loops; a partial second wave only adds a tail)
        int gj = 0, ga = 0;
        SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&gj, srd::k_frag_gather_join, srd::GATHER_BLOCK, 0));
        if (f->expand)
            SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ga, srd::k_frag_gather_agg_expand, srd::GATHER_BLOCK, 0));
        else if (f->agg->host.num_keys == 0)
            SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ga, srd::k_frag_gather_agg<false, true>, srd::GATHER_BLOCK, 0));
        else if (f->smem_agg)
            SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ga, srd::k_frag_gather_agg<true>, srd::GATHER_BLOCK, f->agg->smem_bytes));
        else
            SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ga, srd::k_frag_gather_agg<false>, srd::GATHER_BLOCK, 0));
        f->grid = std::max(gj, 1) * ctx->num_sms;
        f->final_grid = std::max(ga, 1) * ctx->num_sms;
        SR_TRY(f->pass_counters.reserve(ctx, 16 * sizeof(uint64_t)));
        f->compiled = true;
        return SR_OK;
    }
    // dynamic shared memory: [aggregate accumulators | bitmaps | per-warp queues]
    size_t words = 0;
    f->smem_agg = f->agg->smem_bytes > 0;
    if (f->smem_agg) words += (f->agg->smem_bytes + 15) / 16 * 4;
    const size_t budget_words = (96 * 1024) / 4; // keeps 2 CTAs of 512 threads resident per SM
    const size_t queue_words = (size_t)srd::FRAG_WARPS * srd::FRAG_WARP_QWORDS;
    for (int q = 0; q < f->num_joins; q++) {
        srd::FragJoinDev& fj = h.joins[q];
        fj.smem_off = -1;
        if (fj.use_bitmap && words + (size_t)fj.bitmap_words + queue_words <= budget_words) {
            fj.smem_off = (int32_t)words;
            words += (size_t)fj.bitmap_words;
            words = (words + 3) & ~(size_t)3;
        }
    }
    f->queue_word_off = (int32_t)words;
    words += queue_words;
    f->smem_bytes = words * 4;
    SR_CUDA(ctx, cudaMemcpyAsync(f->dev.p, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    // occupancy-sized persistent grid
    int per_sm = 0;
    SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_fragment<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f->smem_bytes));
    SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_fragment<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f->smem_bytes));
    if (f->smem_agg)
        SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, srd::k_fragment<true>, srd::FRAG_BLOCK, f->smem_bytes));
    else
        SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, srd::k_fragment<false>, srd::FRAG_BLOCK, f->smem_bytes));
    if (per_sm < 1) return sr_fail(ctx, SR_ERR_CUDA, "fragment kernel does not fit on an SM (smem %zu)", f->smem_bytes);
    f->grid = per_sm * ctx->num_sms;
    f->compiled = true;
    return SR_OK;
}

static int32_t frag_push(sr_fragment* f, const sr_chunk_view* fact) {
    sr_ctx* ctx = f->ctx;
    if (f->agg->finished) return sr_fail(ctx, SR_ERR_STATE, "fragment push after sink_finish");
    if (fact->num_rows >= 0xFFFFFFF0ll) return sr_fail(ctx, SR_ERR_NOT_SUPPORTED, "fragment batch of more than 2^32 rows; push smaller morsels");
    // page-locked mapped host columns are read in place: the passes after the first only touch the sectors of
    // surviving rows, so most of the batch never crosses PCIe
    SR_TRY(f->staged.stage(ctx, fact, nullptr, /*in_place_pinned=*/true));
    const int64_t n = fact->num_rows;
    bool first = !f->compiled;
    if (first) SR_TRY(frag_compile(f));
    VTab vt;
    SR_TRY(frag_bind_vtab(f, &vt));
    if (first) {
        SR_TRY(frag_plan(f, vt, n));
        SR_TRY(frag_bind_vtab(f, &vt)); // the plan reorders the joins: payload values now point at the new positions
    }
    if (n == 0) return SR_OK;
    SR_TRY(agg_check_nullability(f->agg, vt));
    if (f->agg->smem_bytes == 0 && f->smem_agg) f->smem_agg = false; // a nullability change forced global accumulation
    sr_agg* a = f->agg;
    a->table_touched = true;
    const srd::AggDev& ah = a->host;
    const bool hash = !ah.dense && ah.num_keys > 0;
    if (hash) {
        // Survivors are unknown before the pass.  The single-kernel cascade has no way to retry a row, so its table is
        // made large enough for the worst case (every row a new group).  The selection-vector passes size the table
        // from the sampled survivor estimate (x2 + slack) and re-apply the rows the table refused after growing it.
        uint64_t want = (uint64_t)n;
        if (f->selective) want = std::min<uint64_t>((uint64_t)n, (uint64_t)((double)n * std::min(1.0, f->est_rate) * 2.0) + (1u << 16));
        while ((uint64_t)a->ngroups_host + want > a->host.limit) {
            if (a->host.cap >= (1ull << 33)) return sr_fail(ctx, SR_ERR_OUT_OF_MEMORY, "aggregate table would exceed 2^33 slots; push smaller batches");
            SR_TRY(agg_grow(a, a->host.cap * 4));
        }
    }
    if (f->selective) {
        const srd::FragDev* fdev = (const srd::FragDev*)f->dev.p;
        // worst case every row survives, plus one partly used chunk per warp of the writing pass
        const size_t slack = (size_t)srd::SEL_CHUNK * ((size_t)f->stream_grid * (srd::STREAM_BLOCK / 32) + (size_t)f->grid * (srd::GATHER_BLOCK / 32));
        SR_TRY(f->sel[0].reserve(ctx, sizeof(srd::SelEntry) * ((size_t)n + slack)));
        if (!f->gather_joins.empty()) SR_TRY(f->sel[1].reserve(ctx, sizeof(srd::SelEntry) * ((size_t)n + slack)));
        // this push's pass parameters: the carried key (planned in f->pass) is only used for host-resident input
        srd::PassDev pass = f->pass;
        const bool pinned_input = fact->mem == SR_MEM_HOST_PINNED;
        const bool carry = pinned_input && pass.carry_join >= 0; // (HBM input, measured: stream +0.27 ms, final -0.09 ms)
        if (!carry) pass.carry_join = pass.carry_value_id = -1;
        unsigned long long* cnt = f->pass_counters.as<unsigned long long>();
        SR_CUDA(ctx, cudaMemsetAsync(cnt, 0, 16 * sizeof(uint64_t), ctx->stream));
        const int sgrid = (int)std::min<int64_t>(f->stream_grid, (n + srd::STREAM_TILE - 1) / srd::STREAM_TILE);
        // pass boundaries are bracketed with CUDA events (bench.py reads them back as per-kernel durations)
        if (!f->ev[0])
            for (int e = 0; e < 4; e++) SR_CUDA(ctx, cudaEventCreate(&f->ev[e]));
        SR_CUDA(ctx, cudaEventRecord(f->ev[0], ctx->stream));
        // range-form conjuncts and streamed joins on plain (non-nullable) int32 columns -> the tests kernel;
        // everything else -> the generic streaming kernel
        bool tests = pass.num_tests > 0;
        for (int t = 0; t < pass.num_tests && tests; t++) {
            const VDesc& d = vt.v[pass.tests[t].value_id];
            if (d.nulls != nullptr || (t < pass.num_vec && (((uintptr_t)d.data) & 15) != 0)) tests = false;
        }
        if (tests) {
            if (carry)
                srd::k_frag_stream_tests<true><<<sgrid, srd::STREAM_BLOCK, f->stream_smem, ctx->stream>>>(fdev, pass, vt, n, f->sel[0].as<srd::SelEntry>(), cnt);
            else
                srd::k_frag_stream_tests<false><<<sgrid, srd::STREAM_BLOCK, f->stream_smem, ctx->stream>>>(fdev, pass, vt, n, f->sel[0].as<srd::SelEntry>(), cnt);
        } else if (carry) {
            srd::k_frag_stream<true><<<sgrid, srd::STREAM_BLOCK, f->stream_smem, ctx->stream>>>(fdev, pass, vt, n, f->sel[0].as<srd::SelEntry>(), cnt);
        } else {
            srd::k_frag_stream<false><<<sgrid, srd::STREAM_BLOCK, f->stream_smem, ctx->stream>>>(fdev, pass, vt, n, f->sel[0].as<srd::SelEntry>(), cnt);
        }
        SR_LAUNCH_CHECK(ctx);
        SR_CUDA(ctx, cudaEventRecord(f->ev[1], ctx->stream));
        int cur = 0, k = 0;
        for (int q : f->gather_joins) {
            srd::k_frag_gather_join<<<f->grid, srd::GATHER_BLOCK, 0, ctx->stream>>>(fdev, q, vt, f->sel[cur].as<srd::SelEntry>(), cnt + k,
                                                                                  f->sel[cur ^ 1].as<srd::SelEntry>(), cnt + k + 1);
            SR_LAUNCH_CHECK(ctx);
            cur ^= 1;
            k++;
        }
        SR_CUDA(ctx, cudaEventRecord(f->ev[2], ctx->stream));
        // the final pass over sel_in[0, *n_in); rows the hash table refuses are appended to fail_list (nullptr: no hash
        // table).  Only a dense table is accumulated in shared memory (agg_compile), so a hash table always takes
        // k_frag_gather_agg<false> or the expand kernel, the first pass and its retries alike.
        auto final_pass = [&](const srd::SelEntry* sel_in, const unsigned long long* n_in, srd::SelEntry* fail_list,
                              unsigned long long* fail_count) -> int32_t {
            const srd::AggDev* adev = (const srd::AggDev*)a->dev.p;
            if (f->expand)
                srd::k_frag_gather_agg_expand<<<f->final_grid, srd::GATHER_BLOCK, 0, ctx->stream>>>(fdev, adev, pass, vt, sel_in, n_in, fail_list, fail_count);
            else if (ah.num_keys == 0)
                srd::k_frag_gather_agg<false, true><<<f->final_grid, srd::GATHER_BLOCK, 0, ctx->stream>>>(fdev, adev, pass, vt, sel_in, n_in, fail_list, fail_count);
            else if (f->smem_agg)
                srd::k_frag_gather_agg<true><<<f->final_grid, srd::GATHER_BLOCK, a->smem_bytes, ctx->stream>>>(fdev, adev, pass, vt, sel_in, n_in, fail_list, fail_count);
            else
                srd::k_frag_gather_agg<false><<<f->final_grid, srd::GATHER_BLOCK, 0, ctx->stream>>>(fdev, adev, pass, vt, sel_in, n_in, fail_list, fail_count);
            SR_LAUNCH_CHECK(ctx);
            return SR_OK;
        };
        // hash table: rows it refuses go to the other selection buffer (free by now) and are retried after a growth
        if (hash) SR_TRY(f->sel[cur ^ 1].reserve(ctx, sizeof(srd::SelEntry) * ((size_t)n + slack)));
        SR_TRY(final_pass(f->sel[cur].as<srd::SelEntry>(), cnt + k, hash ? f->sel[cur ^ 1].as<srd::SelEntry>() : nullptr, cnt + 8));
        SR_CUDA(ctx, cudaEventRecord(f->ev[3], ctx->stream));
        f->timed_push = true;
        if (hash) {
            int fc = 8; // index of the live fail counter in `cnt`
            while (true) {
                uint64_t ng;
                int32_t ovf, bad;
                SR_CUDA(ctx, cudaMemcpyAsync(ctx->pinned + 16, cnt + fc, 8, cudaMemcpyDeviceToHost, ctx->stream));
                SR_TRY(agg_read_counters(a, &ng, &ovf, &bad)); // synchronises
                a->ngroups_host = (int64_t)ng;
                const uint64_t failed = ctx->pinned[16];
                if (failed == 0) break;
                // grow so that the refused rows fit even if each of them is a new group, then re-apply them
                SR_CUDA(ctx, cudaMemsetAsync((uint8_t*)a->counters.p + 8, 0, 8, ctx->stream)); // overflow / range flags
                // (always at least doubled: a refused row of a one-to-many join may bring several new groups, and a
                // full 256-slot slice refuses rows below the admission limit)
                uint64_t cap = a->host.cap * 2;
                while ((uint64_t)a->ngroups_host + failed > cap / 2) cap *= 2;
                if (cap > (1ull << 33)) return sr_fail(ctx, SR_ERR_OUT_OF_MEMORY, "aggregate table would exceed 2^33 slots; push smaller batches");
                SR_TRY(agg_grow(a, cap));
                cur ^= 1; // the fail list becomes the input, the old input buffer the new fail list
                const int nfc = fc == 8 ? 9 : 8;
                SR_CUDA(ctx, cudaMemsetAsync(cnt + nfc, 0, 8, ctx->stream));
                SR_TRY(final_pass(f->sel[cur].as<srd::SelEntry>(), cnt + fc, f->sel[cur ^ 1].as<srd::SelEntry>(), cnt + nfc));
                fc = nfc;
            }
        }
        return SR_OK;
    }
    const int grid = (int)std::min<int64_t>(f->grid, (n + srd::FRAG_TILE - 1) / srd::FRAG_TILE);
    if (f->smem_agg)
        srd::k_fragment<true><<<grid, srd::FRAG_BLOCK, f->smem_bytes, ctx->stream>>>((const srd::FragDev*)f->dev.p, (const srd::AggDev*)a->dev.p, vt, n,
                                                                                    f->queue_word_off);
    else
        srd::k_fragment<false><<<grid, srd::FRAG_BLOCK, f->smem_bytes, ctx->stream>>>((const srd::FragDev*)f->dev.p, (const srd::AggDev*)a->dev.p, vt, n,
                                                                                     f->queue_word_off);
    SR_LAUNCH_CHECK(ctx);
    if (hash) {
        uint64_t ng;
        int32_t ovf, bad;
        SR_TRY(agg_read_counters(a, &ng, &ovf, &bad));
        a->ngroups_host = (int64_t)ng;
        if (ovf) return sr_fail(ctx, SR_ERR_STATE, "aggregate hash table overflow (internal)");
    }
    return SR_OK;
}
