// sr_agg_part_host.cuh -- host side of the radix-partitioned aggregate push (kernels: sr_agg_part.cuh).
#pragma once

static const int64_t kPartitionedMinRows = 1 << 20;   // smaller batches take the direct (global atomics) push
static const int64_t kPartitionedMaxRows = 1ll << 30; // staged records per round
static const uint64_t kPartitionSliceBytes = 32ull << 20; // global-atomics mode: table bytes one bucket maps to

template <int W, int MODE>
static int32_t aggp_launch_scatter(sr_ctx* ctx, int grid, const srd::AggDev* dev, const VTab& vt, const srd::PartPlan& pl, const srd::ScatterArgs& sa) {
    const size_t smem = srd::aggp_scatter_smem<W>();
    SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_aggp_scatter<W, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, srd::k_aggp_scatter<W, MODE>, srd::AGGP_BLOCK, smem));
    grid = ctx->num_sms * std::max(occ, 1); // one wave of resident CTAs (persistent loop over the tiles)
    srd::k_aggp_scatter<W, MODE><<<grid, srd::AGGP_BLOCK, smem, ctx->stream>>>(dev, vt, pl, sa);
    SR_LAUNCH_CHECK(ctx);
    return SR_OK;
}

static int32_t aggp_scatter(sr_ctx* ctx, bool from_chunk, int grid, const srd::AggDev* dev, const VTab& vt, const srd::PartPlan& pl, const srd::ScatterArgs& sa) {
    if (from_chunk && pl.simple) {
        switch (pl.words) { // (plans of more than 4 words take the general kernel)
        case 1:
            return aggp_launch_scatter<1, srd::SCATTER_CHUNK_SIMPLE>(ctx, grid, dev, vt, pl, sa);
        case 2:
            return aggp_launch_scatter<2, srd::SCATTER_CHUNK_SIMPLE>(ctx, grid, dev, vt, pl, sa);
        case 3:
            return aggp_launch_scatter<3, srd::SCATTER_CHUNK_SIMPLE>(ctx, grid, dev, vt, pl, sa);
        case 4:
            return aggp_launch_scatter<4, srd::SCATTER_CHUNK_SIMPLE>(ctx, grid, dev, vt, pl, sa);
        default:
            break;
        }
    }
    switch (pl.words) {
#define SR_AGGP_CASE(W)                                                                                   \
    case W:                                                                                               \
        return from_chunk ? aggp_launch_scatter<W, srd::SCATTER_CHUNK>(ctx, grid, dev, vt, pl, sa)        \
                          : aggp_launch_scatter<W, srd::SCATTER_RECORDS>(ctx, grid, dev, vt, pl, sa);
        SR_AGGP_CASE(1)
        SR_AGGP_CASE(2)
        SR_AGGP_CASE(3)
        SR_AGGP_CASE(4)
        SR_AGGP_CASE(5)
        SR_AGGP_CASE(6)
        SR_AGGP_CASE(7)
        SR_AGGP_CASE(8)
        SR_AGGP_CASE(9)
        SR_AGGP_CASE(10)
        SR_AGGP_CASE(11)
#undef SR_AGGP_CASE
    default:
        return sr_fail(ctx, SR_ERR_NOT_SUPPORTED, "record of %d words", pl.words);
    }
}

// records a bucket region can take when `mean` are expected: + 6 sigma of a uniform hash (Poisson) + a constant, even
static uint64_t aggp_region_cap(double mean) {
    // (rows of one key hash alike, so the spread of a bucket's row count grows with the duplication factor: + 10 %)
    const uint64_t c = (uint64_t)(mean * 1.1 + 6.0 * sqrt(mean > 1.0 ? mean : 1.0) + 64.0) + 1;
    return (c + 1) & ~1ull;
}

// k_aggp_apply_l2 over records [r0, r1) of `rec` (or the fail list when list_n > 0), then -- while records are refused by the
// admission limit or a full slice -- grow the table and re-apply them.  Leaves ngroups_host current.
static int32_t aggp_apply_l2_drain(sr_agg* a, const srd::PartPlan& pl, const unsigned long long* rec, int64_t max_records) {
    sr_ctx* ctx = a->ctx;
    unsigned long long* fail_count = a->counters.as<unsigned long long>() + 4;
    while (true) {
        SR_CUDA(ctx, cudaMemcpyAsync(ctx->pinned + 8, a->counters.p, 48, cudaMemcpyDeviceToHost, ctx->stream));
        SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        a->ngroups_host = (int64_t)ctx->pinned[8];
        const uint64_t failed = ctx->pinned[8 + 4];
        if (failed == 0) break;
        if (a->host.cap >= (1ull << 33)) return sr_fail(ctx, SR_ERR_OUT_OF_MEMORY, "aggregate table would exceed 2^33 slots");
        SR_CUDA(ctx, cudaMemsetAsync((uint8_t*)a->counters.p + 8, 0, 8, ctx->stream)); // overflow / range flags
        SR_CUDA(ctx, cudaMemsetAsync(fail_count, 0, 8, ctx->stream));
        SR_TRY(agg_grow(a, a->host.cap * 2));
        SR_TRY(a->part_fail64b.reserve(ctx, sizeof(uint64_t) * (size_t)std::min<int64_t>((int64_t)failed, max_records)));
        const int agrid = std::min(grid_for((int64_t)failed, srd::AGG_BLOCK), ctx->num_sms * 8);
        srd::k_aggp_apply_l2<<<agrid, srd::AGG_BLOCK, 0, ctx->stream>>>((const srd::AggDev*)a->dev.p, pl, rec, 0, (int64_t)failed, a->part_fail64.as<uint64_t>(), 0, 0,
                                                                         a->part_fail64b.as<uint64_t>(), fail_count);
        SR_LAUNCH_CHECK(ctx);
        std::swap(a->part_fail64, a->part_fail64b);
    }
    return SR_OK;
}

// Rows [0, n) of the bound chunk: scatter the packed records by the top bits of their home slot (one or two levels), then
// apply them bucket by bucket.
static int32_t agg_push_partitioned(sr_agg* a, const VTab& vt, int64_t n, bool fresh) {
    sr_ctx* ctx = a->ctx;
    int64_t done = 0;
    const bool trace = getenv("SR_AGG_TRACE") != nullptr; // phase times (CUDA events) on stderr
    cudaEvent_t tev[4] = {nullptr, nullptr, nullptr, nullptr};
    if (trace)
        for (auto& e : tev) SR_CUDA(ctx, cudaEventCreate(&e));
    while (done < n) {
        const srd::AggDev& h = a->host;
        const int64_t m = std::min<int64_t>(n - done, kPartitionedMaxRows); // bounded by the staging buffers
        int log2cap = 0;
        while ((1ull << log2cap) < h.cap) log2cap++;
        srd::PartPlan pl;
        memset(&pl, 0, sizeof(pl));
        // record layout
        int w = 0;
        pl.word_kind[w++] = srd::WK_KEY_LO;
        if (h.wide) pl.word_kind[w++] = srd::WK_KEY_HI;
        bool any_nullable = false;
        for (int f = 0; f < h.num_fns; f++) {
            pl.val_word[f] = -1;
            const srd::AggFnDev& fn = h.fns[f];
            if (fn.mode == srd::M_COUNT_STAR) continue;
            pl.word_kind[w] = srd::WK_VALUE;
            pl.word_fn[w] = f;
            pl.val_word[f] = w++;
            for (int k = 0; k < fn.input.num_nodes; k++)
                if ((fn.input.nodes[k].op == srd::C_LOAD_I || fn.input.nodes[k].op == srd::C_LOAD_D) && vt.v[fn.input.nodes[k].arg].nulls) any_nullable = true;
        }
        pl.null_word = -1;
        if (any_nullable) {
            pl.word_kind[w] = srd::WK_NULLS;
            pl.null_word = w++;
        }
        pl.words = w;
        // SIMPLE plan?
        pl.simple = (h.num_keys == 1 && !h.wide && !h.key_nullable[0] && !any_nullable && w <= 4) ? 1 : 0;
        if (pl.simple) {
            const auto typed = [&](int w, int vid) { // 4-byte signed integers or raw 8-byte values only
                const int32_t t = vt.v[vid].type;
                const int tw = srd::type_width(t);
                if (vt.v[vid].nulls || (tw != 4 && tw != 8) || t == SR_TYPE_FLOAT) pl.simple = 0;
                pl.word_ptr[w] = vt.v[vid].data;
                pl.word_w8[w] = tw == 8 ? 1 : 0;
            };
            typed(0, h.key_value_id[0]);
            pl.simple_key_mask = h.key_width[0] == 8 ? ~0ull : ((1ull << (8 * h.key_width[0])) - 1);
            for (int f = 0; f < h.num_fns; f++) {
                if (pl.val_word[f] < 0) continue;
                if (h.fns[f].input.form != srd::F_COL)
                    pl.simple = 0;
                else
                    typed(pl.val_word[f], h.fns[f].input.nodes[0].arg);
            }
        }
        // bucket = the slices one apply CTA loads: as many (power of two, <= 8) as fit 48 KB (four CTAs per SM)
        const size_t slot_bytes = agg_slot_bytes(h);
        int nw = srd::AGGP_MAX_APPLY_SLICES;
        while (nw > 1 && ((size_t)nw << srd::AGGP_SLICE_LOG2) * slot_bytes > 48 * 1024) nw >>= 1;
        int log2nw = 0;
        while ((1 << log2nw) < nw) log2nw++;
        const size_t apply_smem = ((size_t)nw << srd::AGGP_SLICE_LOG2) * slot_bytes;
        const int bucket_log2 = srd::AGGP_SLICE_LOG2 + log2nw;
        const bool smem_mode = log2cap > bucket_log2 && log2cap - bucket_log2 <= 2 * srd::AGGP_MAX_FAN_BITS && apply_smem <= 200 * 1024 &&
                               h.slice_log2 == srd::AGGP_SLICE_LOG2 && !getenv("SR_AGG_PARTITION_FORCE_L2");
        pl.apply_slices = nw;
        if (smem_mode) {
            pl.bits = log2cap - bucket_log2;
            pl.bucket_shift = bucket_log2;
        } else {
            const uint64_t table_bytes = (h.cap + 1) * slot_bytes;
            int log2p = 1;
            while (log2p < srd::AGGP_MAX_FAN_BITS && (table_bytes >> log2p) > kPartitionSliceBytes) log2p++;
            if (log2p > log2cap) log2p = log2cap;
            pl.bits = log2p;
            pl.bucket_shift = log2cap - log2p;
        }
        pl.bits2 = pl.bits > srd::AGGP_MAX_FAN_BITS ? pl.bits / 2 : 0;
        const int P = 1 << pl.bits;
        const int F1 = 1 << (pl.bits - pl.bits2);
        pl.cap2 = aggp_region_cap((double)m / P);
        pl.cap1 = pl.bits2 ? aggp_region_cap((double)m / F1) : 0;
        const int tile_rows = srd::AGGP_BLOCK * srd::aggp_rows_per_thread(pl.words);
        const size_t rb = (size_t)pl.words * 8;
        SR_TRY(a->part_cursor.reserve(ctx, sizeof(uint32_t) * ((size_t)P + F1)));
        SR_TRY(a->part_tiles.reserve(ctx, sizeof(uint32_t) * ((size_t)F1 + 1)));
        SR_TRY(a->part_rec[0].reserve(ctx, (size_t)P * pl.cap2 * rb + 16));
        if (pl.bits2) SR_TRY(a->part_rec[1].reserve(ctx, (size_t)F1 * pl.cap1 * rb + 16));
        SR_TRY(a->part_ovf.reserve(ctx, (size_t)m * rb + 16));
        uint32_t* cursor = a->part_cursor.as<uint32_t>();
        uint32_t* cursor1 = cursor + P;
        unsigned long long* rec_final = a->part_rec[0].as<unsigned long long>();
        unsigned long long* rec_mid = pl.bits2 ? a->part_rec[1].as<unsigned long long>() : nullptr;
        unsigned long long* fail_count = a->counters.as<unsigned long long>() + 4;
        unsigned long long* ovf_count = a->counters.as<unsigned long long>() + 5;
        const srd::AggDev* dev = (const srd::AggDev*)a->dev.p;
        const int grid2 = ctx->num_sms * 2;
        if (trace) SR_CUDA(ctx, cudaEventRecord(tev[0], ctx->stream));
        SR_CUDA(ctx, cudaMemsetAsync(cursor, 0, sizeof(uint32_t) * ((size_t)P + F1), ctx->stream));
        SR_CUDA(ctx, cudaMemsetAsync(fail_count, 0, 16, ctx->stream));
        srd::ScatterArgs sa;
        memset(&sa, 0, sizeof(sa));
        sa.row_base = done;
        sa.n = m;
        sa.ovf = a->part_ovf.as<unsigned long long>();
        sa.ovf_count = ovf_count;
        sa.ovf_cap = (unsigned long long)m;
        if (pl.bits2 == 0) {
            sa.cursor = cursor;
            sa.dst = rec_final;
            sa.dst_cap = pl.cap2;
            sa.fan_bits = pl.bits;
            sa.local_shift = 0;
            SR_TRY(aggp_scatter(ctx, true, grid2, dev, vt, pl, sa));
            if (trace) SR_CUDA(ctx, cudaEventRecord(tev[1], ctx->stream));
        } else {
            sa.cursor = cursor1;
            sa.dst = rec_mid;
            sa.dst_cap = pl.cap1;
            sa.fan_bits = pl.bits - pl.bits2;
            sa.local_shift = pl.bits2;
            SR_TRY(aggp_scatter(ctx, true, grid2, dev, vt, pl, sa));
            if (trace) SR_CUDA(ctx, cudaEventRecord(tev[1], ctx->stream));
            srd::k_aggp_tiles<<<1, 1024, 0, ctx->stream>>>(cursor1, F1, pl.cap1, tile_rows, a->part_tiles.as<uint32_t>());
            SR_LAUNCH_CHECK(ctx);
            sa.src = rec_mid;
            sa.src_count = cursor1;
            sa.tile_start = a->part_tiles.as<uint32_t>();
            sa.cursor = cursor;
            sa.dst = rec_final;
            sa.dst_cap = pl.cap2;
            sa.fan_bits = pl.bits2;
            sa.local_shift = 0;
            SR_TRY(aggp_scatter(ctx, false, grid2, dev, vt, pl, sa));
        }
        if (trace) SR_CUDA(ctx, cudaEventRecord(tev[2], ctx->stream));
        uint64_t failed_buckets = 0, overflowed = 0;
        if (smem_mode) {
            SR_TRY(a->part_fail.reserve(ctx, sizeof(uint32_t) * (size_t)P));
            srd::ApplyArgs aa;
            aa.rec = rec_final;
            aa.count = cursor;
            aa.num_buckets = (uint32_t)P;
            aa.fresh = fresh ? 1 : 0;
            aa.fail_list = a->part_fail.as<uint32_t>();
            aa.fail_count = fail_count;
            SR_CUDA(ctx, cudaFuncSetAttribute(srd::k_aggp_apply, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)apply_smem));
            int occ = 1;
            SR_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, srd::k_aggp_apply, srd::AGGP_APPLY_BLOCK, apply_smem));
            srd::k_aggp_apply<<<std::min(P, ctx->num_sms * std::max(occ, 1)), srd::AGGP_APPLY_BLOCK, apply_smem, ctx->stream>>>(dev, pl, aa);
            SR_LAUNCH_CHECK(ctx);
        }
        fresh = false;
        if (trace) SR_CUDA(ctx, cudaEventRecord(tev[3], ctx->stream));
        SR_CUDA(ctx, cudaMemcpyAsync(ctx->pinned + 8, a->counters.p, 48, cudaMemcpyDeviceToHost, ctx->stream));
        SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        a->ngroups_host = (int64_t)ctx->pinned[8];
        failed_buckets = ctx->pinned[8 + 4];
        overflowed = std::min<uint64_t>(ctx->pinned[8 + 5], (uint64_t)m);
        if (trace) {
            float t[3];
            for (int k = 0; k < 3; k++) cudaEventElapsedTime(&t[k], tev[k], tev[k + 1]);
            fprintf(stderr, "[sr_agg partitioned push] rows %lld, %d-word records, 2^%d buckets (%d + %d bits) of %d slices, regions of %llu / %llu records: scatter %.3f ms, "
                            "scatter-2 %.3f ms, apply %.3f ms (%s), %llu buckets handed back, %llu records overflowed\n",
                    (long long)m, pl.words, pl.bits, pl.bits - pl.bits2, pl.bits2, nw, (unsigned long long)pl.cap1, (unsigned long long)pl.cap2, t[0], t[1], t[2],
                    smem_mode ? "shared-memory slices" : "global atomics follow", (unsigned long long)failed_buckets, (unsigned long long)overflowed);
        }
        SR_CUDA(ctx, cudaMemsetAsync(fail_count, 0, 8, ctx->stream));
        if (!smem_mode || failed_buckets > 0 || overflowed > 0) SR_TRY(a->part_fail64.reserve(ctx, sizeof(uint64_t) * (size_t)m));
        if (!smem_mode || failed_buckets > 0) {
            // global-atomics apply: every bucket, or the buckets with a slice that filled up (after a growth)
            std::vector<uint32_t> counts((size_t)P), todo;
            SR_CUDA(ctx, cudaMemcpyAsync(counts.data(), cursor, sizeof(uint32_t) * (size_t)P, cudaMemcpyDeviceToHost, ctx->stream));
            if (smem_mode) {
                todo.resize((size_t)failed_buckets);
                SR_CUDA(ctx, cudaMemcpyAsync(todo.data(), a->part_fail.p, sizeof(uint32_t) * (size_t)failed_buckets, cudaMemcpyDeviceToHost, ctx->stream));
            }
            SR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            if (smem_mode) {
                if (a->host.cap >= (1ull << 33)) return sr_fail(ctx, SR_ERR_OUT_OF_MEMORY, "aggregate table would exceed 2^33 slots");
                SR_TRY(agg_grow(a, a->host.cap * 2));
            } else {
                todo.resize((size_t)P);
                for (int b = 0; b < P; b++) todo[(size_t)b] = (uint32_t)b;
            }
            for (uint32_t b : todo) {
                const int64_t r0 = (int64_t)((uint64_t)b * pl.cap2), r1 = r0 + (int64_t)std::min<uint64_t>(counts[b], pl.cap2);
                if (r1 <= r0) continue;
                const int agrid = std::min(grid_for(r1 - r0, srd::AGG_BLOCK), ctx->num_sms * 8);
                // the slot range to prefetch is only known without a growth in between
                const unsigned long long s_lo = smem_mode ? 0ull : (unsigned long long)b << pl.bucket_shift;
                const unsigned long long s_hi = smem_mode ? 0ull : (unsigned long long)(b + 1) << pl.bucket_shift;
                srd::k_aggp_apply_l2<<<agrid, srd::AGG_BLOCK, 0, ctx->stream>>>((const srd::AggDev*)a->dev.p, pl, rec_final, r0, r1, nullptr, s_lo, s_hi,
                                                                                 a->part_fail64.as<uint64_t>(), fail_count);
                SR_LAUNCH_CHECK(ctx);
            }
            SR_TRY(aggp_apply_l2_drain(a, pl, rec_final, m));
        }
        if (overflowed > 0) { // records that found their bucket's region full (skewed input)
            const int agrid = std::min(grid_for((int64_t)overflowed, srd::AGG_BLOCK), ctx->num_sms * 8);
            srd::k_aggp_apply_l2<<<agrid, srd::AGG_BLOCK, 0, ctx->stream>>>((const srd::AggDev*)a->dev.p, pl, a->part_ovf.as<unsigned long long>(), 0, (int64_t)overflowed,
                                                                             nullptr, 0, 0, a->part_fail64.as<uint64_t>(), fail_count);
            SR_LAUNCH_CHECK(ctx);
            SR_TRY(aggp_apply_l2_drain(a, pl, a->part_ovf.as<unsigned long long>(), m));
        }
        // keep the load below the admission limit for the pushes that follow
        while ((uint64_t)a->ngroups_host > a->host.limit) {
            if (a->host.cap >= (1ull << 33)) return sr_fail(ctx, SR_ERR_OUT_OF_MEMORY, "aggregate table would exceed 2^33 slots");
            SR_TRY(agg_grow(a, a->host.cap * 2));
        }
        a->partitioned_pushes++;
        done += m;
    }
    if (trace)
        for (auto& e : tev) cudaEventDestroy(e);
    return SR_OK;
}
