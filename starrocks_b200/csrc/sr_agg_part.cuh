// sr_agg_part.cuh -- radix-partitioned push of the hash aggregate (device side; included by sr_agg.cuh).
//
// Replaces, for large batches, the row-at-a-time lazy_emplace + update of
//   AggHashMap*::compute_agg_states            be/src/exec/aggregate/agg_hash_map.h:303-361
//   Aggregator::compute_batch_agg_states       be/src/exec/aggregator.cpp:1616-1640
// whose GPU transcription (k_agg_push) pays one L2 atomic transaction per row and state word (measured: 60-90 G
// atomics/s whatever the table size).  Here the batch is first moved next to the table slices it updates:
//
//   k_aggp_scatter   packed RECORDS (key, evaluated function inputs, null mask; W 8-byte words) are partitioned by the
//                    top bits of their home slot.  Inside a tile every row takes its rank in its bucket with one shared-memory
//                    atomic, the counters are scanned, the tile is copied out bucket by bucket
//                    into the buckets' regions (ONE global atomicAdd per tile and non-empty bucket reserves the run).
//                    Regions have a fixed capacity (mean + 6 sigma of a uniform hash); what does not fit goes to an
//                    overflow list -- no histogram pass.  Fan-out <= 2^9 per level, two levels for up to 2^18 buckets.
//   k_aggp_tiles     tile list of the second level from the first level's counts
//   k_aggp_apply     one CTA per bucket (a few 256-slot probing slices of the table, 48 KB of keys + states): the slices are
//                    loaded / initialised in shared memory, the bucket's records are applied with shared-memory atomics,
//                    the slices are written back with coalesced stores.
//   k_aggp_apply_l2  global-atomics apply for the overflow list, for slices that filled up, and for tables of more
//                    than 2^18 buckets (buckets of several CTA-loads: table range prefetched into L2, as in round 1).
#pragma once

namespace srd {

#ifndef SR_AGGP_BLOCK
#define SR_AGGP_BLOCK 512
#endif
constexpr int AGGP_BLOCK = SR_AGGP_BLOCK; // scatter CTA: 16 warps (tile of 4096 two-word records), two CTAs per SM
constexpr int AGGP_WARPS = AGGP_BLOCK / 32;
constexpr int AGGP_MAX_FAN_BITS = 9;     // fan-out of one scatter level
constexpr int AGGP_MAX_FAN = 1 << AGGP_MAX_FAN_BITS;
constexpr int AGGP_MAX_WORDS = 2 + SR_MAX_AGG_FNS + 1;
constexpr int AGGP_SLICE_LOG2 = 8;       // slots of one probing slice (owned by one warp in k_aggp_apply)
constexpr int AGGP_MAX_APPLY_SLICES = 8; // probing slices per bucket (one apply CTA loads a bucket's slices)

enum PartWordKind : int32_t { WK_KEY_LO = 0, WK_KEY_HI = 1, WK_VALUE = 2, WK_NULLS = 3 };

struct PartPlan {
    int32_t bits;         // log2(buckets)
    int32_t bits2;        // bits of the second scatter level (0: one level)
    int32_t bucket_shift; // bucket = (hash & mask) >> bucket_shift
    int32_t words;        // W: 8-byte words per record
    int32_t null_word;    // word holding the null mask (bit f: input of function f is NULL), -1: no input is nullable
    int32_t apply_slices; // probing slices per bucket (k_aggp_apply)
    int32_t word_kind[AGGP_MAX_WORDS];
    int32_t word_fn[AGGP_MAX_WORDS];
    int32_t val_word[SR_MAX_AGG_FNS]; // word of function f's input, -1 for COUNT(*)
    // SIMPLE plans (one non-nullable group-by column of <= 8 bytes, every function input a plain non-nullable column):
    // word 0 = the key column's value & simple_key_mask, word w = value id word_vid[w]; no expression interpreter
    int32_t simple;
    int32_t word_w8[4];        // SIMPLE: 1 = the word's column holds 8-byte values, 0 = 4-byte signed integers
    const void* word_ptr[4];   // SIMPLE: the word's column
    unsigned long long simple_key_mask;
    unsigned long long cap1, cap2; // records a first-level / final bucket region can take
};

// rows per thread and tile: 8 for records of <= 2 words (tile = 4096 rows = 64 KB), fewer for wider records
__host__ __device__ constexpr int aggp_rows_per_thread(int W) { return W <= 2 ? 8 : (W <= 4 ? 4 : (W <= 8 ? 2 : 1)); }

__device__ __forceinline__ uint32_t aggp_bucket(const AggDev& a, const PartPlan& pl, const HKey& key) {
    return (uint32_t)((hkey_hash(a, key) & a.mask) >> pl.bucket_shift);
}

// ---- scatter ----------------------------------------------------------------------------------------------------
struct ScatterArgs {
    int64_t row_base, n;                 // from a chunk: rows [row_base, row_base + n) of the bound chunk
    const unsigned long long* src;       // from records: the first level's regions
    const uint32_t* src_count;           //   records in every first-level region (may exceed cap1: capped)
    const uint32_t* tile_start;          //   first tile of every first-level bucket (+ total)
    uint32_t* cursor;                    // records reserved so far per destination bucket
    unsigned long long* dst;             // destination regions (bucket b at b * dst_cap records)
    unsigned long long dst_cap;
    unsigned long long* ovf;             // overflow list (records) + its counter
    unsigned long long* ovf_count;
    unsigned long long ovf_cap;
    int32_t fan_bits;                    // log2 of this level's fan-out
    int32_t local_shift;                 // local bucket = (bucket >> local_shift) & (fan - 1)
};

// ask L2 for the 128-byte lines of [p, p + bytes): one line per thread and step (sequential input only -- a prefetch
// fetches whole lines)
__device__ __forceinline__ void aggp_prefetch_l2(const void* p, size_t bytes, int tid, int nthreads) {
    const char* c = (const char*)((uintptr_t)p & ~(uintptr_t)127);
    const size_t lines = (((uintptr_t)p & 127) + bytes + 127) >> 7;
    for (size_t i = (size_t)tid; i < lines; i += (size_t)nthreads) asm volatile("prefetch.global.L2 [%0];" ::"l"(c + (i << 7)));
}

// general plans: build the record of `row` straight into shared memory (one out-of-line copy of the key packing and of the
// expression interpreter for all record widths); returns the row's bucket, or 0xFFFFFFFF when the packed key equals the
// table's empty marker -- such rows live in the special slot and are applied here, exactly once, never staged
__device__ __noinline__ uint32_t aggp_stage_row(const AggDev* ad, const PartPlan* plp, const VTab* vtp, int64_t row, unsigned long long* dst) {
    const AggDev& a = *ad;
    const PartPlan& pl = *plp;
    ChunkLoader ld{*vtp, row};
    HKey key;
    agg_pack_key(a, ld, key);
    if (hkey_is_empty(a, key)) {
        AccPtrs gp;
        acc_ptrs_global(a, gp);
        agg_apply_row<false>(a, gp, (long long)a.cap, ld);
        return 0xFFFFFFFFu;
    }
    unsigned long long nm = 0;
#pragma unroll 1
    for (int w = 0; w < pl.words; w++) {
        const int kind = pl.word_kind[w];
        if (kind == WK_KEY_LO) {
            dst[w] = key.lo;
        } else if (kind == WK_KEY_HI) {
            dst[w] = key.hi;
        } else if (kind == WK_NULLS) {
            dst[w] = nm; // the null word is the last one: every function has been evaluated
        } else {
            const int f = pl.word_fn[w];
            int64_t bits;
            const bool nul = eval_expr(a.fns[f].input, ld, bits);
            dst[w] = nul ? 0ull : (unsigned long long)bits;
            nm |= (nul ? 1ull : 0ull) << f;
        }
    }
    return aggp_bucket(a, pl, key);
}

template <int W>
__device__ __forceinline__ void aggp_load_record(const unsigned long long* __restrict__ p, unsigned long long (&rec)[W]) {
    if (W == 2) {
        const ulonglong2 v = __ldg((const ulonglong2*)p);
        rec[0] = v.x;
        rec[1] = v.y;
    } else {
#pragma unroll
        for (int w = 0; w < W; w++) rec[w] = __ldg(p + w);
    }
}
template <int W>
__device__ __forceinline__ void aggp_store_record(unsigned long long* p, const unsigned long long* s) {
    if (W == 2) {
        *(ulonglong2*)p = *(const ulonglong2*)s;
    } else {
#pragma unroll
        for (int w = 0; w < W; w++) p[w] = s[w];
    }
}

template <int W>
constexpr size_t aggp_scatter_smem() {
    // records + (perm, bucket) per position + warp counters / offsets + bucket start / run base
    return (size_t)AGGP_BLOCK * aggp_rows_per_thread(W) * (W * 8 + 4) + (size_t)AGGP_MAX_FAN * 4 + (size_t)(AGGP_MAX_FAN + 1) * 8 + 16;
}

enum ScatterMode { SCATTER_RECORDS = 0, SCATTER_CHUNK = 1, SCATTER_CHUNK_SIMPLE = 2 };

// One tile = T consecutive rows (first level: of the input chunk; second level: of one first-level region).  Warp w takes
// rows [w * 32 R, (w + 1) * 32 R) of the tile, 32 consecutive rows per step: the record goes to shared memory in row
// order, the row's rank inside (warp, bucket) comes from aggp_warp_rank.  After a barrier the (warp, bucket) counters are
// scanned into tile positions and every non-empty bucket reserves its run in the destination region; a second pass over
// the rows fills the inverse permutation; the copy-out walks the tile in bucket order: consecutive threads write
// consecutive records of a run.
template <int W, int MODE>
__global__ void __launch_bounds__(AGGP_BLOCK, 1024 / AGGP_BLOCK) k_aggp_scatter(const AggDev* __restrict__ ad, const __grid_constant__ VTab vt, const __grid_constant__ PartPlan pl,
                                                                 const __grid_constant__ ScatterArgs sa) {
    constexpr int R = aggp_rows_per_thread(W);
    constexpr int T = AGGP_BLOCK * R;
    constexpr int WR = 32 * R; // rows of one warp
    constexpr bool FROM_CHUNK = MODE != SCATTER_RECORDS;
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ uint32_t s_scan[AGGP_BLOCK / 32 + 1];
    unsigned long long* s_rec = (unsigned long long*)s_raw;                  // T records in row order
    uint32_t* s_start = (uint32_t*)(s_rec + (size_t)T * W);                   // first tile position of the bucket (+ total)
    uint32_t* s_gbase = s_start + AGGP_MAX_FAN + 1;                           // first record of the bucket's reserved run
    uint32_t* s_hist = s_gbase + AGGP_MAX_FAN + 1;                            // rows of the tile per bucket
    uint16_t* s_perm = (uint16_t*)(s_hist + AGGP_MAX_FAN);                    // tile position -> row of the tile
    uint16_t* s_bkt = s_perm + T;                                             // tile position -> bucket
    const AggDev& a = *ad;
    const int tid = threadIdx.x;
    const int wid = tid >> 5, lane = tid & 31;
    const int F = 1 << sa.fan_bits;
    const uint32_t fmask = (uint32_t)F - 1;
    for (int i = tid; i < F; i += AGGP_BLOCK) s_hist[i] = 0;
    const int64_t ntiles = FROM_CHUNK ? (sa.n + T - 1) / T : (int64_t)sa.tile_start[1 << (pl.bits - pl.bits2)];
    // first row / record of a tile, its length, and the destination bucket of its local bucket 0
    auto locate = [&](int64_t tile, int64_t& row0, int& tile_n, uint32_t& cbase) {
        cbase = 0;
        if (FROM_CHUNK) {
            row0 = tile * T;
            tile_n = (int)(sa.n - row0 < T ? sa.n - row0 : T);
        } else {
            // first-level bucket owning this tile: last entry of tile_start <= tile
            const int F1 = 1 << (pl.bits - pl.bits2);
            int lo = 0, hi = F1;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(sa.tile_start + mid) <= (uint32_t)tile) lo = mid; else hi = mid;
            }
            const unsigned long long cnt = min((unsigned long long)__ldg(sa.src_count + lo), pl.cap1);
            const int64_t off = (tile - (int64_t)__ldg(sa.tile_start + lo)) * T;
            row0 = (int64_t)((unsigned long long)lo * pl.cap1) + off;
            tile_n = (int)((int64_t)cnt - off < T ? (int64_t)cnt - off : T);
            cbase = (uint32_t)lo << pl.bits2;
        }
    };
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int64_t row0;
        int tile_n;
        uint32_t cbase;
        locate(tile, row0, tile_n, cbase);
        if (MODE == SCATTER_CHUNK_SIMPLE && tile + gridDim.x < ntiles) {
            // the input columns of the CTA's NEXT tile are requested into L2 while this tile is ranked, scanned and copied
            // out.  Measured per 1e9 rows against the same kernel without it: level 1 11.90 -> 11.47 ms.  The same
            // prefetch on the record tiles of level 2 and on the next bucket of the apply pass cost 0.5 ms each (8.09 ->
            // 8.65, 9.94 -> 10.40 ms: their input was written by the previous kernel and is largely L2-resident already,
            // the prefetch instructions only compete for issue slots) and is not done.
            int64_t nrow0;
            int ntile_n;
            uint32_t ncbase;
            locate(tile + gridDim.x, nrow0, ntile_n, ncbase);
#pragma unroll
            for (int w = 0; w < W; w++) {
                const int wb = pl.word_w8[w] ? 8 : 4;
                aggp_prefetch_l2((const char*)pl.word_ptr[w] + (size_t)(sa.row_base + nrow0) * wb, (size_t)ntile_n * wb, tid, AGGP_BLOCK);
            }
        }
        __syncthreads(); // s_hist is clear (initial clear, or the scan of the previous tile); s_rec / s_perm are free
        uint32_t lr[R];  // bucket << 16 | rank inside (warp, bucket); 0xFFFFFFFF: no record
        // first the loads of all R rows (issued back to back: the compiler does not move the volatile streaming loads
        // across the shared-memory stores of a fused loop, which left ONE load in flight per thread -- eight serial DRAM
        // latencies per tile), then the staging + bucket of every row, then the warp-synchronous ranking
        if (MODE == SCATTER_CHUNK) {
#pragma unroll
            for (int k = 0; k < R; k++) {
                const int q = wid * WR + k * 32 + lane;
                lr[k] = 0xFFFFFFFFu;
                if (q < tile_n) {
                    const uint32_t bk = aggp_stage_row(ad, &pl, &vt, sa.row_base + row0 + q, s_rec + (size_t)q * W);
                    if (bk != 0xFFFFFFFFu) lr[k] = (bk >> sa.local_shift) & fmask;
                }
            }
        } else {
            constexpr int G = R < 4 ? R : 4; // rows whose loads are in flight together (registers: G * W words)
            uint32_t special = 0;
#pragma unroll
            for (int k0 = 0; k0 < R; k0 += G) {
                unsigned long long rec[G][W];
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const int q = wid * WR + (k0 + g) * 32 + lane;
                    if (q < tile_n) {
                        if (MODE == SCATTER_CHUNK_SIMPLE) {
#pragma unroll
                            for (int w = 0; w < W; w++) {
                                if (pl.word_w8[w])
                                    rec[g][w] = (unsigned long long)ldg_stream_s64((const int64_t*)pl.word_ptr[w] + sa.row_base + row0 + q);
                                else
                                    rec[g][w] = (unsigned long long)(int64_t)ldg_stream_s32((const int32_t*)pl.word_ptr[w] + sa.row_base + row0 + q);
                            }
                        } else {
                            aggp_load_record<W>(sa.src + (size_t)(row0 + q) * W, rec[g]);
                        }
                    }
                }
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const int k = k0 + g;
                    const int q = wid * WR + k * 32 + lane;
                    lr[k] = 0xFFFFFFFFu;
                    if (q < tile_n) {
                        HKey key;
                        if (MODE == SCATTER_CHUNK_SIMPLE) rec[g][0] &= pl.simple_key_mask;
                        key.lo = rec[g][0];
                        key.hi = (MODE == SCATTER_RECORDS && a.wide) ? rec[g][W > 1 ? 1 : 0] : 0ull;
                        if (MODE == SCATTER_CHUNK_SIMPLE && key.lo == SR_AGG_EMPTY) {
                            special |= 1u << k; // the special slot's row: applied below (out of line), not staged
                        } else {
                            aggp_store_record<W>(s_rec + (size_t)q * W, rec[g]);
                            lr[k] = (aggp_bucket(a, pl, key) >> sa.local_shift) & fmask;
                        }
                    }
                }
            }
            if (MODE == SCATTER_CHUNK_SIMPLE && special) {
#pragma unroll 1
                for (int k = 0; k < R; k++)
                    if ((special >> k) & 1u) {
                        const int q = wid * WR + k * 32 + lane;
                        (void)aggp_stage_row(ad, &pl, &vt, sa.row_base + row0 + q, s_rec + (size_t)q * W);
                    }
            }
        }
        // rank inside (tile, bucket): one shared-memory atomic per row.  (Measured against a ballot-per-bit match with
        // warp-private counters, which needs no atomic: 14.4 / 11.1 ms vs 13.3 / 8.7 ms per 1e9 rows for the two levels.)
#pragma unroll
        for (int k = 0; k < R; k++)
            if (lr[k] != 0xFFFFFFFFu) lr[k] = lr[k] << 16 | atomicAdd(&s_hist[lr[k]], 1u);
        __syncthreads();
        {   // (warp, bucket) counters -> offsets; exclusive scan over the buckets; reserve the destination runs
            constexpr int PER = (AGGP_MAX_FAN + AGGP_BLOCK - 1) / AGGP_BLOCK; // buckets per thread (consecutive)
            uint32_t tot_l[PER];
            uint32_t mine = 0;
#pragma unroll
            for (int i = 0; i < PER; i++) {
                const int l = tid * PER + i;
                tot_l[i] = 0;
                if (l < F) {
                    tot_l[i] = s_hist[l];
                    s_hist[l] = 0; // the next tile's counter
                }
                mine += tot_l[i];
            }
            uint32_t tot;
            uint32_t run = block_excl_scan<AGGP_BLOCK>(mine, s_scan, &tot);
#pragma unroll
            for (int i = 0; i < PER; i++) {
                const int l = tid * PER + i;
                if (l < F) {
                    s_start[l] = run;
                    if (tot_l[i]) s_gbase[l] = atomicAdd(sa.cursor + cbase + l, tot_l[i]);
                    run += tot_l[i];
                }
            }
            if (tid == 0) s_start[F] = tot;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < R; k++) {
            if (lr[k] != 0xFFFFFFFFu) {
                const uint32_t l = lr[k] >> 16;
                const uint32_t pos = s_start[l] + (lr[k] & 0xFFFFu);
                s_perm[pos] = (uint16_t)(wid * WR + k * 32 + lane);
                s_bkt[pos] = (uint16_t)l;
            }
        }
        __syncthreads();
        const int staged = (int)s_start[F]; // records of the tile (rows of the special slot dropped out)
        for (int pos = tid; pos < staged; pos += AGGP_BLOCK) {
            const uint32_t l = s_bkt[pos];
            const unsigned long long d = (unsigned long long)s_gbase[l] + (unsigned long long)(pos - s_start[l]);
            const unsigned long long* src = s_rec + (size_t)s_perm[pos] * W;
            if (d < sa.dst_cap) {
                aggp_store_record<W>(sa.dst + ((unsigned long long)(cbase + l) * sa.dst_cap + d) * W, src);
            } else { // the bucket's region is full (skewed input): the record goes to the overflow list
                const unsigned long long o = atomicAdd(sa.ovf_count, 1ull);
                if (o < sa.ovf_cap) aggp_store_record<W>(sa.ovf + o * W, src);
            }
        }
    }
}

// first tile of every first-level region for the second level (one CTA)
__global__ void __launch_bounds__(1024) k_aggp_tiles(const uint32_t* __restrict__ count1, int f1, unsigned long long cap1, int tile_rows, uint32_t* __restrict__ tile_start) {
    __shared__ uint32_t s_scan[1024 / 32 + 1];
    const int i = threadIdx.x; // f1 <= 512
    uint32_t tiles = 0;
    if (i < f1) {
        const unsigned long long c = min((unsigned long long)count1[i], cap1);
        tiles = (uint32_t)((c + (unsigned long long)tile_rows - 1) / (unsigned long long)tile_rows);
    }
    uint32_t tot;
    const uint32_t ex = block_excl_scan<1024>(tiles, s_scan, &tot);
    if (i < f1) tile_start[i] = ex;
    if (i == 0) tile_start[f1] = tot;
}

// ---- apply ----------------------------------------------------------------------------------------------------------
// bytes of table state one group slot owns (keys + COUNT(*) + every accumulator array)
__host__ __device__ inline size_t agg_slot_bytes_of(const AggDev& h) {
    size_t b = 8 * (h.wide ? 2 : 1) + 8;
    for (int f = 0; f < h.num_fns; f++) {
        if (h.fns[f].mode == M_COUNT_STAR) continue;
        b += 8 + (h.fns[f].mode == M_SUM_I128 ? 8 : 0) + (h.fns[f].track_n ? 8 : 0);
    }
    return b;
}

// shared-memory image of a bucket's slices: [keys | cnt | per fn: acc0, acc1?, accn?], S slots each
__device__ __forceinline__ void aggp_slice_ptrs(const AggDev& a, unsigned char* smem, int S, unsigned long long*& keys, AccPtrs& p) {
    keys = (unsigned long long*)smem;
    long long* q = (long long*)(keys + (size_t)S * (a.wide ? 2 : 1));
    p.cnt = q;
    q += S;
    for (int f = 0; f < SR_MAX_AGG_FNS; f++) {
        p.acc0[f] = p.acc1[f] = p.accn[f] = nullptr;
        if (f < a.num_fns && a.fns[f].mode != M_COUNT_STAR) {
            p.acc0[f] = q;
            q += S;
            if (a.fns[f].mode == M_SUM_I128) {
                p.acc1[f] = q;
                q += S;
            }
            if (a.fns[f].track_n) {
                p.accn[f] = q;
                q += S;
            }
        }
    }
}

struct ApplyArgs {
    const unsigned long long* rec;  // final regions (bucket b at b * cap2 records)
    const uint32_t* count;          // records reserved per bucket (may exceed cap2: capped)
    uint32_t num_buckets;
    int32_t fresh; // the table holds no group yet: slices are initialised in shared memory instead of loaded
    uint32_t* fail_list;            // buckets with a slice that filled up (their records are re-applied by k_aggp_apply_l2)
    unsigned long long* fail_count;
};

struct ApplyFn {
    int32_t mode, val_word, track_n, fn;
};

// multi-word add into shared memory through native 32-bit atomics: every carry out of a word is seen by exactly one
// adder (atom returns the old value) and forwarded as a +1 to the next word.  Readers look at the words after a barrier.
__device__ __forceinline__ void smem_add_i128(long long* lo, long long* hi, long long v) {
    const uint32_t base_lo = (uint32_t)__cvta_generic_to_shared(lo), base_hi = (uint32_t)__cvta_generic_to_shared(hi);
    const uint32_t sign = v < 0 ? 0xFFFFFFFFu : 0u;
    const uint32_t w[4] = {(uint32_t)v, (uint32_t)((unsigned long long)v >> 32), sign, sign};
    uint32_t carry = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t addr = (i < 2 ? base_lo : base_hi) + 4u * (uint32_t)(i & 1);
        if (w[i] == 0xFFFFFFFFu && carry) continue; // + 2^32: the word is unchanged, the carry moves on
        const uint32_t add = w[i] + carry;
        carry = 0;
        if (add) {
            uint32_t old;
            asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(add) : "memory");
            carry = (old + add) < old ? 1u : 0u;
        }
    }
}
__device__ __forceinline__ void acc_apply_slice(int32_t mode, long long* a0, long long* a1, long long slot, long long bits) {
    if (mode == M_SUM_I128)
        smem_add_i128(a0 + slot, a1 + slot, bits);
    else
        acc_apply_shared(mode, a0, a1, slot, bits);
}

constexpr int AGGP_APPLY_BLOCK = 256;
// One CTA per bucket (= pl.apply_slices probing slices): the slices' key / state arrays are loaded into shared memory (or
// initialised there while the table is still empty), every thread takes records straight from the bucket's region: probe
// (64-bit / 128-bit CAS claims an empty slot), then shared-memory atomics on the state words (64-bit adds as 32-bit adds
// with carry); the slices are written back with coalesced stores.  48 KB of slices per CTA -> four CTAs per SM.
__global__ void __launch_bounds__(AGGP_APPLY_BLOCK, 4) k_aggp_apply(const AggDev* __restrict__ ad, const __grid_constant__ PartPlan pl, const __grid_constant__ ApplyArgs aa) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ AccPtrs sp;
    __shared__ ApplyFn s_fn[SR_MAX_AGG_FNS];
    __shared__ int s_nfn;
    __shared__ unsigned long long* s_keys_p;
    __shared__ int s_fail;
    __shared__ uint32_t s_new[AGGP_APPLY_BLOCK / 32];
    const AggDev& a = *ad;
    const int S = pl.apply_slices << AGGP_SLICE_LOG2;
    const int W = pl.words;
    const int tid = threadIdx.x;
    const int kw = a.wide ? 2 : 1;
    if (tid == 0) {
        unsigned long long* kp;
        AccPtrs t;
        aggp_slice_ptrs(a, s_raw, S, kp, t);
        sp = t;
        s_keys_p = kp;
        int n = 0;
        for (int f = 0; f < a.num_fns; f++)
            if (a.fns[f].mode != M_COUNT_STAR) s_fn[n++] = ApplyFn{a.fns[f].mode, pl.val_word[f], a.fns[f].track_n, f};
        s_nfn = n;
    }
    __syncthreads();
    unsigned long long* const s_keys = s_keys_p;
    const bool fast2 = W == 2 && !a.wide;
    const bool sumcount = fast2 && s_nfn == 1 && s_fn[0].mode == M_SUM_I64 && !s_fn[0].track_n && pl.null_word < 0;
    long long* const cnt_p = sp.cnt;
    long long* const sum_p = s_nfn > 0 ? sp.acc0[s_fn[0].fn] : nullptr;
    for (uint32_t b = blockIdx.x; b < aa.num_buckets; b += gridDim.x) {
        const int64_t nrec = (int64_t)min((unsigned long long)aa.count[b], pl.cap2);
        if (nrec <= 0) continue;
        const unsigned long long* const brec = aa.rec + (unsigned long long)b * pl.cap2 * W;
        const size_t g0 = (size_t)b * S;
        if (tid == 0) s_fail = 0;
        if (aa.fresh) {
            for (int i = tid; i < S * kw; i += AGGP_APPLY_BLOCK) s_keys[i] = SR_AGG_EMPTY;
            for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) {
                sp.cnt[i] = 0;
                for (int f = 0; f < a.num_fns; f++) {
                    if (sp.acc0[f]) sp.acc0[f][i] = acc_init_value(a.fns[f].mode);
                    if (sp.acc1[f]) sp.acc1[f][i] = 0;
                    if (sp.accn[f]) sp.accn[f][i] = 0;
                }
            }
        } else {
            for (int i = tid; i < S * kw; i += AGGP_APPLY_BLOCK) s_keys[i] = a.hkeys[g0 * kw + i];
            for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) sp.cnt[i] = a.cnt_star[g0 + i];
            for (int f = 0; f < a.num_fns; f++) {
                if (sp.acc0[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) sp.acc0[f][i] = a.fns[f].acc0[g0 + i];
                if (sp.acc1[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) sp.acc1[f][i] = a.fns[f].acc1[g0 + i];
                if (sp.accn[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) sp.accn[f][i] = a.fns[f].accn[g0 + i];
            }
        }
        __syncthreads();
        uint32_t my_new = 0;
        // (Measured and rejected: a special loop for the 8-byte-key COUNT + SUM shape with four record loads in flight per
        // thread and the probe on 32-bit shared addresses (ld.volatile.shared / atom.shared.cas): 9.9 -> 14.4 ms per 1e9 rows.
        // The four CTAs of an SM already overlap each other's load latency; the wider loop body only cost issue slots.)
        for (int64_t q = tid; q < nrec; q += AGGP_APPLY_BLOCK) {
            const unsigned long long* rp = brec + (size_t)q * W;
            HKey key;
            unsigned long long w1 = 0;
            if (fast2) {
                const ulonglong2 v = __ldg((const ulonglong2*)rp);
                key.lo = v.x;
                w1 = v.y;
                key.hi = 0;
            } else {
                key.lo = __ldg(rp);
                key.hi = a.wide ? __ldg(rp + 1) : 0ull;
            }
            const uint32_t home = (uint32_t)hkey_hash(a, key) & (uint32_t)(S - 1);
            const uint32_t sbase = home & ~((1u << AGGP_SLICE_LOG2) - 1);
            uint32_t s = home & ((1u << AGGP_SLICE_LOG2) - 1);
            int slot = -1;
            for (int tries = 0; tries < (1 << AGGP_SLICE_LOG2); tries++) {
                if (!a.wide) {
                    unsigned long long cur = *(volatile unsigned long long*)(s_keys + sbase + s);
                    if (cur == SR_AGG_EMPTY) {
                        cur = atomicCAS(s_keys + sbase + s, SR_AGG_EMPTY, key.lo);
                        if (cur == SR_AGG_EMPTY) {
                            my_new++;
                            cur = key.lo;
                        }
                    }
                    if (cur == key.lo) {
                        slot = (int)(sbase + s);
                        break;
                    }
                } else {
                    const uint32_t addr = (uint32_t)__cvta_generic_to_shared(s_keys + 2 * (sbase + s));
                    HKey cur;
                    asm volatile("ld.volatile.shared.v2.u64 {%0, %1}, [%2];" : "=l"(cur.lo), "=l"(cur.hi) : "r"(addr) : "memory");
                    if (cur.lo == SR_AGG_EMPTY && cur.hi == SR_AGG_EMPTY) {
                        asm volatile(
                                "{ .reg .b128 c, n, o;\n"
                                "  mov.b128 c, {%2, %3};\n"
                                "  mov.b128 n, {%4, %5};\n"
                                "  atom.shared.cas.b128 o, [%6], c, n;\n"
                                "  mov.b128 {%0, %1}, o; }"
                                : "=l"(cur.lo), "=l"(cur.hi)
                                : "l"(SR_AGG_EMPTY), "l"(SR_AGG_EMPTY), "l"(key.lo), "l"(key.hi), "r"(addr)
                                : "memory");
                        if (cur.lo == SR_AGG_EMPTY && cur.hi == SR_AGG_EMPTY) {
                            my_new++;
                            cur = key;
                        }
                    }
                    if (cur.lo == key.lo && cur.hi == key.hi) {
                        slot = (int)(sbase + s);
                        break;
                    }
                }
                s = (s + 1) & ((1u << AGGP_SLICE_LOG2) - 1);
            }
            if (slot < 0) {
                s_fail = 1;
                continue;
            }
            smem_add_u64(cnt_p + slot, 1ull);
            if (sumcount) {
                smem_add_u64(sum_p + slot, w1);
            } else {
                const unsigned long long nm = pl.null_word >= 0 ? __ldg(rp + pl.null_word) : 0ull;
#pragma unroll 1
                for (int i = 0; i < s_nfn; i++) {
                    const ApplyFn fn = s_fn[i];
                    if ((nm >> fn.fn) & 1ull) continue;
                    acc_apply_slice(fn.mode, sp.acc0[fn.fn], sp.acc1[fn.fn], slot, (long long)__ldg(rp + fn.val_word));
                    if (fn.track_n) smem_add_u64(sp.accn[fn.fn] + slot, 1ull);
                }
            }
        }
        __syncthreads();
        if (s_fail) {
            if (tid == 0) aa.fail_list[atomicAdd(aa.fail_count, 1ull)] = b;
        } else {
            for (int i = tid; i < S * kw; i += AGGP_APPLY_BLOCK) a.hkeys[g0 * kw + i] = s_keys[i];
            for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) a.cnt_star[g0 + i] = sp.cnt[i];
            for (int f = 0; f < a.num_fns; f++) {
                if (sp.acc0[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) a.fns[f].acc0[g0 + i] = sp.acc0[f][i];
                if (sp.acc1[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) a.fns[f].acc1[g0 + i] = sp.acc1[f][i];
                if (sp.accn[f])
                    for (int i = tid; i < S; i += AGGP_APPLY_BLOCK) a.fns[f].accn[g0 + i] = sp.accn[f][i];
            }
            const uint32_t wn = warp_sum(my_new);
            if ((tid & 31) == 0) s_new[tid >> 5] = wn;
            __syncthreads();
            if (tid == 0) {
                unsigned long long t = 0;
                for (int w = 0; w < AGGP_APPLY_BLOCK / 32; w++) t += s_new[w];
                if (t) atomicAdd(a.ngroups, t);
            }
        }
        __syncthreads();
    }
}

// ---- apply: global atomics on an L2-prefetched table range ----------------------------------------------------------
// records [r0, r1) of `rec`, or the records named by `list` (refused by the admission limit before a growth).
// [s_lo, s_hi): the slots the records map to, requested into L2 with full-line prefetches up front.
__global__ void __launch_bounds__(AGG_BLOCK) k_aggp_apply_l2(const AggDev* __restrict__ ad, const __grid_constant__ PartPlan pl, const unsigned long long* __restrict__ rec,
                                                              int64_t r0, int64_t r1, const uint64_t* __restrict__ list, unsigned long long s_lo, unsigned long long s_hi,
                                                              uint64_t* __restrict__ fail_list, unsigned long long* __restrict__ fail_count) {
    const AggDev& a = *ad;
    AccPtrs p;
    acc_ptrs_global(a, p);
    const int W = pl.words;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nth = (int64_t)gridDim.x * blockDim.x;
    if (s_hi > s_lo) {
        const unsigned long long lines = ((s_hi - s_lo) * 8 + 127) / 128; // 8-byte state words, 128-byte lines
        for (unsigned long long l = (unsigned long long)tid; l < lines; l += (unsigned long long)nth) {
            const unsigned long long w = s_lo + l * 16;
            if (a.wide) {
                prefetch_l2(a.hkeys + 2 * w);
                prefetch_l2(a.hkeys + 2 * w + 16);
            } else {
                prefetch_l2(a.hkeys + w);
            }
            prefetch_l2(p.cnt + w);
            for (int f = 0; f < a.num_fns; f++) {
                if (p.acc0[f]) prefetch_l2(p.acc0[f] + w);
                if (p.acc1[f]) prefetch_l2(p.acc1[f] + w);
                if (p.accn[f]) prefetch_l2(p.accn[f] + w);
            }
        }
    }
    unsigned long long known_groups = *(volatile unsigned long long*)a.ngroups;
    for (int64_t q = r0 + tid; q < r1; q += nth) {
        const int64_t i = list ? (int64_t)list[q] : q;
        const unsigned long long* rp = rec + (size_t)i * W;
        const HKey key{rp[0], a.wide ? rp[1] : 0ull};
        bool inserted;
        const long long slot = agg_find_slot_key(a, key, inserted, known_groups);
        agg_count_new_groups(a, inserted, known_groups);
        if (slot < 0) { // table / slice full: remember the record, the host grows the table and re-applies the list
            fail_list[atomicAdd(fail_count, 1ull)] = (uint64_t)i;
            continue;
        }
        atomicAdd((unsigned long long*)p.cnt + slot, 1ull);
        const unsigned long long nm = pl.null_word >= 0 ? rp[pl.null_word] : 0ull;
#pragma unroll 1
        for (int f = 0; f < a.num_fns; f++) {
            const AggFnDev& fn = a.fns[f];
            if (fn.mode == M_COUNT_STAR || ((nm >> f) & 1ull)) continue;
            acc_apply(fn.mode, p.acc0[f], p.acc1[f], slot, (long long)rp[pl.val_word[f]]);
            if (fn.track_n) atomicAdd((unsigned long long*)p.accn[f] + slot, 1ull);
        }
    }
}

} // namespace srd
