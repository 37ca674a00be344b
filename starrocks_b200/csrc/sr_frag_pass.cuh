// sr_frag_pass.cuh -- the SELECTIVE mode of the fused fragment: a short pipeline of passes connected by
// device-resident selection vectors (the GPU form of the reference's Filter / selection vector,
// be/src/column/chunk.cpp:362 and storage late materialisation):
//
//   pass S  k_frag_stream       streams the scan-predicate columns and the key columns of the leading joins
//                               (128-bit loads, next tile prefetched), tests their bitmaps, appends the
//                               surviving row ids to a selection vector (warp-aggregated atomicAdd);
//   pass G  k_frag_gather_join  one per remaining selective join: lane-per-row gather of the key for the
//                               selected rows only (late materialisation at DRAM-sector granularity),
//                               bitmap / hash test, appends survivors to the next selection vector;
//   pass F  k_frag_gather_agg   remaining non-selective joins inline, build-row lookups, payload gathers,
//                               group slot, aggregate update in shared-memory accumulators.
//
// Every pass runs with full warps; the selection vectors are tiny next to the fact columns (4 B per
// surviving row), and no pass waits on the host: a pass reads its input length from the counter the
// previous pass bumped (same stream).  Row order inside a selection vector is not kept -- the consumer
// is an aggregate.
#pragma once

#include "sr_frag_kernel.cuh"

namespace srd {

// one test of the streaming pass in "fast" form (k_frag_stream_tests)
struct StreamTest {
    int32_t kind;     // 0: scan predicate as a range, lo <= v <= lo + span; 1: streamed join `join`
    int32_t value_id; // the int32-class column it reads
    int32_t join;
    uint32_t lo, span;
};
#define SR_MAX_STREAM_TESTS 6

struct PassDev {
    int32_t num_tests; // > 0: the streaming pass can run as k_frag_stream_tests (subject to the batch's nullability)
    int32_t num_vec;   // its first num_vec (1 or 2) tests read their column with prefetched 128-bit loads
    StreamTest tests[SR_MAX_STREAM_TESTS];
    int32_t num_stream_joins; // joins [0, num_stream_joins) are tested by the streaming pass
    int32_t final_first_join; // joins [final_first_join, S) are tested inline by the final pass
    // the int32 key of one streamed join whose build row the final pass needs travels in the upper half of the
    // selection-vector entries, so the final pass does not gather it from the fact table again
    int8_t carry_join;     // index of that join among the streamed joins, -1 = none
    int8_t carry_value_id; // its key's value id
    int8_t pad[2];
};

// selection-vector entry: row id (low 32 bits) + carried key (high 32 bits)
typedef unsigned long long SelEntry;
__device__ __forceinline__ uint32_t sel_row(SelEntry e) { return (uint32_t)e; }
__device__ __forceinline__ int32_t sel_carry(SelEntry e) { return (int32_t)(e >> 32); }
__device__ __forceinline__ SelEntry sel_make(uint32_t row, int32_t carry) { return (SelEntry)row | ((SelEntry)(uint32_t)carry << 32); }

// bitmap / hash test against the global copies only (gather passes do not stage bitmaps)
__device__ __forceinline__ bool join_hit_global(const FragJoinDev& fj, int64_t key) {
    if (fj.use_bitmap) {
        if (key < fj.j.min_value || key > fj.j.max_value) return false;
        const uint64_t idx = (uint64_t)(key - fj.j.min_value);
        return (__ldg(fj.j.bitmap + (idx >> 5)) >> (idx & 31)) & 1u;
    }
    return join_lookup(fj.j, key) != 0;
}

// bitmap word of a row that is still alive (alive_bit != 0) and whose index lies in the table's range; 0 otherwise.  The
// predicate is formed inside the asm block from the raw operands: handing a C++ bool in costs a select to 0 / 1 and a
// compare back (ncu: 6.6 instructions per row on this line of the issue-bound streaming pass)
__device__ __forceinline__ uint32_t ldg_bitmap_word(const uint32_t* bm, uint32_t idx, uint32_t span, uint32_t alive_bit) {
    uint32_t r;
    asm volatile(
            "{ .reg .pred q;\n"
            "  setp.le.u32 q, %2, %3;\n"
            "  setp.ne.and.u32 q, %4, 0, q;\n"
            "  mov.u32 %0, 0;\n"
            "  @q ld.global.nc.u32 %0, [%1]; }"
            : "=r"(r)
            : "l"(bm + (idx >> 5)), "r"(idx), "r"(span), "r"(alive_bit));
    return r;
}

__device__ __forceinline__ uint32_t ldg_u32_pred(const uint32_t* p, bool pred) {
    uint32_t r;
    asm volatile(
            "{ .reg .pred q; setp.ne.u32 q, %2, 0; mov.u32 %0, 0;\n"
            "  @q ld.global.nc.u32 %0, [%1]; }"
            : "=r"(r)
            : "l"(p), "r"((uint32_t)pred));
    return r;
}

// Test N keys (bit i of `alive` says whether key i is still wanted) against one join and clear the bits of
// the misses.  For bitmap joins the N word fetches are issued back to back (predicated, branch-free) so a
// thread pays one L2 round trip for its whole group instead of one per row.
template <int N, typename K>
__device__ __forceinline__ uint32_t join_test_batch(const FragJoinDev& fj, const uint32_t* smem, const K (&keys)[N], uint32_t alive) {
    if (sizeof(K) == 4 && fj.use_bitmap && fj.idx32) {
        // int32 keys against a table whose [min, max] fits int32: one unsigned subtract + compare does the
        // range check, and the whole test stays in 32-bit arithmetic (the stream kernel is issue bound)
        const uint32_t umin = (uint32_t)(int32_t)fj.j.min_value;
        const uint32_t span = (uint32_t)(fj.j.max_value - fj.j.min_value);
        uint32_t out = 0;
        if (fj.smem_off >= 0) {
            const uint32_t* bm = smem + fj.smem_off;
#pragma unroll
            for (int i = 0; i < N; i++) {
                const uint32_t idx = (uint32_t)keys[i] - umin;
                const bool p = ((alive >> i) & 1u) && idx <= span;
                const uint32_t word = p ? bm[idx >> 5] : 0u;
                // rotate bit (idx mod 32) of the word to position i, then one 3-input logic op merges it into `out`
                out |= __funnelshift_r(word, word, idx - (uint32_t)i) & (1u << i);
            }
        } else {
            uint32_t words[N];
#pragma unroll
            for (int i = 0; i < N; i++) {
                const uint32_t idx = (uint32_t)keys[i] - umin;
                const bool p = ((alive >> i) & 1u) && idx <= span;
                words[i] = ldg_u32_pred(fj.j.bitmap + (idx >> 5), p);
            }
#pragma unroll
            for (int i = 0; i < N; i++) {
                const uint32_t idx = (uint32_t)keys[i] - umin;
                out |= __funnelshift_r(words[i], words[i], idx - (uint32_t)i) & (1u << i);
            }
        }
        return out;
    }
    if (fj.use_bitmap) {
        const int64_t mn = fj.j.min_value, mx = fj.j.max_value;
        uint32_t words[N];
        uint32_t want = 0;
#pragma unroll
        for (int i = 0; i < N; i++) {
            const bool p = ((alive >> i) & 1u) && keys[i] >= mn && keys[i] <= mx;
            const uint64_t idx = (uint64_t)(keys[i] - mn);
            want |= (p ? 1u : 0u) << i;
            if (fj.smem_off >= 0)
                words[i] = p ? smem[fj.smem_off + (idx >> 5)] : 0u;
            else
                words[i] = ldg_u32_pred(fj.j.bitmap + (idx >> 5), p);
        }
        uint32_t out = 0;
#pragma unroll
        for (int i = 0; i < N; i++) {
            const uint64_t idx = (uint64_t)(keys[i] - mn);
            out |= (((want >> i) & 1u) & (words[i] >> (idx & 31))) << i;
        }
        return out;
    }
    uint32_t out = alive;
#pragma unroll
    for (int i = 0; i < N; i++)
        if (((alive >> i) & 1u) && join_lookup(fj.j, keys[i]) == 0) out &= ~(1u << i);
    return out;
}

constexpr int STREAM_BLOCK = 512;
constexpr int STREAM_ROWS = 4;
constexpr int STREAM_GROUPS = 2;
constexpr int STREAM_TILE = STREAM_BLOCK * STREAM_ROWS * STREAM_GROUPS;
constexpr int STREAM_MAX_JOINS = 2;

// Selection vectors are written through a per-warp chunk allocator: a warp takes SEL_CHUNK entries at a
// time from the global counter (one same-address atomic per ~SEL_CHUNK survivors instead of one per
// tile -- same-address atomics serialise in L2) and pads what it leaves unused with SEL_INVALID, which
// the consuming pass skips.  The counter therefore counts allocated entries, valid or not.
#define SEL_INVALID 0xFFFFFFFFu
constexpr uint32_t SEL_CHUNK = 256;

struct WarpSelWriter {
    SelEntry* __restrict__ out;
    unsigned long long* __restrict__ counter;
    unsigned long long pos, end; // warp-uniform
    __device__ __forceinline__ void init(SelEntry* o, unsigned long long* c) {
        out = o;
        counter = c;
        pos = end = 0;
    }
    // reserve `total` (<= SEL_CHUNK, warp-uniform) entries, returns the start index
    __device__ __forceinline__ unsigned long long reserve(uint32_t total) {
        if (pos + total > end) {
            for (unsigned long long i = pos + lane_id(); i < end; i += 32) out[i] = SEL_INVALID;
            unsigned long long base = 0;
            if (lane_id() == 0) base = atomicAdd(counter, (unsigned long long)SEL_CHUNK);
            pos = __shfl_sync(SR_FULL_MASK, base, 0);
            end = pos + SEL_CHUNK;
        }
        const unsigned long long p = pos;
        pos += total;
        return p;
    }
    __device__ __forceinline__ void finish() {
        for (unsigned long long i = pos + lane_id(); i < end; i += 32) out[i] = SEL_INVALID;
        pos = end;
    }
};

// append the rows flagged in `alive` (bit i -> row base_i + (i & 3)) with their carried keys to the selection vector
template <bool CARRY>
__device__ __forceinline__ void warp_append_rows(uint32_t alive_all, int64_t row0_g0, int64_t row0_g1,
                                                 const int32_t (&carry)[STREAM_GROUPS * STREAM_ROWS], WarpSelWriter& w) {
    const uint32_t cnt = __popc(alive_all);
    const uint32_t incl = warp_incl_scan(cnt);
    const uint32_t total = __shfl_sync(SR_FULL_MASK, incl, 31);
    if (total == 0) return;
    SelEntry* __restrict__ sel_out = w.out + (w.reserve(total) + incl - cnt);
    if (CARRY) {
        uint32_t pos = 0;
#pragma unroll
        for (int i = 0; i < STREAM_GROUPS * STREAM_ROWS; i++) {
            if ((alive_all >> i) & 1u) {
                const int64_t row = (i < STREAM_ROWS ? row0_g0 : row0_g1) + (i & (STREAM_ROWS - 1));
                sel_out[pos++] = sel_make((uint32_t)row, carry[i]);
            }
        }
    } else {
        // few rows survive (a lane holds 0..2 of its 8): walk the set bits instead of testing all eight
        const uint32_t r0 = (uint32_t)row0_g0, r1 = (uint32_t)row0_g1 - STREAM_ROWS;
        uint32_t m = alive_all, pos = 0;
        while (m) {
            const uint32_t i = (uint32_t)__ffs((int)m) - 1u;
            m &= m - 1u;
            sel_out[pos++] = (SelEntry)((i < STREAM_ROWS ? r0 : r1) + i);
        }
    }
}

// prologue of both streaming kernels: the descriptors of the streamed joins [0, SJ) into s_joins, and their shared-memory
// bitmaps into smem, each followed by the zero guard word that frag_plan reserves behind it (stream_test_reg kind 1)
__device__ __forceinline__ void stream_stage_joins(const FragDev& fd, int SJ, FragJoinDev* s_joins, uint32_t* smem) {
    for (int i = threadIdx.x; i < (int)(sizeof(FragJoinDev) / 4) * SJ; i += blockDim.x) ((uint32_t*)s_joins)[i] = ((const uint32_t*)fd.joins)[i];
    for (int j = 0; j < SJ; j++) {
        const FragJoinDev& fj = fd.joins[j];
        if (fj.smem_off >= 0)
            for (int w = threadIdx.x; w <= fj.bitmap_words; w += blockDim.x) smem[fj.smem_off + w] = w < fj.bitmap_words ? fj.j.bitmap[w] : 0u;
    }
}

// Each CTA streams a CONTIGUOUS run of tiles [begin, end) (not a grid-stride walk): the rows a warp appends to one
// selection-vector chunk then come from a narrow band of the table (~25 tiles) instead of being spread over the whole
// batch, so the later gather passes touch neighbouring sectors / pages back to back.
__device__ __forceinline__ void stream_tile_range(int64_t n, int64_t& begin, int64_t& end) {
    const int64_t num_tiles = (n + STREAM_TILE - 1) / STREAM_TILE;
    const int64_t tiles_per_cta = (num_tiles + gridDim.x - 1) / gridDim.x;
    begin = (int64_t)blockIdx.x * tiles_per_cta;
    end = begin + tiles_per_cta < num_tiles ? begin + tiles_per_cta : num_tiles;
}

// CARRY: the key of streamed join pd.carry_join rides in the upper half of the entries.  Only instantiated for
// host-resident input: holding the tile's keys in registers through the append costs the streaming kernel ~25 %
// when it runs at HBM speed (register spills; re-reading the key for the survivors instead was worse still, it puts
// an L2 round trip on every tile's critical path) but nothing when the kernel waits on PCIe, and there every sector
// the final pass does not have to fetch is worth ~2.5 ns of bus time.
template <bool CARRY>
__global__ void __launch_bounds__(STREAM_BLOCK, 2) k_frag_stream(const FragDev* __restrict__ fdp, PassDev pd, const __grid_constant__ VTab vt, int64_t n,
                                                                 SelEntry* __restrict__ sel_out, unsigned long long* __restrict__ counter) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ FragJoinDev s_joins[STREAM_MAX_JOINS];
    __shared__ CPred s_preds[8];
    const FragDev& fd = *fdp;
    const int SJ = pd.num_stream_joins;
    stream_stage_joins(fd, SJ, s_joins, smem);
    for (int i = threadIdx.x; i < (int)(sizeof(CPred) / 4) * fd.num_preds; i += blockDim.x) ((uint32_t*)s_preds)[i] = ((const uint32_t*)fd.preds)[i];
    __syncthreads();

    // (the common shapes -- range conjuncts and joins on plain int32 columns -- run in k_frag_stream_tests below;
    // this kernel is the general form: any predicate, generic filter expressions, nullable / wide key columns)
    const int64_t full_tiles = n / STREAM_TILE;
    int64_t tile_begin, tile_end;
    stream_tile_range(n, tile_begin, tile_end);
    WarpSelWriter writer;
    writer.init(sel_out, counter);

    for (int64_t tile = tile_begin; tile < tile_end; tile++) {
        int64_t row0[STREAM_GROUPS];
        uint32_t alive[STREAM_GROUPS];
#pragma unroll
        for (int g = 0; g < STREAM_GROUPS; g++) {
            row0[g] = tile * STREAM_TILE + (int64_t)g * (STREAM_BLOCK * STREAM_ROWS) + (int64_t)threadIdx.x * STREAM_ROWS;
            alive[g] = 0xFu;
        }
        if (tile >= full_tiles) { // only the last tile can be ragged
#pragma unroll
            for (int g = 0; g < STREAM_GROUPS; g++) {
                alive[g] = 0;
#pragma unroll
                for (int r = 0; r < STREAM_ROWS; r++)
                    if (row0[g] + r < n) alive[g] |= 1u << r;
            }
        }
        int32_t carry[STREAM_GROUPS * STREAM_ROWS];
        if (CARRY) {
#pragma unroll
            for (int i = 0; i < STREAM_GROUPS * STREAM_ROWS; i++) carry[i] = 0;
        }
        {
            int64_t vals[STREAM_GROUPS][STREAM_ROWS];
            uint32_t nullmask[STREAM_GROUPS];
#pragma unroll 1
            for (int p = 0; p < fd.num_preds; p++) {
                const VDesc& d = vt.v[s_preds[p].value_id];
#pragma unroll
                for (int g = 0; g < STREAM_GROUPS; g++) load_rows4(d, row0[g], alive[g], vals[g], nullmask[g]);
#pragma unroll
                for (int g = 0; g < STREAM_GROUPS; g++)
#pragma unroll
                    for (int r = 0; r < STREAM_ROWS; r++)
                        if ((alive[g] & (1u << r)) && !eval_pred(s_preds[p], vals[g][r], (nullmask[g] >> r) & 1u)) alive[g] &= ~(1u << r);
            }
#pragma unroll 1
            for (int e = 0; e < fd.num_exprs; e++) {
#pragma unroll 1
                for (int g = 0; g < STREAM_GROUPS; g++)
#pragma unroll 1
                    for (int r = 0; r < STREAM_ROWS; r++) {
                        if (alive[g] & (1u << r)) {
                            ChunkLoader ld{vt, row0[g] + r};
                            int64_t bits;
                            const bool nul = eval_expr(fd.exprs[e], ld, bits);
                            if (nul || bits == 0) alive[g] &= ~(1u << r);
                        }
                    }
            }
#pragma unroll 1
            for (int j = 0; j < SJ; j++) {
                const VDesc& d = vt.v[s_joins[j].key_value_id];
#pragma unroll
                for (int g = 0; g < STREAM_GROUPS; g++) load_rows4(d, row0[g], alive[g], vals[g], nullmask[g]);
#pragma unroll
                for (int g = 0; g < STREAM_GROUPS; g++) {
                    alive[g] &= ~nullmask[g]; // NULL keys never match (join_hash_table.cpp:166-170)
#pragma unroll
                    for (int r = 0; r < STREAM_ROWS; r++)
                        if ((alive[g] & (1u << r)) && !frag_join_hit(s_joins[j], smem, vals[g][r])) alive[g] &= ~(1u << r);
                }
                if (CARRY && j == pd.carry_join) {
#pragma unroll
                    for (int g = 0; g < STREAM_GROUPS; g++)
#pragma unroll
                        for (int r = 0; r < STREAM_ROWS; r++) carry[g * STREAM_ROWS + r] = (int32_t)vals[g][r];
                }
            }
        }
        static_assert(STREAM_GROUPS == 2, "two groups of alive bits are packed into one word");
        warp_append_rows<CARRY>(alive[0] | (alive[1] << STREAM_ROWS), row0[0], row0[1], carry, writer);
    }
    writer.finish();
}

// Streaming pass over a list of TESTS (PassDev::tests): scan predicates in range form (lo <= v <= lo + span on an
// int32-class column: EQ / LT / LE / GT / GE / BETWEEN all reduce to one unsigned subtract + compare) followed by the
// streamed joins.  The columns of the first one or two tests are read with 128-bit loads prefetched a tile ahead (most
// of their sectors are needed anyway); every later test loads its column only for the rows still alive (predicated
// loads, issued back to back).  The host picks this kernel when every test column is int32-class and not nullable
// (frag_push); anything else takes the generic path of k_frag_stream.
template <int N>
__device__ __forceinline__ uint32_t stream_test(const StreamTest& st, const FragJoinDev* s_joins, const uint32_t* smem, const int32_t (&k)[N], uint32_t alive) {
    if (st.kind == 0) {
        uint32_t out = 0;
#pragma unroll
        for (int i = 0; i < N; i++) out |= ((uint32_t)k[i] - st.lo <= st.span ? 1u : 0u) << i;
        return out & alive;
    }
    return join_test_batch<N>(s_joins[st.join], smem, k, alive);
}

// The two vector-column tests of k_frag_stream_tests with their parameters held in REGISTERS for the whole kernel.  ncu
// (profiles/r2_notes.md) showed that kernel issue bound at 47.8 instructions per row, 6.4 of them re-reading the
// warp-uniform test descriptors from shared memory on every call (the compiler cannot hoist them over the selection-vector
// stores) and 13.5 in the shared-memory bitmap test.  kind: 0 = range conjunct, 1 = bitmap in shared memory (int32 index
// arithmetic, zero GUARD bit at index span + 1: an out-of-range key is clamped onto it, so the test needs neither a
// predicate nor a select), 2 = bitmap in global memory (predicated word fetches, issued back to back), 3 = anything else
// (falls back to stream_test).
struct TestReg {
    uint32_t kind;
    uint32_t lo, span;
    const uint32_t* bm;
};

__device__ __forceinline__ TestReg make_test_reg(const StreamTest& st, const FragJoinDev* s_joins, const uint32_t* smem) {
    TestReg t;
    t.kind = 3;
    t.lo = st.lo;
    t.span = st.span;
    t.bm = nullptr;
    if (st.kind == 0) {
        t.kind = 0;
    } else {
        const FragJoinDev& fj = s_joins[st.join];
        if (fj.use_bitmap && fj.idx32) {
            t.lo = (uint32_t)(int32_t)fj.j.min_value;
            t.span = (uint32_t)(fj.j.max_value - fj.j.min_value);
            if (fj.smem_off >= 0 && t.span != 0xFFFFFFFFu) {
                t.kind = 1;
                t.bm = smem + fj.smem_off;
            } else {
                t.kind = 2;
                t.bm = fj.j.bitmap;
            }
        }
    }
    return t;
}

template <int N>
__device__ __forceinline__ uint32_t stream_test_reg(const TestReg& t, const StreamTest& st, const FragJoinDev* s_joins, const uint32_t* smem,
                                                    const int32_t (&k)[N], uint32_t alive) {
    uint32_t out = 0;
    if (t.kind == 1) {
        const uint32_t guard = t.span + 1u;
#pragma unroll
        for (int i = 0; i < N; i++) {
            const uint32_t idx = min((uint32_t)k[i] - t.lo, guard);
            const uint32_t word = t.bm[idx >> 5];
            out |= __funnelshift_r(word, word, idx - (uint32_t)i) & (1u << i);
        }
        return out & alive;
    }
    if (t.kind == 2) {
        uint32_t words[N];
#pragma unroll
        for (int i = 0; i < N; i++) {
            const uint32_t idx = (uint32_t)k[i] - t.lo;
            words[i] = ldg_bitmap_word(t.bm, idx, t.span, alive & (1u << i));
        }
#pragma unroll
        for (int i = 0; i < N; i++) {
            const uint32_t idx = (uint32_t)k[i] - t.lo;
            out |= __funnelshift_r(words[i], words[i], idx - (uint32_t)i) & (1u << i);
        }
        return out;
    }
    if (t.kind == 0) {
#pragma unroll
        for (int i = 0; i < N; i++) out |= ((uint32_t)k[i] - t.lo <= t.span ? 1u : 0u) << i;
        return out & alive;
    }
    return stream_test<N>(st, s_joins, smem, k, alive);
}

template <bool CARRY>
__global__ void __launch_bounds__(STREAM_BLOCK, 2) k_frag_stream_tests(const FragDev* __restrict__ fdp, PassDev pd, const __grid_constant__ VTab vt, int64_t n,
                                                                       SelEntry* __restrict__ sel_out, unsigned long long* __restrict__ counter) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ FragJoinDev s_joins[STREAM_MAX_JOINS];
    __shared__ StreamTest s_tests[SR_MAX_STREAM_TESTS];
    const FragDev& fd = *fdp;
    const int SJ = pd.num_stream_joins;
    const int NT = pd.num_tests;
    const int NV = pd.num_vec;
    stream_stage_joins(fd, SJ, s_joins, smem);
    for (int i = threadIdx.x; i < (int)(sizeof(StreamTest) / 4) * NT; i += blockDim.x) ((uint32_t*)s_tests)[i] = ((const uint32_t*)pd.tests)[i];
    __syncthreads();
    const TestReg t0 = make_test_reg(s_tests[0], s_joins, smem);
    const TestReg t1 = make_test_reg(s_tests[NV > 1 ? 1 : 0], s_joins, smem);
    const bool carry0 = CARRY && s_tests[0].kind == 1 && s_tests[0].join == pd.carry_join;
    const bool carry1 = CARRY && NV > 1 && s_tests[1].kind == 1 && s_tests[1].join == pd.carry_join;
    const int32_t* col0 = (const int32_t*)vt.v[pd.tests[0].value_id].data;
    const int32_t* col1 = NV > 1 ? (const int32_t*)vt.v[pd.tests[1].value_id].data : nullptr;
    const int64_t full_tiles = n / STREAM_TILE;
    int64_t tile_begin, tile_end;
    stream_tile_range(n, tile_begin, tile_end);
    const int64_t prefetch_end = tile_end < full_tiles ? tile_end : full_tiles;
    int4 pk[2][STREAM_GROUPS];
#pragma unroll
    for (int j = 0; j < 2; j++)
#pragma unroll
        for (int g = 0; g < STREAM_GROUPS; g++) pk[j][g] = make_int4(0, 0, 0, 0);
    auto prefetch = [&](int64_t tile) {
        if (tile < prefetch_end) {
#pragma unroll
            for (int g = 0; g < STREAM_GROUPS; g++) {
                const int64_t r0 = tile * STREAM_TILE + (int64_t)g * (STREAM_BLOCK * STREAM_ROWS) + (int64_t)threadIdx.x * STREAM_ROWS;
                pk[0][g] = ldg_stream_v4(col0 + r0);
                if (col1) pk[1][g] = ldg_stream_v4(col1 + r0);
            }
        }
    };
    prefetch(tile_begin);
    WarpSelWriter writer;
    writer.init(sel_out, counter);
    static_assert(STREAM_GROUPS == 2 && STREAM_ROWS == 4, "8 rows per thread and tile");
    for (int64_t tile = tile_begin; tile < tile_end; tile++) {
        int64_t row0[STREAM_GROUPS];
#pragma unroll
        for (int g = 0; g < STREAM_GROUPS; g++)
            row0[g] = tile * STREAM_TILE + (int64_t)g * (STREAM_BLOCK * STREAM_ROWS) + (int64_t)threadIdx.x * STREAM_ROWS;
        int32_t carry[8];
        if (CARRY) {
#pragma unroll
            for (int i = 0; i < 8; i++) carry[i] = 0;
        }
        uint32_t a8 = 0xFFu;
        int first_pred = 0; // tests [first_pred, NT) load their column for the live rows only
        if (tile < full_tiles) {
            const int32_t k0[8] = {pk[0][0].x, pk[0][0].y, pk[0][0].z, pk[0][0].w, pk[0][1].x, pk[0][1].y, pk[0][1].z, pk[0][1].w};
            const int32_t k1[8] = {pk[1][0].x, pk[1][0].y, pk[1][0].z, pk[1][0].w, pk[1][1].x, pk[1][1].y, pk[1][1].z, pk[1][1].w};
            prefetch(tile + 1); // the next tile's vector columns stay in flight while this tile is tested
            a8 = stream_test_reg<8>(t0, s_tests[0], s_joins, smem, k0, 0xFFu);
            if (carry0) {
#pragma unroll
                for (int i = 0; i < 8; i++) carry[i] = k0[i];
            }
            if (NV > 1) {
                a8 = stream_test_reg<8>(t1, s_tests[1], s_joins, smem, k1, a8);
                if (carry1) {
#pragma unroll
                    for (int i = 0; i < 8; i++) carry[i] = k1[i];
                }
            }
            first_pred = NV;
        } else { // the ragged last tile: every test through predicated loads
            a8 = 0;
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (row0[i >> 2] + (i & 3) < n) a8 |= 1u << i;
        }
#pragma unroll 1
        for (int t = first_pred; t < NT; t++) {
            const StreamTest& st = s_tests[t];
            const int32_t* col = (const int32_t*)vt.v[st.value_id].data;
            int32_t kk[8];
#pragma unroll
            for (int i = 0; i < 8; i++) kk[i] = ldg_stream_s32_pred(col + row0[i >> 2] + (i & 3), (a8 >> i) & 1u);
            a8 = stream_test<8>(st, s_joins, smem, kk, a8);
            if (CARRY && st.kind == 1 && st.join == pd.carry_join) {
#pragma unroll
                for (int i = 0; i < 8; i++) carry[i] = kk[i];
            }
        }
        warp_append_rows<CARRY>(a8, row0[0], row0[1], carry, writer);
    }
    writer.finish();
}

constexpr int GATHER_BLOCK = 256;

// the contiguous run [begin, end) of a selection vector of n entries that the calling warp owns (a multiple
// of 32 entries, so every warp-wide read of the vector is one aligned 128-byte line)
__device__ __forceinline__ void warp_sel_range(unsigned long long n, unsigned long long& begin, unsigned long long& end) {
    const unsigned long long warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    const unsigned long long me = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    unsigned long long per = (n + warps - 1) / warps;
    per = (per + 31) & ~31ull;
    begin = me * per;
    end = begin + per < n ? begin + per : n;
    if (begin > n) begin = n;
}

// the final pass is a chain of dependent gathers per row: latency bound, so resident warps matter more than spills.
// Measured on SSB Q4.1 SF100 (9.6 M rows reach it): 66 registers / 3 CTAs per SM 0.89 ms, 62 / 4: 0.73, 48 / 5: 0.667,
// 40 / 6: 0.669, 32 / 8: 0.70 ms.
#ifndef SR_GATHER_AGG_MIN_BLOCKS
#define SR_GATHER_AGG_MIN_BLOCKS 5
#endif
// one selective join on the selected rows: sel_in[0, *n_in) -> sel_out (appended at *counter_out)
__global__ void __launch_bounds__(GATHER_BLOCK) k_frag_gather_join(const FragDev* __restrict__ fdp, int32_t j, const __grid_constant__ VTab vt,
                                                                    const SelEntry* __restrict__ sel_in, const unsigned long long* __restrict__ n_in_ptr,
                                                                    SelEntry* __restrict__ sel_out, unsigned long long* __restrict__ counter_out) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ FragJoinDev s_join;
    for (int i = threadIdx.x; i < (int)(sizeof(FragJoinDev) / 4); i += blockDim.x) ((uint32_t*)&s_join)[i] = ((const uint32_t*)&fdp->joins[j])[i];
    __syncthreads();
    const unsigned long long n_in = *n_in_ptr;
    const FragJoinDev& fj = s_join;
    const VDesc& d = vt.v[fj.key_value_id];
    WarpSelWriter writer;
    writer.init(sel_out, counter_out);
    // each warp walks its own contiguous run of the input vector (whole chunks of one producer warp), so what
    // it appends keeps the producer's locality
    unsigned long long w_begin, w_end;
    warp_sel_range(n_in, w_begin, w_end);
    for (unsigned long long i0 = w_begin; i0 < w_end; i0 += 32) {
        const unsigned long long i = i0 + lane_id();
        bool hit = false;
        SelEntry entry = (SelEntry)SEL_INVALID;
        if (i < n_in) entry = sel_in[i];
        const uint32_t row = sel_row(entry);
        if (row != SEL_INVALID) {
            const int64_t key = load_int(d.data, d.type, (int64_t)row);
            const bool nul = d.nulls != nullptr && d.nulls[row] != 0;
            hit = !nul && join_hit_global(fj, key); // global bitmap copy: L1/L2 resident
        }
        const uint32_t m = __ballot_sync(SR_FULL_MASK, hit);
        if (m) {
            const unsigned long long base = writer.reserve(__popc(m));
            if (hit) sel_out[base + __popc(m & lanemask_lt())] = entry; // the carried key travels along
        }
    }
    writer.finish();
}

// the joins of one row in the final pass: joins [final_first_join, S) are tested, and every join whose build row is read
// downstream (or that has no bitmap) leaves its chain head in ld.bidx -- the other entries keep the 0 they start with.
// false: the row fails a tested join
__device__ __forceinline__ bool final_join_walk(const FragJoinDev* s_joins, int S, int final_first_join, FragLoader& ld) {
#pragma unroll 1
    for (int j = 0; j < S; j++) {
        const FragJoinDev& fj = s_joins[j];
        const bool test = j >= final_first_join;
        if (!test && !fj.need_head) continue;
        int64_t key;
        const bool nul = ld.load(fj.key_value_id, key);
        if (test && nul) return false;
        if (fj.need_head || !fj.use_bitmap) {
            const uint32_t head = join_lookup(fj.j, key);
            ld.bidx[j] = head;
            if (test && head == 0) return false;
        } else if (test && !join_hit_global(fj, key)) {
            return false;
        }
    }
    return true;
}

// final pass: remaining joins inline, payload lookups, aggregate update.  SINGLE: no GROUP BY (its register state
// would only cost the grouped instantiations spills).
template <bool SMEM_AGG, bool SINGLE = false>
__global__ void __launch_bounds__(GATHER_BLOCK, SR_GATHER_AGG_MIN_BLOCKS) k_frag_gather_agg(const FragDev* __restrict__ fdp, const AggDev* __restrict__ adp, const __grid_constant__ PassDev pd,
                                                                   const __grid_constant__ VTab vt, const SelEntry* __restrict__ sel_in,
                                                                   const unsigned long long* __restrict__ n_in_ptr, SelEntry* __restrict__ fail_list,
                                                                   unsigned long long* __restrict__ fail_count) {
    // Hash aggregate tables are sized from the SAMPLED survivor estimate, not for the worst case "every row is a new
    // group" (a 65 M-row batch would allocate and clear a 13 GB table for 0.2 M groups).  A row the table cannot admit
    // (admission limit) is appended to fail_list; the host grows the table and runs this kernel again over that list.
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ FragJoinDev s_joins[SR_MAX_FRAG_JOINS];
    const FragDev& fd = *fdp;
    const AggDev& ad = *adp;
    const int S = fd.num_joins;
    const bool hash_table = !SINGLE && !ad.dense && ad.num_keys > 0;
    unsigned long long known_groups = hash_table && fail_list ? *(volatile unsigned long long*)ad.ngroups : 0ull;
    for (int i = threadIdx.x; i < (int)(sizeof(FragJoinDev) / 4) * S; i += blockDim.x) ((uint32_t*)s_joins)[i] = ((const uint32_t*)fd.joins)[i];
    AccPtrs acc;
    if (SMEM_AGG) {
        acc_ptrs_smem(ad, (long long*)smem, acc);
        acc_smem_init(ad, acc);
    } else {
        acc_ptrs_global(ad, acc);
    }
    __syncthreads(); // s_joins and the shared accumulators are filled cooperatively: no warp may run ahead of that
    // Measured and rejected (profiles/r1_notes.md): requesting the NEXT row's fact sectors with prefetch.global.L2
    // while the current row walks its dependent chain.  HBM-resident input: 0.73 -> 1.27 ms (the prefetch fetches
    // whole 128-byte lines where the loads need one 32-byte sector: 4x the DRAM traffic of a pass that is bound by
    // random-sector throughput, not latency).  Host-resident input: mapped host memory is not kept in L2, the
    // prefetch only doubled the PCIe requests (117 -> 224 ms on SSB Q4.1 SF100).
    const unsigned long long n_in = *n_in_ptr;
    unsigned long long passed = 0;
    constexpr bool single = SINGLE;
    SingleAcc sacc;
    if (single) single_acc_init(ad, sacc);
    unsigned long long w_begin, w_end;
    warp_sel_range(n_in, w_begin, w_end);
    for (unsigned long long i = w_begin + lane_id(); i < w_end; i += 32) {
        const SelEntry entry = sel_in[i];
        const uint32_t row = sel_row(entry);
        if (row == SEL_INVALID) continue;
        // (a variant that fetched every fact value of the row in one burst before the dependent lookups was
        // measured slower on B200 -- more issue slots and registers than latency hidden, see profiles/)
        FragLoader ld{vt, (int64_t)row, {0, 0, 0, 0, 0, 0}, pd.carry_join >= 0 ? (int32_t)pd.carry_value_id : -1, sel_carry(entry)};
        if (!final_join_walk(s_joins, S, pd.final_first_join, ld)) continue;
        if (single) { // no GROUP BY: the state lives in the thread, not behind an atomic
            single_acc_row(ad, sacc, ld);
        } else if (hash_table) {
            HKey key;
            agg_pack_key(ad, ld, key);
            bool inserted;
            const long long slot = agg_find_slot_key(ad, key, inserted, known_groups);
            agg_count_new_groups(ad, inserted, known_groups);
            if (slot < 0) {
                if (fail_list) fail_list[atomicAdd(fail_count, 1ull)] = entry; // retried after the table has grown
                continue;
            }
            agg_apply_row<SMEM_AGG>(ad, acc, slot, ld);
        } else {
            const long long slot = agg_find_slot(ad, ld);
            if (slot >= 0) agg_apply_row<SMEM_AGG>(ad, acc, slot, ld);
        }
        passed++;
    }
    __syncwarp();
    if (single) single_acc_flush(ad, sacc);
    if (SMEM_AGG) {
        __syncthreads();
        acc_smem_flush(ad, acc);
    }
    passed = warp_sum(passed);
    if (lane_id() == 0 && passed) atomicAdd(fd.rows_passed, passed);
}

// Final pass of a fragment with one-to-many joins (reference: JoinHashMap::_probe_from_ht one-to-many walk,
// be/src/exec/join/join_hash_map.hpp:718-795 -- every probe row is emitted once per entry of the build chain of its
// key).  The probe output is never materialised: the thread that owns a surviving fact row walks the chains of its
// expanding joins like an odometer (last join fastest) and applies the aggregate once per combination, reading the
// payload columns at the current chain entries.  Hash-table aggregate: a first walk only finds / inserts the group
// slots; when the table refuses one, nothing of the row has been applied yet and the row goes to the retry list
// (a row is either applied with all its combinations or not at all).
__global__ void __launch_bounds__(GATHER_BLOCK) k_frag_gather_agg_expand(const FragDev* __restrict__ fdp, const AggDev* __restrict__ adp, const __grid_constant__ PassDev pd,
                                                                          const __grid_constant__ VTab vt, const SelEntry* __restrict__ sel_in,
                                                                          const unsigned long long* __restrict__ n_in_ptr, SelEntry* __restrict__ fail_list,
                                                                          unsigned long long* __restrict__ fail_count) {
    __shared__ FragJoinDev s_joins[SR_MAX_FRAG_JOINS];
    const FragDev& fd = *fdp;
    const AggDev& ad = *adp;
    const int S = fd.num_joins;
    const bool single = ad.num_keys == 0;
    const bool hash_table = !ad.dense && ad.num_keys > 0;
    unsigned long long known_groups = hash_table && fail_list ? *(volatile unsigned long long*)ad.ngroups : 0ull;
    for (int i = threadIdx.x; i < (int)(sizeof(FragJoinDev) / 4) * S; i += blockDim.x) ((uint32_t*)s_joins)[i] = ((const uint32_t*)fd.joins)[i];
    AccPtrs acc;
    acc_ptrs_global(ad, acc);
    __syncthreads();
    const unsigned long long n_in = *n_in_ptr;
    unsigned long long passed = 0;
    SingleAcc sacc;
    if (single) single_acc_init(ad, sacc);
    unsigned long long w_begin, w_end;
    warp_sel_range(n_in, w_begin, w_end);
    for (unsigned long long i = w_begin + lane_id(); i < w_end; i += 32) {
        const SelEntry entry = sel_in[i];
        const uint32_t row = sel_row(entry);
        if (row == SEL_INVALID) continue;
        FragLoader ld{vt, (int64_t)row, {0, 0, 0, 0, 0, 0}, pd.carry_join >= 0 ? (int32_t)pd.carry_value_id : -1, sel_carry(entry)};
        if (!final_join_walk(s_joins, S, pd.final_first_join, ld)) continue;
        uint32_t head[SR_MAX_FRAG_JOINS];
#pragma unroll 1
        for (int j = 0; j < S; j++) head[j] = ld.bidx[j];
        bool refused = false;
#pragma unroll 1
        for (int phase = hash_table ? 0 : 1; phase < 2 && !refused; phase++) {
            while (true) {
                if (single) {
                    single_acc_row(ad, sacc, ld);
                } else if (hash_table) {
                    HKey key;
                    agg_pack_key(ad, ld, key);
                    bool inserted;
                    const long long slot = agg_find_slot_key(ad, key, inserted, known_groups);
                    agg_count_new_groups(ad, inserted, known_groups);
                    if (slot < 0) {
                        refused = true;
                        break;
                    }
                    if (phase == 1) agg_apply_row<false>(ad, acc, slot, ld);
                } else {
                    const long long slot = agg_find_slot(ad, ld);
                    if (slot >= 0) agg_apply_row<false>(ad, acc, slot, ld);
                }
                if (phase == 1) passed++;
                // next combination: advance the last expanding join, carry into the one before it when its chain ends
                int j = S - 1;
#pragma unroll 1
                for (; j >= 0; j--) {
                    if (!s_joins[j].expand) continue;
                    const uint32_t nx = __ldg(s_joins[j].j.next + ld.bidx[j]);
                    if (nx) {
                        ld.bidx[j] = nx;
                        break;
                    }
                    ld.bidx[j] = head[j];
                }
                if (j < 0) break;
            }
            if (refused) {
                // phase 0 only (phase 1 finds the slots phase 0 created; tables never shrink in between)
                if (fail_list) fail_list[atomicAdd(fail_count, 1ull)] = entry;
            } else if (phase == 0) {
#pragma unroll 1
                for (int j = 0; j < S; j++) ld.bidx[j] = head[j]; // the odometer ends on the heads anyway; keeps the second walk independent of that
            }
        }
    }
    __syncwarp();
    if (single) single_acc_flush(ad, sacc);
    passed = warp_sum(passed);
    if (lane_id() == 0 && passed) atomicAdd(fd.rows_passed, passed);
}

} // namespace srd
