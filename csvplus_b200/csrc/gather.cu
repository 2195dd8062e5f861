// gather.cu — column-level primitives shared by Filter / IndexOn / Join:
//   * device-wide exclusive scan (single pass, decoupled look-back);
//   * string-column gather by row ids (lengths -> scan -> byte copy) = the columnar form of the
//     per-row map copies the reference makes (Row.Select csvplus.go:122-134, mergeRows :571-583);
//   * Filter(Like/All/Any/Not) over a materialised table (csvplus.go:276-286, :1243-1293);
//   * row-wise concatenation of tables (assembling all-gathered shards).
#include <algorithm>

#include "core.hpp"
#include "pred.cuh"
#include "util.cuh"

namespace cpb {

// ------------------------------------------------------------------ exclusive scan (uint32 in, uint32 out, uint64 total)
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// tile state word: bits 63:62 status (0 none, 1 aggregate, 2 inclusive), bits 61:0 value
// GATHER: the scanned values are the lengths of the strings picked by `ids` (identity when null) from the offsets
// array `in` -- the length array of a gather is never materialised.
template <bool GATHER>
__global__ void __launch_bounds__(SCAN_THREADS) scan_u32_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ ids,
                                                                uint32_t* out, uint64_t n, unsigned long long* state,
                                                                uint32_t* ticket, unsigned long long* total) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[SCAN_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    for (;;) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint64_t tile = s_tile;
        if (tile >= ntiles) break;
        const uint64_t base = tile * SCAN_TILE + (uint64_t)tid * SCAN_ITEMS;
        uint32_t v[SCAN_ITEMS];
        uint32_t sum = 0;
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++) {
            v[i] = 0;
            if (base + i < n) {
                if (GATHER) { const uint32_t r = ids ? ids[base + i] : (uint32_t)(base + i); v[i] = in[r + 1] - in[r]; }
                else v[i] = in[base + i];
            }
            sum += v[i];
        }
        uint32_t inc = warp_incl_scan(sum);
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        uint32_t woff = 0, tot = 0;
#pragma unroll
        for (int i = 0; i < SCAN_THREADS / 32; i++) { uint32_t t = s_warp[i]; if (i < warp) woff += t; tot += t; }
        if (warp == 0) {
            unsigned long long excl = 0;
            if (tile == 0) {
                if (lane == 0) atomicExch(&state[0], (2ull << 62) | tot);
            } else {
                if (lane == 0) atomicExch(&state[tile], (1ull << 62) | tot);
                int64_t b = (int64_t)tile - 1;
                for (;;) {
                    int64_t p = b - lane;
                    unsigned long long s = 2ull << 62;
                    if (p >= 0) { do { s = ld_relaxed_u64((const uint64_t*)&state[p]); } while ((s >> 62) == 0); }
                    uint32_t incl = __ballot_sync(0xffffffffu, (s >> 62) == 2);
                    int f = __ffs(incl) - 1;
                    unsigned long long val = (f < 0 || lane <= f) ? (s & ((1ull << 62) - 1)) : 0ull;
                    excl += warp_sum_u64(val);
                    if (f >= 0) break;
                    b -= 32;
                }
                if (lane == 0) atomicExch(&state[tile], (2ull << 62) | (excl + tot));
            }
            if (lane == 0) { s_prefix = excl; if (tile == ntiles - 1) { *total = excl + tot; out[n] = (uint32_t)(excl + tot); } }
        }
        __syncthreads();
        uint32_t run = (uint32_t)s_prefix + woff + (inc - sum);
#pragma unroll
        for (int i = 0; i < SCAN_ITEMS; i++) { if (base + i < n) out[base + i] = run; run += v[i]; }
        __syncthreads();
    }
}

__global__ void scan_empty_kernel(uint32_t* out, unsigned long long* total) { out[0] = 0; *total = 0; }

// out may alias in; out has n+1 entries (out[n] = total, truncated to 32 bits); *total_dev holds the 64-bit total.
// gather_off != nullptr: scan the lengths off[ids[i]+1]-off[ids[i]] instead of `in` (ids may be null = identity).
static void scan_impl(Ctx* c, const uint32_t* in, const uint32_t* gather_off, const uint32_t* ids, uint32_t* out, uint64_t n,
                      uint64_t* total_dev) {
    if (n == 0) {
        KernelTimer kt(c, "scan_u32", 0);
        scan_empty_kernel<<<1, 1, 0, c->stream>>>(out, (unsigned long long*)total_dev);
        return;
    }
    uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    Buf st = dev_alloc(c, ntiles * 8 + 64);
    CPB_CUDA(cudaMemsetAsync(st->p, 0, ntiles * 8 + 64, c->stream));
    unsigned long long* state = st->as<unsigned long long>() + 8;
    uint32_t* ticket = st->as<uint32_t>();
    uint32_t grid = (uint32_t)std::min<uint64_t>(ntiles, (uint64_t)c->sm_count * 8);
    if (gather_off) {
        KernelTimer kt(c, "scan_gather_len", n * (ids ? 16 : 12));
        scan_u32_kernel<true><<<grid, SCAN_THREADS, 0, c->stream>>>(gather_off, ids, out, n, state, ticket, (unsigned long long*)total_dev);
    } else {
        KernelTimer kt(c, "scan_u32", n * 8);
        scan_u32_kernel<false><<<grid, SCAN_THREADS, 0, c->stream>>>(in, nullptr, out, n, state, ticket, (unsigned long long*)total_dev);
    }
    CPB_CUDA(cudaGetLastError());
}
void exclusive_scan_u32(Ctx* c, const uint32_t* in, uint32_t* out, uint64_t n, uint64_t* total_dev) {
    scan_impl(c, in, nullptr, nullptr, out, n, total_dev);
}

// ------------------------------------------------------------------ gather by row ids
// One warp gathers 32 consecutive output values.  Their destination bytes are contiguous, so the lanes first
// copy their (randomly placed) source strings into a per-warp shared-memory stage laid out like the
// destination, then the warp writes the stage with aligned 16-byte stores: HBM/L2 see full sectors instead of one
// scattered byte store per lane.  ids==nullptr means identity (compaction of a view).
// Copies len bytes from an arbitrarily aligned source to an arbitrarily aligned destination in whole aligned 8-byte
// words on both sides: every destination word is one funnel shift of two consecutive aligned source words (each
// source word is loaded once).  The lanes of a warp read unrelated strings, so every load instruction costs 32 L1
// wavefronts and a byte-wise loop is wavefront-bound.  Source buffers are allocated in multiples of 512 bytes
// (DevBuf), so the aligned word holding the last byte is always readable; no word past it is read.
// `put(p, v, mask)` stores destination word p: v holds the copied bytes where mask is 0xff and zeros elsewhere.  A
// word the copy covers only in part (mask != ~0) may share bytes with a neighbouring value, and the policy decides how
// it is merged (StagePut, PrivatePut, GlobalPut).  GLOBAL: the source is global memory (read through the
// non-coherent path), else shared.
template <bool GLOBAL, class Put>
__device__ __forceinline__ void copy_unaligned(uint8_t* q, const uint8_t* sp, uint32_t len, Put put) {
    if (len == 0) return;
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(sp) & 7u), dm = (uint32_t)(reinterpret_cast<uintptr_t>(q) & 7u);
    const unsigned long long* wp = reinterpret_cast<const unsigned long long*>(sp - mis);
    unsigned long long* dp = reinterpret_cast<unsigned long long*>(q - dm);
    auto ld = [&](uint32_t k) { return GLOBAL ? __ldg(wp + k) : wp[k]; };
    const uint32_t lastw = (mis + len - 1) >> 3, nw = (dm + len + 7) >> 3, ec = (dm + len) & 7u;
    // destination word t starts at source stream byte (mis - dm) + 8t: bytes e.. of source word t + (mis < dm ? -1 : 0)
    // and the low bytes of the one after it (a word before the first is never read: its bytes are all masked off)
    const uint32_t es = ((mis - dm) & 7u) * 8;
    uint32_t m = mis < dm ? 0u : 1u;
    unsigned long long a = mis < dm ? 0ull : ld(0);
    for (uint32_t t = 0; t < nw; t++, m++) {
        const unsigned long long b = m <= lastw ? ld(m) : 0ull;
        const unsigned long long v = es ? (a >> es) | (b << (64 - es)) : a;
        unsigned long long mask = t == 0 ? ~0ull << (8 * dm) : ~0ull;
        if (t == nw - 1 && ec) mask &= (1ull << (8 * ec)) - 1;
        put(dp + t, v & mask, mask);
        a = b;
    }
}
// a warp stage zeroed beforehand: neighbouring lanes may share a partial word, they merge it with a shared atomic OR
// per 4-byte half (native ATOMS.OR; the 8-byte OR is a compare-and-swap loop)
struct StagePut {
    __device__ __forceinline__ void operator()(unsigned long long* p, unsigned long long v, unsigned long long mask) const {
        if (mask == ~0ull) { *p = v; return; }
        uint32_t* h = reinterpret_cast<uint32_t*>(p);
        const uint32_t ml = (uint32_t)mask, mh = (uint32_t)(mask >> 32);
        if (ml == ~0u) h[0] = (uint32_t)v; else if (ml) atomicOr(h, (uint32_t)v);
        if (mh == ~0u) h[1] = (uint32_t)(v >> 32); else if (mh) atomicOr(h + 1, (uint32_t)(v >> 32));
    }
};
// a lane-private buffer written left to right: a word is first written from its byte 0 (plain store, zeros above the
// value), a later value that starts inside it ORs its bytes in
struct PrivatePut {
    __device__ __forceinline__ void operator()(unsigned long long* p, unsigned long long v, unsigned long long mask) const {
        if (mask & 0xffull) *p = v; else *p |= v;
    }
};
// global memory other threads write next to: the bytes of a partial word are stored one by one
struct GlobalPut {
    __device__ __forceinline__ void operator()(unsigned long long* p, unsigned long long v, unsigned long long mask) const {
        if (mask == ~0ull) { *p = v; return; }
        uint8_t* b = reinterpret_cast<uint8_t*>(p);
#pragma unroll
        for (int k = 0; k < 8; k++) if ((mask >> (8 * k)) & 0xffull) b[k] = (uint8_t)(v >> (8 * k));
    }
};
// zeroes stage bytes [0, end) (rounded up to 16) for StagePut
__device__ __forceinline__ void warp_zero_stage(uint8_t* stage, uint32_t end, int lane) {
    for (uint32_t x = lane * 16; x < end; x += 32 * 16) *reinterpret_cast<uint4*>(stage + x) = make_uint4(0, 0, 0, 0);
}
// Writes stage bytes [sh, end) to gb (16-byte aligned, laid out like the stage): whole vectors with 16-byte
// stores, the partial first / last vector one byte per lane (lanes 0-15 / 16-31) -- no lane loops over bytes.
__device__ __forceinline__ void warp_store_stage(uint8_t* gb, const uint8_t* stage, uint32_t sh, uint32_t end, int lane) {
    for (uint32_t x = lane * 16; x + 16 <= end; x += 32 * 16)
        if (x >= sh) *reinterpret_cast<uint4*>(gb + x) = *reinterpret_cast<const uint4*>(stage + x);
    const uint32_t t0 = end & ~15u;
    const bool head = lane < 16;
    const uint32_t y = head ? (uint32_t)lane : t0 + (uint32_t)(lane - 16);
    const bool on = head ? sh != 0 : ((end & 15u) != 0 && (t0 != 0 || sh == 0));
    if (on && y >= sh && y < end) gb[y] = stage[y];
}
constexpr int GW_WARPS = 8;
constexpr int GW_STAGE = 2048;  // bytes staged per warp; longer groups take the direct path
__global__ void __launch_bounds__(GW_WARPS * 32) gather_copy_kernel(const uint32_t* __restrict__ src_off, const uint8_t* __restrict__ src,
                                                                    const uint32_t* __restrict__ ids, const uint32_t* __restrict__ dst_off,
                                                                    uint8_t* __restrict__ dst, uint64_t n) {
    __shared__ __align__(16) uint8_t stage_all[GW_WARPS][GW_STAGE + 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* stage = stage_all[warp];
    const uint64_t nwarps = (uint64_t)gridDim.x * GW_WARPS;
    for (uint64_t g = (uint64_t)blockIdx.x * GW_WARPS + warp; g * 32 < n; g += nwarps) {
        const uint64_t i = g * 32 + lane;
        uint32_t s = 0, len = 0, d = 0;
        if (i < n) {
            const uint32_t r = ids ? ids[i] : (uint32_t)i;
            s = src_off[r]; len = src_off[r + 1] - s; d = dst_off[i];
        }
        const uint32_t d0 = __shfl_sync(0xffffffffu, d, 0);
        const uint64_t last = (g * 32 + 31 < n ? g * 32 + 31 : n - 1) - g * 32;
        const uint32_t dl = __shfl_sync(0xffffffffu, d + len, (int)last);
        const uint32_t total = dl - d0, sh = d0 & 15u;
        const uint8_t* sp = src + s;
        if (sh + total <= GW_STAGE) {
            warp_zero_stage(stage, sh + total, lane);
            __syncwarp();
            copy_unaligned<true>(stage + sh + (d - d0), sp, len, StagePut{});
            __syncwarp();
            warp_store_stage(dst + (d0 - sh), stage, sh, sh + total, lane);
            __syncwarp();
        } else {
            copy_unaligned<true>(dst + d, sp, len, GlobalPut{});
        }
    }
}

static inline uint32_t blocks_for(uint64_t n, int threads) { return (uint32_t)((n + threads - 1) / threads); }

struct PendingGather { Column col; const Column* src; Buf total; };

// gathers several columns with ONE host synchronisation (totals of all columns read back together)
static std::vector<Column> gather_columns(Ctx* c, const std::vector<const Column*>& srcs, const uint32_t* ids, int64_t nout) {
    std::vector<Column> out(srcs.size());
    if (srcs.empty()) return out;
    Buf totals = dev_alloc(c, srcs.size() * 8);
    for (size_t k = 0; k < srcs.size(); k++) {
        out[k].name = srcs[k]->name;
        out[k].offsets = dev_alloc(c, ((size_t)nout + 1) * 4);
        uint32_t* o = out[k].offsets->as<uint32_t>();
        scan_impl(c, nullptr, srcs[k]->off(), ids, o, (uint64_t)nout, totals->as<uint64_t>() + k);
    }
    uint64_t* ht = (uint64_t*)c->pinned_scratch(srcs.size() * 8);
    CPB_CUDA(cudaMemcpyAsync(ht, totals->p, srcs.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    std::vector<uint64_t> tot(ht, ht + srcs.size());
    for (size_t k = 0; k < srcs.size(); k++) {
        if (tot[k] > 0xffffffffull) throw DataError{CPB_E_TOO_LARGE, (int)k, 0, false, "a result column exceeds 4 GiB; process in smaller batches"};
        out[k].data = dev_alloc(c, tot[k] + 16);
        if (nout && tot[k]) {
            KernelTimer kt(c, "gather_copy", 2 * tot[k] + (uint64_t)nout * 12);
            const uint32_t gblocks = (uint32_t)std::min<uint64_t>(((uint64_t)nout + GW_WARPS * 32 - 1) / (GW_WARPS * 32), (uint64_t)c->sm_count * 16);
            gather_copy_kernel<<<gblocks, GW_WARPS * 32, 0, c->stream>>>(srcs[k]->off(), srcs[k]->bytes(), ids,
                                                                              out[k].offsets->as<uint32_t>(), out[k].data->as<uint8_t>(), (uint64_t)nout);
            CPB_CUDA(cudaGetLastError());
        }
    }
    return out;
}

Column gather_column(Ctx* c, const Column& src, const uint32_t* row_ids, int64_t nout) {
    return gather_columns(c, {&src}, row_ids, nout)[0];
}

std::shared_ptr<Table> gather_rows(Ctx* c, const Table& t, const uint32_t* row_ids, int64_t nout) {
    auto r = std::make_shared<Table>(); r->ctx = c; r->nrows = nout; r->first_line = t.first_line;
    // columns sharing buffers (AssumeHeader aliases) are gathered once
    std::vector<const Column*> uniq; std::vector<int> which(t.cols.size());
    for (size_t i = 0; i < t.cols.size(); i++) {
        int f = -1;
        for (size_t u = 0; u < uniq.size(); u++)
            if (uniq[u]->offsets == t.cols[i].offsets && uniq[u]->data == t.cols[i].data && uniq[u]->row0 == t.cols[i].row0) f = (int)u;
        if (f < 0) { f = (int)uniq.size(); uniq.push_back(&t.cols[i]); }
        which[i] = f;
    }
    auto g = gather_columns(c, uniq, row_ids, nout);
    for (size_t i = 0; i < t.cols.size(); i++) { Column col = g[which[i]]; col.name = t.cols[i].name; r->cols.push_back(col); }
    return r;
}

Column materialize(Ctx* c, const Column& col, int64_t nrows) { return gather_columns(c, {&col}, nullptr, nrows)[0]; }

// ------------------------------------------------------------------ row slots: one random access per gathered index row
// A join reads index rows in probe order, i.e. at random: per output column that is one access to the offsets and
// one to the bytes, each a 64-byte DRAM granule once the index outgrows L2 (measured: 9 GB of DRAM reads to gather
// 0.7 GB).  Short rows are therefore re-laid once per index as fixed-size slots (all output columns back to back) +
// one packed word of lengths; a gather then costs one L2-friendly 4-byte read (lengths -> offsets of all columns in
// one scan) and one slot read (bytes of all columns in one pass).
constexpr int RS_MAXC = 4;       // columns per slot set (lengths are 8 bits each in one word)
constexpr uint32_t RS_MAXS = 64; // bytes per slot
struct SlotCols { int nc; const uint32_t* off[RS_MAXC]; const uint8_t* data[RS_MAXC]; };
struct SlotOut { uint32_t* off[RS_MAXC]; uint8_t* data[RS_MAXC]; };

// (`perm`: slot r holds source row perm[r] — the slots are laid out in sorted order straight from the unsorted rows
// of the index source; null = identity)
// (grid-stride; the longest row and the overflow flag are reduced per block before one global atomic each)
template <int NC>
__global__ void __launch_bounds__(256) slot_lens_kernel(SlotCols sc, const uint32_t* __restrict__ perm, uint64_t n, uint32_t* lens,
                                                        uint32_t* stat) {  // stat: [0] max row bytes, [1] a value > 255 bytes
    __shared__ uint32_t s_max, s_bad;
    if (threadIdx.x == 0) { s_max = 0; s_bad = 0; }
    __syncthreads();
    uint32_t mx = 0, bad = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t sr = perm ? perm[r] : r;
        uint32_t tot = 0, packed = 0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const uint32_t l = sc.off[c][sr + 1] - sc.off[c][sr];
            bad |= l > 255u;
            packed |= (l & 255u) << (8 * c);
            tot += l;
        }
        lens[r] = packed;
        mx = max(mx, tot);
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) { if (mx) atomicMax(&s_max, mx); if (bad) s_bad = 1u; }
    __syncthreads();
    if (threadIdx.x == 0) { if (s_max) atomicMax(&stat[0], s_max); if (s_bad) stat[1] = 1u; }
}
// one block lays out 256 consecutive slots in shared memory, each lane its own slot with 8-byte word stores (row
// stride padded to an odd number of 8-byte words: no bank conflicts), and writes them with coalesced 8-byte stores
constexpr uint32_t RS_PAD = 8;
template <int NC>
__global__ void __launch_bounds__(256) slot_fill_kernel(SlotCols sc, const uint32_t* __restrict__ perm, uint64_t n, uint32_t S, uint8_t* slots) {
    __shared__ __align__(16) uint8_t sm[256 * (RS_MAXS + RS_PAD)];
    const uint64_t r0 = (uint64_t)blockIdx.x * 256, r = r0 + threadIdx.x;
    uint8_t* q = sm + threadIdx.x * (S + RS_PAD);
    if (r < n) {
        const uint64_t sr = perm ? perm[r] : r;
        uint32_t pos = 0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const uint32_t s = sc.off[c][sr], l = sc.off[c][sr + 1] - s;
            copy_unaligned<true>(q + pos, sc.data[c] + s, l, PrivatePut{});
            pos += l;
        }
        // the word holding the last byte is zero above it; the words after it are zeroed here
        for (uint32_t w = (pos + 7) / 8; w < S / 8; w++) reinterpret_cast<unsigned long long*>(q)[w] = 0ull;
    }
    __syncthreads();
    const uint32_t rows = (uint32_t)(n - r0 < 256 ? n - r0 : 256), wps = S / 8;  // 8-byte words per slot
    unsigned long long* g = reinterpret_cast<unsigned long long*>(slots + r0 * S);
    const unsigned long long* sw = reinterpret_cast<const unsigned long long*>(sm);
    for (uint32_t x = threadIdx.x; x < rows * wps; x += 256) g[x] = sw[(x / wps) * (wps + RS_PAD / 8) + x % wps];
}

// exclusive scans of the NC length fields of lens[ids[i]] in one pass (same chained look-back as scan_u32_kernel;
// warp c resolves column c)
constexpr int LS_ITEMS = 8;
constexpr int LS_TILE = SCAN_THREADS * LS_ITEMS;
template <int NC>
__global__ void __launch_bounds__(SCAN_THREADS) scan_lens_kernel(const uint32_t* __restrict__ lens, const uint32_t* __restrict__ ids, uint64_t n,
                                                                 SlotOut out, unsigned long long* state, uint32_t* ticket,
                                                                 unsigned long long* totals) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[NC][SCAN_THREADS / 32];
    __shared__ unsigned long long s_prefix[NC];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t ntiles = (n + LS_TILE - 1) / LS_TILE;
    for (;;) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint64_t tile = s_tile;
        if (tile >= ntiles) break;
        const uint64_t base = tile * LS_TILE + (uint64_t)tid * LS_ITEMS;
        uint32_t p[LS_ITEMS];
        if (base + LS_ITEMS <= n) {
            const uint4 a = *reinterpret_cast<const uint4*>(ids + base), b = *reinterpret_cast<const uint4*>(ids + base + 4);
            p[0] = lens[a.x]; p[1] = lens[a.y]; p[2] = lens[a.z]; p[3] = lens[a.w];
            p[4] = lens[b.x]; p[5] = lens[b.y]; p[6] = lens[b.z]; p[7] = lens[b.w];
        } else {
#pragma unroll
            for (int i = 0; i < LS_ITEMS; i++) p[i] = base + i < n ? lens[ids[base + i]] : 0u;
        }
        uint32_t sum[NC], inc[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) {
            sum[c] = 0;
#pragma unroll
            for (int i = 0; i < LS_ITEMS; i++) sum[c] += (p[i] >> (8 * c)) & 255u;
            inc[c] = warp_incl_scan(sum[c]);
            if (lane == 31) s_warp[c][warp] = inc[c];
        }
        __syncthreads();
        if (warp < NC) {
            const int c = warp;
            uint32_t tot = 0;
#pragma unroll
            for (int i = 0; i < SCAN_THREADS / 32; i++) tot += s_warp[c][i];
            unsigned long long* st = state + c;  // state[tile * NC + c]
            unsigned long long excl = 0;
            if (tile == 0) {
                if (lane == 0) atomicExch(&st[0], (2ull << 62) | tot);
            } else {
                if (lane == 0) atomicExch(&st[tile * NC], (1ull << 62) | tot);
                int64_t b = (int64_t)tile - 1;
                for (;;) {
                    const int64_t q = b - lane;
                    unsigned long long sv = 2ull << 62;
                    if (q >= 0) { do { sv = ld_relaxed_u64((const uint64_t*)&st[q * NC]); } while ((sv >> 62) == 0); }
                    const uint32_t incl = __ballot_sync(0xffffffffu, (sv >> 62) == 2);
                    const int f = __ffs(incl) - 1;
                    const unsigned long long val = (f < 0 || lane <= f) ? (sv & ((1ull << 62) - 1)) : 0ull;
                    excl += warp_sum_u64(val);
                    if (f >= 0) break;
                    b -= 32;
                }
                if (lane == 0) atomicExch(&st[tile * NC], (2ull << 62) | (excl + tot));
            }
            if (lane == 0) {
                s_prefix[c] = excl;
                if (tile == ntiles - 1) { totals[c] = excl + tot; out.off[c][n] = (uint32_t)(excl + tot); }
            }
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NC; c++) {
            uint32_t run = (uint32_t)s_prefix[c] + (inc[c] - sum[c]);
#pragma unroll
            for (int i = 0; i < SCAN_THREADS / 32; i++) if (i < warp) run += s_warp[c][i];
            uint32_t* o = out.off[c];
            if (base + LS_ITEMS <= n) {
                uint32_t v[LS_ITEMS];
#pragma unroll
                for (int i = 0; i < LS_ITEMS; i++) { v[i] = run; run += (p[i] >> (8 * c)) & 255u; }
                *reinterpret_cast<uint4*>(o + base) = make_uint4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<uint4*>(o + base + 4) = make_uint4(v[4], v[5], v[6], v[7]);
            } else {
#pragma unroll
                for (int i = 0; i < LS_ITEMS; i++) { if (base + i < n) o[base + i] = run; run += (p[i] >> (8 * c)) & 255u; }
            }
        }
        __syncthreads();
    }
}

// One warp gathers 32 consecutive output rows: every lane pulls its row's slot into shared memory with 16-byte
// loads (the one random access), then, column by column, the warp lays the values out like the destination in the
// staging buffer with 8-byte word copies and writes it with aligned 16-byte stores (as gather_copy_kernel does).
// Slot stride: the smallest odd number of 16-byte units above S, so the 16-byte stores of 8 lanes (one shared-memory
// phase) hit 8 distinct bank quads.
constexpr uint32_t SC_MAXSTRIDE = RS_MAXS + 16;
__host__ __device__ __forceinline__ uint32_t slot_stride(uint32_t S) { return 16 * ((S / 16 + 1) | 1u); }
template <int NC>
__global__ void __launch_bounds__(GW_WARPS * 32) slot_copy_kernel(const uint8_t* __restrict__ slots, uint32_t S, const uint32_t* __restrict__ ids,
                                                                  SlotOut out, uint64_t n) {
    __shared__ __align__(16) uint8_t slot_sm[GW_WARPS][32 * SC_MAXSTRIDE];
    __shared__ __align__(16) uint8_t stage_all[GW_WARPS][GW_STAGE + 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* stage = stage_all[warp];
    uint8_t* myslot = slot_sm[warp] + lane * slot_stride(S);
    const uint64_t nwarps = (uint64_t)gridDim.x * GW_WARPS;
    for (uint64_t g = (uint64_t)blockIdx.x * GW_WARPS + warp; g * 32 < n; g += nwarps) {
        const uint64_t i = g * 32 + lane;
        const bool valid = i < n;
        if (valid) {
            const uint4* sp = reinterpret_cast<const uint4*>(slots + (uint64_t)ids[i] * S);
            for (uint32_t j = 0; j < S / 16; j++) reinterpret_cast<uint4*>(myslot)[j] = __ldg(sp + j);
        }
        const uint64_t last = (g * 32 + 31 < n ? g * 32 + 31 : n - 1) - g * 32;
        uint32_t pos = 0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            uint32_t d = 0, len = 0;
            if (valid) { d = out.off[c][i]; len = out.off[c][i + 1] - d; }
            const uint32_t d0 = __shfl_sync(0xffffffffu, d, 0);
            const uint32_t dl = __shfl_sync(0xffffffffu, d + len, (int)last);
            const uint32_t total = dl - d0, sh = d0 & 15u;
            const uint8_t* sp = myslot + pos;
            uint8_t* dst = out.data[c];
            if (sh + total <= GW_STAGE) {
                warp_zero_stage(stage, sh + total, lane);
                __syncwarp();
                copy_unaligned<false>(stage + sh + (d - d0), sp, len, StagePut{});
                __syncwarp();
                warp_store_stage(dst + (d0 - sh), stage, sh, sh + total, lane);
                __syncwarp();
            } else {
                copy_unaligned<false>(dst + d, sp, len, GlobalPut{});
            }
            pos += len;
        }
        __syncwarp();  // the slots are overwritten by the next round
    }
}

static RowSlots& ensure_row_slots(Ctx* c, Index& ix, const std::vector<int>& cols, bool by_src) {
    std::lock_guard<std::mutex> lk(ix.mu);
    auto& smap = by_src ? ix.row_slots_src : ix.row_slots;
    auto it = smap.find(cols);
    if (it != smap.end()) { wait_ready(c, it->second.ready); return it->second; }
    RowSlots rs;
    // by_src: slot r = source row r (filled sequentially); else sorted order: the sorted rows if they exist, else the source
    // rows through the permutation
    const Table& t = by_src ? *ix.src : (ix.table ? *ix.table : *ix.src);
    const uint32_t* perm = (by_src || ix.table) ? nullptr : ix.perm->as<uint32_t>();
    const uint64_t n = (uint64_t)ix.nrows;
    if (n > 0 && !cols.empty() && cols.size() <= (size_t)RS_MAXC) {
        SlotCols sc{};
        sc.nc = (int)cols.size();
        for (int k = 0; k < sc.nc; k++) { sc.off[k] = t.cols[cols[k]].off(); sc.data[k] = t.cols[cols[k]].bytes(); }
        Buf lens = dev_alloc_owned(ix.ctx, c, n * 4), stat = dev_alloc(c, 8);  // kept structures: the index owner's pool
        CPB_CUDA(cudaMemsetAsync(stat->p, 0, 8, c->stream));
        uint64_t col_bytes = n * 4 * sc.nc;
        {
            KernelTimer kt(c, "slot_build", col_bytes + n * 4);
            const uint32_t grid = (uint32_t)std::min<uint64_t>(blocks_for(n, 256), (uint64_t)c->sm_count * 8);
#define CPB_SL(NC) slot_lens_kernel<NC><<<grid, 256, 0, c->stream>>>(sc, perm, n, lens->as<uint32_t>(), stat->as<uint32_t>())
            switch (sc.nc) { case 1: CPB_SL(1); break; case 2: CPB_SL(2); break; case 3: CPB_SL(3); break; default: CPB_SL(4); break; }
#undef CPB_SL
            CPB_CUDA(cudaGetLastError());
        }
        uint32_t* hs = (uint32_t*)c->pinned_scratch(8);
        CPB_CUDA(cudaMemcpyAsync(hs, stat->p, 8, cudaMemcpyDeviceToHost, c->stream));
        sync_stream(c);
        if (hs[1] == 0 && hs[0] <= RS_MAXS) {
            rs.S = std::max<uint32_t>(16, (hs[0] + 15) & ~15u);
            rs.slots = dev_alloc_owned(ix.ctx, c, n * rs.S);
            rs.lens = lens;
            KernelTimer kt(c, "slot_build", n * rs.S * 2);
#define CPB_SF(NC) slot_fill_kernel<NC><<<blocks_for(n, 256), 256, 0, c->stream>>>(sc, perm, n, rs.S, rs.slots->as<uint8_t>())
            switch (sc.nc) { case 1: CPB_SF(1); break; case 2: CPB_SF(2); break; case 3: CPB_SF(3); break; default: CPB_SF(4); break; }
#undef CPB_SF
            CPB_CUDA(cudaGetLastError());
            rs.usable = true;
        }
    }
    rs.ready = record_ready(c);  // another context (stream) that finds it in the map waits for this event, not the host
    return smap.emplace(cols, std::move(rs)).first->second;
}

std::shared_ptr<Table> gather_index_rows(Ctx* c, Index& ix, const std::vector<int>& cols, const uint32_t* ids, int64_t nout, bool by_src) {
    auto plain = [&]() {  // per-column gather: from the source rows (ids = source rows), or from the physically sorted rows
        std::shared_ptr<Table> keep = by_src ? ix.src : sorted_table(c, ix);
        const Table& st = *keep;
        Table sub; sub.ctx = c; sub.nrows = st.nrows; sub.first_line = st.first_line;
        for (int ci : cols) sub.cols.push_back(st.cols[ci]);
        return gather_rows(c, sub, ids, nout);
    };
    static const bool disabled = getenv("CPB_NO_ROWSLOTS") != nullptr;
    bool use = !disabled && ids != nullptr && nout > 0 && !cols.empty() && cols.size() <= (size_t)RS_MAXC;
    if (use) {
        bool built;
        { std::lock_guard<std::mutex> lk(ix.mu); built = (by_src ? ix.row_slots_src : ix.row_slots).count(cols) != 0; }
        if (!built && nout < ix.nrows) use = false;  // laying the slots out costs about one gather of the whole index
    }
    if (!use) return plain();
    RowSlots& rs = ensure_row_slots(c, ix, cols, by_src);
    if (!rs.usable) return plain();
    const Table& t = ix.schema();

    const int nc = (int)cols.size();
    auto r = std::make_shared<Table>(); r->ctx = c; r->nrows = nout; r->first_line = t.first_line;
    SlotOut so{};
    std::vector<Column> out(nc);
    for (int k = 0; k < nc; k++) {
        out[k].name = t.cols[cols[k]].name;
        out[k].offsets = dev_alloc(c, ((size_t)nout + 1) * 4);
        so.off[k] = out[k].offsets->as<uint32_t>();
    }
    const uint64_t n = (uint64_t)nout, ntiles = (n + LS_TILE - 1) / LS_TILE;
    Buf st = dev_alloc(c, ntiles * nc * 8 + 64 + RS_MAXC * 8);
    CPB_CUDA(cudaMemsetAsync(st->p, 0, ntiles * nc * 8 + 64 + RS_MAXC * 8, c->stream));
    uint32_t* ticket = st->as<uint32_t>();
    unsigned long long* totals = st->as<unsigned long long>() + 1;
    unsigned long long* state = st->as<unsigned long long>() + 8 + RS_MAXC;
    {
        KernelTimer kt(c, "slot_scan_lens", n * (8 + 4 * (uint64_t)nc));
        const uint32_t grid = (uint32_t)std::min<uint64_t>(ntiles, (uint64_t)c->sm_count * 8);
#define CPB_LS(NC) scan_lens_kernel<NC><<<grid, SCAN_THREADS, 0, c->stream>>>(rs.lens->as<uint32_t>(), ids, n, so, state, ticket, totals)
        switch (nc) { case 1: CPB_LS(1); break; case 2: CPB_LS(2); break; case 3: CPB_LS(3); break; default: CPB_LS(4); break; }
#undef CPB_LS
        CPB_CUDA(cudaGetLastError());
    }
    uint64_t* ht = (uint64_t*)c->pinned_scratch(RS_MAXC * 8);
    CPB_CUDA(cudaMemcpyAsync(ht, totals, nc * 8, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    uint64_t all = 0;
    for (int k = 0; k < nc; k++) {
        if (ht[k] > 0xffffffffull) throw DataError{CPB_E_TOO_LARGE, k, 0, false, "a result column exceeds 4 GiB; process in smaller batches"};
        out[k].data = dev_alloc(c, ht[k] + 16);
        so.data[k] = out[k].data->as<uint8_t>();
        all += ht[k];
    }
    {
        KernelTimer kt(c, "slot_copy", 2 * all + n * (4 + 4 * (uint64_t)nc));
        const uint32_t gblocks = (uint32_t)std::min<uint64_t>((n + GW_WARPS * 32 - 1) / (GW_WARPS * 32), (uint64_t)c->sm_count * 16);
#define CPB_SC(NC) slot_copy_kernel<NC><<<gblocks, GW_WARPS * 32, 0, c->stream>>>(rs.slots->as<uint8_t>(), rs.S, ids, so, n)
        switch (nc) { case 1: CPB_SC(1); break; case 2: CPB_SC(2); break; case 3: CPB_SC(3); break; default: CPB_SC(4); break; }
#undef CPB_SC
        CPB_CUDA(cudaGetLastError());
    }
    for (int k = 0; k < nc; k++) r->cols.push_back(out[k]);
    return r;
}

// ------------------------------------------------------------------ Filter over a table
struct FilterCols { const uint32_t* off[MAXTERMS]; const uint8_t* data[MAXTERMS]; };

__global__ void filter_flags_kernel(FilterCols cols, PredProg prog, const uint8_t* __restrict__ lits, uint32_t* flags, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t eq = 0;
    for (int t = 0; t < prog.nterms; t++) {
        const uint32_t* off = cols.off[t];
        uint32_t s = off[i], len = off[i + 1] - s;
        if (len != prog.term_len[t]) continue;
        const uint8_t* p = cols.data[t] + s;
        const uint8_t* l = lits + prog.term_off[t];
        bool ok = true;
        for (uint32_t k = 0; k < len; k++) if (p[k] != l[k]) { ok = false; break; }
        if (ok) eq |= 1u << t;
    }
    flags[i] = eval_pred(prog, eq) ? 1u : 0u;
}
__global__ void compact_ids_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos, uint32_t* ids, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i]) ids[pos[i]] = (uint32_t)i;
}

// TakeWhile / DropWhile (csvplus.go:346-374) with a recognisable predicate: the index of the first row for which the
// predicate is FALSE (nrows when there is none) — TakeWhile is then the row range before it, DropWhile the range from it.
__global__ void first_false_kernel(const uint32_t* __restrict__ flags, uint64_t n, unsigned long long* out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i] == 0) atomicMin(out, (unsigned long long)i);
}
int64_t first_false_row(Ctx* c, const Table& t, const cpb_pred* pred) {
    if (!pred) throw ArgError{CPB_ERR_ARG, "nil predicate"};
    Compiled comp;
    compile_pred(pred, [&](const std::string& key) { return t.find(key); }, comp);
    const uint64_t n = (uint64_t)t.nrows;
    if (n == 0) return 0;
    FilterCols fc{};
    for (int i = 0; i < comp.prog.nterms; i++) { fc.off[i] = t.cols[comp.prog.term_col[i]].off(); fc.data[i] = t.cols[comp.prog.term_col[i]].bytes(); }
    Buf lits = dev_alloc(c, comp.lits.size() + 16);
    if (!comp.lits.empty()) CPB_CUDA(cudaMemcpyAsync(lits->p, comp.lits.data(), comp.lits.size(), cudaMemcpyHostToDevice, c->stream));
    Buf flags = dev_alloc(c, n * 4), out = dev_alloc(c, 8);
    CPB_CUDA(cudaMemsetAsync(out->p, 0xff, 8, c->stream));
    {
        KernelTimer kt(c, "filter_like", n * 12, 2);
        filter_flags_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(fc, comp.prog, lits->as<uint8_t>(), flags->as<uint32_t>(), n);
        first_false_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(flags->as<uint32_t>(), n, (unsigned long long*)out->p);
        CPB_CUDA(cudaGetLastError());
    }
    uint64_t* h = (uint64_t*)c->pinned_scratch(8);
    CPB_CUDA(cudaMemcpyAsync(h, out->p, 8, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    return *h == ~0ull ? (int64_t)n : (int64_t)*h;
}

std::shared_ptr<Table> filter_table(Ctx* c, const Table& t, const cpb_pred* pred) {
    if (!pred) throw ArgError{CPB_ERR_ARG, "nil predicate"};
    Compiled comp;
    compile_pred(pred, [&](const std::string& key) { return t.find(key); }, comp);
    const uint64_t n = (uint64_t)t.nrows;
    if (n == 0) return gather_rows(c, t, nullptr, 0);
    FilterCols fc{};
    for (int i = 0; i < comp.prog.nterms; i++) { fc.off[i] = t.cols[comp.prog.term_col[i]].off(); fc.data[i] = t.cols[comp.prog.term_col[i]].bytes(); }
    Buf lits = dev_alloc(c, comp.lits.size() + 16);
    if (!comp.lits.empty()) CPB_CUDA(cudaMemcpyAsync(lits->p, comp.lits.data(), comp.lits.size(), cudaMemcpyHostToDevice, c->stream));
    Buf flags = dev_alloc(c, n * 4), pos = dev_alloc(c, (n + 1) * 4), total = dev_alloc(c, 8);
    {
        KernelTimer kt(c, "filter_like", n * 12);
        filter_flags_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(fc, comp.prog, lits->as<uint8_t>(), flags->as<uint32_t>(), n);
        CPB_CUDA(cudaGetLastError());
    }
    exclusive_scan_u32(c, flags->as<uint32_t>(), pos->as<uint32_t>(), n, total->as<uint64_t>());
    uint64_t* ht = (uint64_t*)c->pinned_scratch(8);
    CPB_CUDA(cudaMemcpyAsync(ht, total->p, 8, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    const uint64_t m = *ht;
    Buf ids = dev_alloc(c, (m + 1) * 4);
    {
        KernelTimer kt(c, "compact_ids", n * 8 + m * 4);
        compact_ids_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(flags->as<uint32_t>(), pos->as<uint32_t>(), ids->as<uint32_t>(), n);
        CPB_CUDA(cudaGetLastError());
    }
    return gather_rows(c, t, ids->as<uint32_t>(), (int64_t)m);
}

// ------------------------------------------------------------------ concat
__global__ void rebase_offsets_kernel(const uint32_t* __restrict__ in, uint32_t* out, uint64_t n, uint32_t add) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) out[i] = in[i] - in[0] + add;  // also writes the sentinel (overwritten by the next part's first entry: same value)
}

std::shared_ptr<Table> concat_tables(Ctx* c, const std::vector<const Table*>& parts) {
    const Table& first = *parts[0];
    for (auto* p : parts) {
        if (p->cols.size() != first.cols.size()) throw ArgError{CPB_ERR_ARG, "concat: column count mismatch"};
        for (size_t k = 0; k < first.cols.size(); k++) if (p->cols[k].name != first.cols[k].name) throw ArgError{CPB_ERR_ARG, "concat: column name mismatch"};
    }
    int64_t nrows = 0;
    for (auto* p : parts) nrows += p->nrows;
    const size_t K = first.cols.size(), NPARTS = parts.size();
    // byte extents of every (part, column): one D2H round trip
    std::vector<uint32_t> ext(2 * K * NPARTS);
    uint32_t* hp = (uint32_t*)c->pinned_scratch(ext.size() * 4);
    for (size_t p = 0; p < NPARTS; p++)
        for (size_t k = 0; k < K; k++) {
            const uint32_t* off = parts[p]->cols[k].off();
            CPB_CUDA(cudaMemcpyAsync(hp + 2 * (p * K + k), off, 4, cudaMemcpyDeviceToHost, c->stream));
            CPB_CUDA(cudaMemcpyAsync(hp + 2 * (p * K + k) + 1, off + parts[p]->nrows, 4, cudaMemcpyDeviceToHost, c->stream));
        }
    sync_stream(c);
    memcpy(ext.data(), hp, ext.size() * 4);
    auto r = std::make_shared<Table>(); r->ctx = c; r->nrows = nrows; r->first_line = first.first_line;
    for (size_t k = 0; k < K; k++) {
        uint64_t total = 0;
        for (size_t p = 0; p < NPARTS; p++) total += ext[2 * (p * K + k) + 1] - ext[2 * (p * K + k)];
        if (total > 0xffffffffull) throw DataError{CPB_E_TOO_LARGE, (int)k, 0, false, "concatenated column exceeds 4 GiB"};
        Column col; col.name = first.cols[k].name;
        col.offsets = dev_alloc(c, ((size_t)nrows + 1) * 4);
        col.data = dev_alloc(c, total + 16);
        uint64_t row = 0, byte = 0;
        for (size_t p = 0; p < NPARTS; p++) {
            uint32_t b0 = ext[2 * (p * K + k)], b1 = ext[2 * (p * K + k) + 1];
            uint64_t pr = (uint64_t)parts[p]->nrows;
            KernelTimer kt(c, "concat", (uint64_t)(b1 - b0) * 2 + pr * 8);
            rebase_offsets_kernel<<<blocks_for(pr + 1, 256), 256, 0, c->stream>>>(parts[p]->cols[k].off(), col.offsets->as<uint32_t>() + row, pr, (uint32_t)byte);
            CPB_CUDA(cudaGetLastError());
            if (b1 > b0) CPB_CUDA(cudaMemcpyAsync(col.data->as<uint8_t>() + byte, parts[p]->cols[k].bytes() + b0, b1 - b0, cudaMemcpyDeviceToDevice, c->stream));
            row += pr; byte += b1 - b0;
        }
        r->cols.push_back(col);
    }
    return r;
}

}  // namespace cpb
