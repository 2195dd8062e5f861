// sort.cu — K5/K6/K7 of SURVEY §2: IndexOn / UniqueIndexOn / ResolveDuplicates.
//
// Replaces (reference): createIndex csvplus.go:707-738 (sort.Sort with indexImpl.Less :794-807),
// createUniqueIndex :740-756 (adjacent equalRows scan), indexImpl.dedup :810-867.
//
// Order = per key column bytewise strings.Compare, columns left to right.  Each row's key is
// packed into an order-preserving fixed-width big-endian image (per column: value zero-padded to
// the column's longest value, then the value length), so comparing images as unsigned integers is
// exactly the reference's comparator (DESIGN.md §index).  The image is sorted with a stable LSD
// radix sort, one 64-bit image word at a time, 8-bit digits, skipping digits that are constant
// over the whole column.  Ties keep input order (the reference's pdqsort is unstable: SURVEY §Q2).
#include <algorithm>

#include "core.hpp"
#include "util.cuh"

namespace cpb {

static inline uint32_t nblk(uint64_t n, int t) { return (uint32_t)((n + t - 1) / t); }


// ------------------------------------------------------------------ key widths
__global__ void max_len_kernel(const uint32_t* __restrict__ off, uint64_t n, uint32_t* out) {
    uint32_t m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        m = max(m, off[i + 1] - off[i]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// ------------------------------------------------------------------ key image
// image[w * n + r] = bytes [8w, 8w+8) of row r's key image, first byte most significant.  A value
// longer than the column width (possible for probe / lookup values only) keeps its first `width`
// bytes and gets the all-ones length, which orders it after every real key sharing those bytes and
// never compares equal.
__global__ void key_pack_kernel(KeyDesc kd, uint64_t n, uint64_t* image) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    uint64_t cur = 0; int cnt = 0; uint32_t word = 0;
    auto push = [&](uint32_t b) {
        cur = (cur << 8) | b;
        if (++cnt == 8) { image[(uint64_t)word * n + r] = cur; word++; cnt = 0; cur = 0; }
    };
    for (int k = 0; k < kd.nkeys; k++) {
        uint32_t s = kd.off[k][r], len = kd.off[k][r + 1] - s;
        const uint8_t* p = kd.data[k] + s;
        uint32_t w = kd.width[k];
        for (uint32_t i = 0; i < w; i++) push(i < len ? p[i] : 0u);
        uint32_t lf = len > w ? 0xffffffffu : len;
        for (int i = (int)kd.lenbytes[k] - 1; i >= 0; i--) push((lf >> (8 * i)) & 0xffu);
    }
    if (cnt) { cur <<= 8 * (8 - cnt); image[(uint64_t)word * n + r] = cur; }
}

// ------------------------------------------------------------------ radix sort of (u64 key, u32 value)
constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 8;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;

__global__ void iota_kernel(uint32_t* p, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = (uint32_t)i;
}
__global__ void gather_u64_kernel(const uint64_t* __restrict__ src, const uint32_t* __restrict__ idx, uint64_t* dst, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}
// histogram of all 8 bytes of every key: hist[b * 256 + v]
__global__ void hist8_kernel(const uint64_t* __restrict__ keys, uint64_t n, uint32_t* hist) {
    __shared__ uint32_t sh[8 * 256];
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t k = keys[i];
#pragma unroll
        for (int b = 0; b < 8; b++) atomicAdd(&sh[b * 256 + ((k >> (8 * b)) & 0xff)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) if (sh[i]) atomicAdd(&hist[i], sh[i]);
}
// per-block digit counts over the block's contiguous tile range: counts[d * nblocks + block]
__global__ void __launch_bounds__(RS_THREADS) radix_count_kernel(const uint64_t* __restrict__ keys, uint64_t n, int shift,
                                                                 uint64_t tiles_per_block, uint32_t* counts) {
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    uint64_t lo = (uint64_t)blockIdx.x * tiles_per_block * RS_TILE;
    uint64_t hi = min(n, lo + tiles_per_block * RS_TILE);
    for (uint64_t i = lo + threadIdx.x; i < hi; i += RS_THREADS) atomicAdd(&sh[(keys[i] >> shift) & 0xff], 1u);
    __syncthreads();
    counts[(uint64_t)threadIdx.x * gridDim.x + blockIdx.x] = sh[threadIdx.x];
}
__global__ void __launch_bounds__(RS_THREADS) radix_scatter_kernel(const uint64_t* __restrict__ kin, const uint32_t* __restrict__ vin,
                                                                   uint64_t* kout, uint32_t* vout, uint64_t n, int shift,
                                                                   uint64_t tiles_per_block, const uint32_t* __restrict__ bases) {
    __shared__ uint32_t cnt[RS_THREADS / 32][256];
    __shared__ uint32_t base[256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    base[tid] = bases[(uint64_t)tid * gridDim.x + blockIdx.x];
    uint64_t lo = (uint64_t)blockIdx.x * tiles_per_block * RS_TILE;
    uint64_t hi = min(n, lo + tiles_per_block * RS_TILE);
    for (uint64_t t0 = lo; t0 < hi; t0 += RS_TILE) {
        for (int i = tid; i < (RS_THREADS / 32) * 256; i += RS_THREADS) (&cnt[0][0])[i] = 0;
        __syncthreads();
        uint64_t k[RS_ITEMS]; uint32_t v[RS_ITEMS], rank[RS_ITEMS];
        const uint64_t wbase = t0 + (uint64_t)warp * 32 * RS_ITEMS;
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            uint64_t idx = wbase + i * 32 + lane;
            bool ok = idx < hi;
            k[i] = ok ? kin[idx] : 0; v[i] = ok ? vin[idx] : 0;
            uint32_t d = ok ? (uint32_t)((k[i] >> shift) & 0xff) : 0x100u;
            uint32_t peers = __match_any_sync(0xffffffffu, d);
            uint32_t pre = ok ? cnt[warp][d] : 0;
            __syncwarp();
            if (ok && lane == __ffs(peers) - 1) cnt[warp][d] = pre + __popc(peers);
            __syncwarp();
            rank[i] = pre + __popc(peers & lanemask_lt());
        }
        __syncthreads();
        {  // thread tid owns digit tid: exclusive prefix over warps, advance the running base
            uint32_t run = base[tid];
#pragma unroll
            for (int w = 0; w < RS_THREADS / 32; w++) { uint32_t c = cnt[w][tid]; cnt[w][tid] = run; run += c; }
            base[tid] = run;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            uint64_t idx = wbase + i * 32 + lane;
            if (idx < hi) {
                uint32_t d = (uint32_t)((k[i] >> shift) & 0xff);
                uint32_t pos = cnt[warp][d] + rank[i];
                kout[pos] = k[i]; vout[pos] = v[i];
            }
        }
        __syncthreads();
    }
}

// Stable sort of `perm` (row ids) by image words [0, words): returns the buffer holding the sorted ids.
// Which digits are constant over the whole column (their pass would be the identity) does not depend on the order of
// the rows: the byte histograms of ALL image words are taken from the unsorted image up front and read back with one
// host round trip for the whole sort (round 1: one per image word).
static Buf sort_by_image(Ctx* c, const uint64_t* image, uint32_t words, uint64_t n, uint64_t* traffic) {
    Buf permA = dev_alloc(c, n * 4), permB = dev_alloc(c, n * 4), keyA = dev_alloc(c, n * 8), keyB = dev_alloc(c, n * 8);
    iota_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(permA->as<uint32_t>(), n);
    const uint64_t ntiles = (n + RS_TILE - 1) / RS_TILE;
    const uint32_t nblocks = (uint32_t)std::min<uint64_t>(ntiles, (uint64_t)c->sm_count * 4);
    const uint64_t tpb = (ntiles + nblocks - 1) / nblocks;
    Buf hist = dev_alloc(c, (size_t)words * 8 * 256 * 4), counts = dev_alloc(c, (256ull * nblocks + 1) * 4), tot = dev_alloc(c, 8);
    CPB_CUDA(cudaMemsetAsync(hist->p, 0, (size_t)words * 8 * 256 * 4, c->stream));
    {
        KernelTimer kt(c, "sort_hist", n * 8 * words, (int)words);
        for (uint32_t w = 0; w < words; w++)
            hist8_kernel<<<c->sm_count * 4, 256, 0, c->stream>>>(image + (uint64_t)w * n, n, hist->as<uint32_t>() + (size_t)w * 8 * 256);
        CPB_CUDA(cudaGetLastError());
    }
    *traffic += n * 8 * words;
    uint32_t* hh = (uint32_t*)c->pinned_scratch((size_t)words * 8 * 256 * 4);
    CPB_CUDA(cudaMemcpyAsync(hh, hist->p, (size_t)words * 8 * 256 * 4, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    std::vector<uint8_t> skip((size_t)words * 8, 0);
    for (uint32_t w = 0; w < words; w++)
        for (int b = 0; b < 8; b++)
            for (int v = 0; v < 256; v++) if (hh[((size_t)w * 8 + b) * 256 + v] == n) skip[(size_t)w * 8 + b] = 1;
    for (int w = (int)words - 1; w >= 0; w--) {
        bool any = false;
        for (int b = 0; b < 8; b++) any = any || !skip[(size_t)w * 8 + b];
        if (!any) continue;  // the whole word is constant
        {
            KernelTimer kt(c, "sort_gather_word", n * 20);
            gather_u64_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(image + (uint64_t)w * n, permA->as<uint32_t>(), keyA->as<uint64_t>(), n);
            CPB_CUDA(cudaGetLastError());
        }
        *traffic += n * 20;
        for (int b = 0; b < 8; b++) {
            if (skip[(size_t)w * 8 + b]) continue;  // every key has the same byte here: the pass would be the identity
            KernelTimer kt(c, "radix_pass", n * 32, 3);
            radix_count_kernel<<<nblocks, RS_THREADS, 0, c->stream>>>(keyA->as<uint64_t>(), n, 8 * b, tpb, counts->as<uint32_t>());
            exclusive_scan_u32(c, counts->as<uint32_t>(), counts->as<uint32_t>(), 256ull * nblocks, tot->as<uint64_t>());
            radix_scatter_kernel<<<nblocks, RS_THREADS, 0, c->stream>>>(keyA->as<uint64_t>(), permA->as<uint32_t>(), keyB->as<uint64_t>(),
                                                                        permB->as<uint32_t>(), n, 8 * b, tpb, counts->as<uint32_t>());
            CPB_CUDA(cudaGetLastError());
            std::swap(keyA, keyB); std::swap(permA, permB);
            *traffic += n * 32;
        }
    }
    return permA;
}

// ------------------------------------------------------------------ adjacent compare (unique check, groups)
// flags[i] = 1 when row i starts a new key (first `pbytes` bytes of the image differ from row i-1)
__device__ __forceinline__ bool image_prefix_equal(const uint64_t* image, uint64_t n, uint64_t a, uint64_t b, uint32_t pbytes) {
    uint32_t full = pbytes >> 3, rem = pbytes & 7;
    for (uint32_t w = 0; w < full; w++) if (image[(uint64_t)w * n + a] != image[(uint64_t)w * n + b]) return false;
    if (rem) {
        uint64_t m = ~0ull << (8 * (8 - rem));
        if ((image[(uint64_t)full * n + a] & m) != (image[(uint64_t)full * n + b] & m)) return false;
    }
    return true;
}
__global__ void head_flags_kernel(const uint64_t* __restrict__ image, uint64_t n, uint32_t pbytes, uint32_t* head) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    head[i] = (i == 0 || !image_prefix_equal(image, n, i, i - 1, pbytes)) ? 1u : 0u;
}
__global__ void first_dup_kernel(const uint32_t* __restrict__ head, uint64_t n, unsigned long long* first) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 1 && i < n && head[i] == 0) atomicMin(first, (unsigned long long)i);
}
// group start: head && next is not head; group end (exclusive hi = i+1): !head && (last || next is head)
__global__ void group_flags_kernel(const uint32_t* __restrict__ head, uint64_t n, uint32_t* gs, uint32_t* ge) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool h = head[i] != 0, nh = (i + 1 == n) || head[i + 1] != 0;
    gs[i] = (h && !nh) ? 1u : 0u;
    ge[i] = (!h && nh) ? 1u : 0u;
}
__global__ void compact_pos_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos, uint32_t* out, uint64_t n, uint32_t add) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i]) out[pos[i]] = (uint32_t)i + add;
}
__global__ void singleton_flags_kernel(const uint32_t* __restrict__ head, uint64_t n, uint32_t* keep) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool h = head[i] != 0, nh = (i + 1 == n) || head[i + 1] != 0;
    keep[i] = (h && nh) ? 1u : 0u;
}
__global__ void set_flags_kernel(const int64_t* __restrict__ rows, uint64_t m, uint32_t* keep, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m && rows[i] >= 0 && (uint64_t)rows[i] < n) keep[rows[i]] = 1u;
}
__global__ void clear_one_kernel(uint32_t* keep, uint64_t i) { keep[i] = 0; }

static uint64_t read_u64(Ctx* c, const void* dev) {
    uint64_t* h = (uint64_t*)c->pinned_scratch(8);
    CPB_CUDA(cudaMemcpyAsync(h, dev, 8, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    return *h;
}

void describe_keys(Ctx* c, const Table& t, const std::vector<int>& kidx, const std::vector<uint32_t>& width, KeyDesc& kd) {
    kd.nkeys = (int)kidx.size();
    uint32_t bytes = 0;
    for (int k = 0; k < kd.nkeys; k++) {
        kd.off[k] = t.cols[kidx[k]].off(); kd.data[k] = t.cols[kidx[k]].bytes();
        kd.width[k] = width[k];
        kd.lenbytes[k] = width[k] < 255 ? 1 : (width[k] < 65535 ? 2 : 4);
        bytes += kd.width[k] + kd.lenbytes[k];
    }
    kd.words = (bytes + 7) / 8;
    (void)c;
}

// bytes of the image covered by the first nk key columns
uint32_t prefix_bytes(const Index& ix, int nk) {
    uint32_t b = 0;
    for (int k = 0; k < nk; k++) b += ix.key_width[k] + (ix.key_width[k] < 255 ? 1 : (ix.key_width[k] < 65535 ? 2 : 4));
    return b;
}

// packs rows of `t` (columns kidx) with the widths of an existing index: probe / lookup images
Buf pack_with_widths(Ctx* c, const Table& t, const std::vector<int>& kidx, const std::vector<uint32_t>& width, uint32_t* words_out) {
    KeyDesc kd{};
    describe_keys(c, t, kidx, width, kd);
    *words_out = kd.words;
    uint64_t n = (uint64_t)t.nrows;
    Buf img = dev_alloc(c, std::max<uint64_t>(1, (uint64_t)kd.words * n) * 8);
    if (n && kd.words) {
        KernelTimer kt(c, "key_pack", n * kd.words * 8);
        key_pack_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(kd, n, img->as<uint64_t>());
        CPB_CUDA(cudaGetLastError());
    }
    return img;
}

static Buf sort_by_image(Ctx* c, const uint64_t* image, uint32_t words, uint64_t n, uint64_t* traffic);
static void ensure_sorted_locked(Ctx* c, Index& ix) {
    if (ix.sorted) return;
    const uint64_t n = (uint64_t)ix.nrows;
    Ctx* prev = c->alloc_for;
    c->alloc_for = ix.ctx;  // what stays inside the index comes from its owner's pool
    try {
        uint64_t traffic = 0;
        Buf perm = sort_by_image(c, ix.uimage->as<uint64_t>(), ix.image_words, n, &traffic);
        Buf simg = dev_alloc(c, std::max<uint64_t>(1, (uint64_t)ix.image_words * n) * 8);
        {
            KernelTimer kt(c, "image_gather", (uint64_t)ix.image_words * n * 20, (int)ix.image_words);
            for (uint32_t w = 0; w < ix.image_words; w++)
                gather_u64_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(ix.uimage->as<uint64_t>() + (uint64_t)w * n, perm->as<uint32_t>(),
                                                                       simg->as<uint64_t>() + (uint64_t)w * n, n);
            CPB_CUDA(cudaGetLastError());
        }
        sync_stream(c);  // complete before another context (stream) can see it
        ix.perm = perm; ix.image = simg; ix.sorted = true;
    } catch (...) { c->alloc_for = prev; throw; }
    c->alloc_for = prev;
}
void ensure_sorted(Ctx* c, Index& ix) {
    std::lock_guard<std::mutex> lk(ix.mu);
    ensure_sorted_locked(c, ix);
}

std::shared_ptr<Table> sorted_table(Ctx* c, Index& ix) {
    std::lock_guard<std::mutex> lk(ix.mu);
    if (ix.table) return ix.table;
    ensure_sorted_locked(c, ix);
    Ctx* prev = c->alloc_for;
    c->alloc_for = ix.ctx;  // the sorted rows stay inside the index: they come from its owner's pool
    try {
        ix.table = gather_rows(c, *ix.src, ix.perm->as<uint32_t>(), ix.nrows);
        ix.table->first_line = 0;  // iterating an Index reports 0-based rows (csvplus.go:243)
        sync_stream(c);  // complete before another context (stream) can see it
    } catch (...) { c->alloc_for = prev; throw; }
    c->alloc_for = prev;
    return ix.table;
}

std::shared_ptr<Index> build_index(Ctx* c, std::shared_ptr<Table> tp, const std::vector<std::string>& keys, bool unique, DataError* derr,
                                   bool* failed) {
    const Table& t = *tp;
    *failed = false;
    if ((int)keys.size() > MAXKEYS) throw ArgError{CPB_ERR_UNSUPPORTED, "more than 16 index key columns"};
    auto ix = std::make_shared<Index>();
    ix->ctx = c; ix->key_cols = keys;
    const uint64_t n = (uint64_t)t.nrows;
    for (size_t k = 0; k < keys.size(); k++) {
        int ci = t.find(keys[k]);
        if (ci < 0) {
            if (n == 0) { ci = -1; }
            else {  // csvplus.go:723-727, raised for the first row pulled
                *failed = true;
                *derr = DataError{CPB_E_MISSING_INDEX_COLUMN, (int)k, t.first_line, true, "missing column " + go_quote(keys[k]) + " while creating an index"};
                return nullptr;
            }
        }
        ix->key_col_idx.push_back(ci);
    }
    if (n == 0) {
        auto e = std::make_shared<Table>(t); e->nrows = 0;
        ix->table = e; ix->src = e; ix->nrows = 0; ix->key_width.assign(keys.size(), 0); ix->image_words = 0; ix->image = dev_alloc(c, 8);
        for (auto& ci : ix->key_col_idx) if (ci < 0) ci = 0;
        return ix;
    }
    if (n > 0xfffffffeull) throw DataError{CPB_E_TOO_LARGE, -1, 0, false, "an index holds at most 2^32-2 rows"};
    // 1. key widths
    Buf wd = dev_alloc(c, keys.size() * 4);
    CPB_CUDA(cudaMemsetAsync(wd->p, 0, keys.size() * 4, c->stream));
    {
        KernelTimer kt(c, "key_width", n * 4 * keys.size(), (int)keys.size());
        for (size_t k = 0; k < keys.size(); k++)
            max_len_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(t.cols[ix->key_col_idx[k]].off(), n, wd->as<uint32_t>() + k);
        CPB_CUDA(cudaGetLastError());
    }
    uint32_t* hw = (uint32_t*)c->pinned_scratch(keys.size() * 4);
    CPB_CUDA(cudaMemcpyAsync(hw, wd->p, keys.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    sync_stream(c);
    ix->key_width.assign(hw, hw + keys.size());
    // 2. image of the unsorted rows.  Its size follows from the widths alone: an oversized key is refused before the
    //    words * n * 8 bytes of the image are allocated and packed.
    KeyDesc kd{};
    describe_keys(c, t, ix->key_col_idx, ix->key_width, kd);
    if ((uint64_t)kd.words * 8 > 4096) throw ArgError{CPB_ERR_UNSUPPORTED, "index keys longer than 4 KiB are not supported"};
    uint32_t words = 0;
    Buf img = pack_with_widths(c, t, ix->key_col_idx, ix->key_width, &words);
    ix->image_words = words;
    // 3a. UniqueIndexOn: the duplicate check does not need the order — a probe table over the rows as they are, in which
    //     every key must find itself.  When it passes (the usual case) the sort is left for whoever needs the order.
    static const bool eager = getenv("CPB_EAGER_SORT") != nullptr;
    if (unique && n >= 2 && !eager) {
        ix->src = tp; ix->nrows = (int64_t)n; ix->uimage = img; ix->sorted = false; ix->unique = true;
        if (!index_has_duplicates(c, *ix)) return ix;
        // a duplicate exists: sort, so that the error names the key the reference would name (the lowest in sort order)
        ix->unique = false; ix->sorted = true; ix->uimage = nullptr; ix->hash_src.clear(); ix->row_slots_src.clear();
    }
    // 3. stable LSD radix sort -> permutation
    uint64_t traffic = 0;
    Buf perm = sort_by_image(c, img->as<uint64_t>(), words, n, &traffic);
    // 4. the sorted key image; the sorted rows themselves stay virtual (src + perm) until something needs them
    ix->src = tp; ix->perm = perm; ix->nrows = (int64_t)n;
    Buf simg = dev_alloc(c, std::max<uint64_t>(1, (uint64_t)words * n) * 8);
    {
        KernelTimer kt(c, "image_gather", (uint64_t)words * n * 20, (int)words);
        for (uint32_t w = 0; w < words; w++)
            gather_u64_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(img->as<uint64_t>() + (uint64_t)w * n, perm->as<uint32_t>(),
                                                                   simg->as<uint64_t>() + (uint64_t)w * n, n);
        CPB_CUDA(cudaGetLastError());
    }
    ix->image = simg;
    // 5. uniqueness (createUniqueIndex, csvplus.go:740-756)
    if (unique && n >= 2) {
        Buf head = dev_alloc(c, n * 4), first = dev_alloc(c, 8);
        CPB_CUDA(cudaMemsetAsync(first->p, 0xff, 8, c->stream));
        {
            KernelTimer kt(c, "unique_check", (uint64_t)words * n * 8, 2);
            head_flags_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(simg->as<uint64_t>(), n, words * 8, head->as<uint32_t>());
            first_dup_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(head->as<uint32_t>(), n, (unsigned long long*)first->p);
            CPB_CUDA(cudaGetLastError());
        }
        uint64_t fd = read_u64(c, first->p);
        if (fd != ~0ull) {
            // "duplicate value while creating unique index: " + rows[i].SelectExisting(columns...).String()  (:751, :90-104)
            std::vector<std::pair<std::string, std::string>> kv;
            for (size_t k = 0; k < keys.size(); k++) {
                const Column& col = sorted_table(c, *ix)->cols[ix->key_col_idx[k]];
                uint32_t oo[2];
                CPB_CUDA(cudaMemcpyAsync(oo, col.off() + fd, 8, cudaMemcpyDeviceToHost, c->stream));
                sync_stream(c);
                std::string v(oo[1] - oo[0], '\0');
                if (!v.empty()) CPB_CUDA(cudaMemcpyAsync(&v[0], col.bytes() + oo[0], v.size(), cudaMemcpyDeviceToHost, c->stream));
                sync_stream(c);
                kv.emplace_back(keys[k], v);
            }
            std::sort(kv.begin(), kv.end());
            std::string s = "{ ";
            for (size_t i = 0; i < kv.size(); i++) { if (i) s += ", "; s += "\"" + kv[i].first + "\" : \"" + kv[i].second + "\""; }
            s += " }";
            *failed = true;
            *derr = DataError{CPB_E_DUPLICATE_KEY, -1, 0, false, "duplicate value while creating unique index: " + s};
            return nullptr;
        }
    }
    ix->unique = unique;
    return ix;
}

// ------------------------------------------------------------------ ResolveDuplicates support
static Buf compact_flags(Ctx* c, const uint32_t* flags, uint64_t n, uint32_t add, uint64_t* count) {
    Buf pos = dev_alloc(c, (n + 1) * 4), tot = dev_alloc(c, 8);
    exclusive_scan_u32(c, flags, pos->as<uint32_t>(), n, tot->as<uint64_t>());
    *count = read_u64(c, tot->p);
    Buf out = dev_alloc(c, (*count + 1) * 4);
    if (n) compact_pos_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(flags, pos->as<uint32_t>(), out->as<uint32_t>(), n, add);
    CPB_CUDA(cudaGetLastError());
    return out;
}

void index_dup_groups(Ctx* c, Index& ix, std::vector<int64_t>& lo, std::vector<int64_t>& hi) {
    lo.clear(); hi.clear();
    const uint64_t n = (uint64_t)ix.nrows;
    if (n < 2 || ix.unique) return;  // (a verified unique index has no duplicate group)
    Buf head = dev_alloc(c, n * 4), gs = dev_alloc(c, n * 4), ge = dev_alloc(c, n * 4);
    {
        KernelTimer kt(c, "dedup_segments", (uint64_t)ix.image_words * n * 8 + n * 12, 2);
        head_flags_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(ix.image->as<uint64_t>(), n, ix.image_words * 8, head->as<uint32_t>());
        group_flags_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(head->as<uint32_t>(), n, gs->as<uint32_t>(), ge->as<uint32_t>());
        CPB_CUDA(cudaGetLastError());
    }
    uint64_t ng = 0, ne = 0;
    Buf los = compact_flags(c, gs->as<uint32_t>(), n, 0, &ng);
    Buf his = compact_flags(c, ge->as<uint32_t>(), n, 1, &ne);
    if (ng != ne) throw ArgError{CPB_ERR_CUDA, "internal: group start/end mismatch"};
    std::vector<uint32_t> a(ng), b(ng);
    if (ng) {
        CPB_CUDA(cudaMemcpyAsync(a.data(), los->p, ng * 4, cudaMemcpyDeviceToHost, c->stream));
        CPB_CUDA(cudaMemcpyAsync(b.data(), his->p, ng * 4, cudaMemcpyDeviceToHost, c->stream));
        sync_stream(c);
    }
    lo.assign(a.begin(), a.end()); hi.assign(b.begin(), b.end());
}

// indexImpl.dedup (csvplus.go:810-867) with the resolver's choices already made on the host.
// keep[g] >= 0: sorted position of the row kept for group g; -1: the group is dropped (the resolver returned an "empty"
// row, :845); <= -2: the resolver returned a row that is not one of the group's rows — row (-2 - keep[g]) of `repl`
// takes the place of the group (:846 stores whatever row came back; the index is NOT re-sorted, exactly like the reference).
__global__ void patch_ids_kernel(const uint32_t* __restrict__ pos, const int64_t* __restrict__ at, const uint32_t* __restrict__ with, uint64_t m, uint32_t* ids) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) ids[pos[at[i]]] = with[i];
}

void index_dedup_apply(Ctx* c, Index& ix, const std::vector<int64_t>& keep_in, bool bug_compatible, const Table* repl) {
    const uint64_t n = (uint64_t)ix.nrows;
    if (n < 2 || keep_in.empty()) return;  // no duplicate group: the reference returns early (:820-822)
    sorted_table(c, ix);
    std::vector<int64_t> keep = keep_in;
    // groups answered with a replacement row keep their first position as the slot the new row goes to
    std::vector<int64_t> rpos; std::vector<uint32_t> rid;
    bool any_repl = false;
    for (auto k : keep) if (k <= -2) any_repl = true;
    if (any_repl) {
        if (!repl) throw ArgError{CPB_ERR_ARG, "replacement rows referenced but no replacement table given"};
        if (repl->cols.size() != ix.table->cols.size()) throw ArgError{CPB_ERR_UNSUPPORTED, "a replacement row must have the columns of the index rows"};
        for (auto& col : ix.table->cols) if (repl->find(col.name) < 0) throw ArgError{CPB_ERR_UNSUPPORTED, "a replacement row must have the columns of the index rows"};
        std::vector<int64_t> lo, hi;
        index_dup_groups(c, ix, lo, hi);
        if (lo.size() != keep.size()) throw ArgError{CPB_ERR_ARG, "keep[] does not match the duplicate groups of the index"};
        for (size_t g = 0; g < keep.size(); g++)
            if (keep[g] <= -2) {
                const int64_t j = -2 - keep[g];
                if (j >= repl->nrows) throw ArgError{CPB_ERR_ARG, "replacement row out of range"};
                rpos.push_back(lo[g]); rid.push_back((uint32_t)(n + (uint64_t)j));
                keep[g] = lo[g];
            }
    }
    Buf head = dev_alloc(c, n * 4), flag = dev_alloc(c, n * 4);
    head_flags_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(ix.image->as<uint64_t>(), n, ix.image_words * 8, head->as<uint32_t>());
    singleton_flags_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(head->as<uint32_t>(), n, flag->as<uint32_t>());
    Buf kd = dev_alloc(c, keep.size() * 8);
    CPB_CUDA(cudaMemcpyAsync(kd->p, keep.data(), keep.size() * 8, cudaMemcpyHostToDevice, c->stream));
    set_flags_kernel<<<nblk(keep.size(), 256), 256, 0, c->stream>>>(kd->as<int64_t>(), keep.size(), flag->as<uint32_t>(), n);
    if (bug_compatible) {
        // SURVEY §Q1: when a group exists and the last sorted row is a singleton it is never copied (:851-864)
        uint32_t hl[2];
        CPB_CUDA(cudaMemcpyAsync(&hl[0], head->as<uint32_t>() + (n - 1), 4, cudaMemcpyDeviceToHost, c->stream));
        sync_stream(c);
        if (hl[0] != 0) clear_one_kernel<<<1, 1, 0, c->stream>>>(flag->as<uint32_t>(), n - 1);
    }
    CPB_CUDA(cudaGetLastError());
    // compaction of the kept positions (the scanned positions are needed again to patch replacement ids in)
    Buf pos = dev_alloc(c, (n + 1) * 4), tot = dev_alloc(c, 8);
    exclusive_scan_u32(c, flag->as<uint32_t>(), pos->as<uint32_t>(), n, tot->as<uint64_t>());
    const uint64_t m = read_u64(c, tot->p);
    Buf ids = dev_alloc(c, (m + 1) * 4);
    compact_pos_kernel<<<nblk(n, 256), 256, 0, c->stream>>>(flag->as<uint32_t>(), pos->as<uint32_t>(), ids->as<uint32_t>(), n, 0);
    CPB_CUDA(cudaGetLastError());
    std::shared_ptr<Table> nt;
    if (!rpos.empty()) {
        Buf dp = dev_alloc(c, rpos.size() * 8), dr = dev_alloc(c, rid.size() * 4);
        CPB_CUDA(cudaMemcpyAsync(dp->p, rpos.data(), rpos.size() * 8, cudaMemcpyHostToDevice, c->stream));
        CPB_CUDA(cudaMemcpyAsync(dr->p, rid.data(), rid.size() * 4, cudaMemcpyHostToDevice, c->stream));
        patch_ids_kernel<<<nblk(rpos.size(), 256), 256, 0, c->stream>>>(pos->as<uint32_t>(), dp->as<int64_t>(), dr->as<uint32_t>(), rpos.size(), ids->as<uint32_t>());
        CPB_CUDA(cudaGetLastError());
        // rows [0, n) = the index, rows [n, n + repl) = the replacement rows in the index's column order
        Table rsel; rsel.ctx = c; rsel.nrows = repl->nrows;
        for (auto& col : ix.table->cols) rsel.cols.push_back(repl->cols[repl->find(col.name)]);
        auto both = concat_tables(c, {ix.table.get(), &rsel});
        nt = gather_rows(c, *both, ids->as<uint32_t>(), (int64_t)m);
        sync_stream(c);  // rpos / rid are pageable host vectors
        // keys may have changed (even their widths): the image is rebuilt from the new rows, their order is kept
        nt->first_line = 0;
        ix.table = nt; ix.src = nullptr; ix.perm = nullptr; ix.nrows = (int64_t)m; ix.unique = false;
        for (size_t k = 0; k < ix.key_cols.size(); k++) ix.key_col_idx[k] = nt->find(ix.key_cols[k]);
        Buf wd = dev_alloc(c, ix.key_cols.size() * 4);
        CPB_CUDA(cudaMemsetAsync(wd->p, 0, ix.key_cols.size() * 4, c->stream));
        for (size_t k = 0; k < ix.key_cols.size() && m; k++)
            max_len_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(nt->cols[ix.key_col_idx[k]].off(), m, wd->as<uint32_t>() + k);
        uint32_t* hw = (uint32_t*)c->pinned_scratch(ix.key_cols.size() * 4);
        CPB_CUDA(cudaMemcpyAsync(hw, wd->p, ix.key_cols.size() * 4, cudaMemcpyDeviceToHost, c->stream));
        sync_stream(c);
        ix.key_width.assign(hw, hw + ix.key_cols.size());
        uint32_t words = 0;
        ix.image = pack_with_widths(c, *nt, ix.key_col_idx, ix.key_width, &words);
        ix.image_words = words;
        ix.hash.clear(); ix.row_slots.clear();
        return;
    }
    nt = gather_rows(c, *ix.table, ids->as<uint32_t>(), (int64_t)m);
    Buf simg = dev_alloc(c, std::max<uint64_t>(1, (uint64_t)ix.image_words * m) * 8);
    for (uint32_t w = 0; w < ix.image_words && m; w++)
        gather_u64_kernel<<<nblk(m, 256), 256, 0, c->stream>>>(ix.image->as<uint64_t>() + (uint64_t)w * n, ids->as<uint32_t>(),
                                                               simg->as<uint64_t>() + (uint64_t)w * m, m);
    CPB_CUDA(cudaGetLastError());
    nt->first_line = 0;
    ix.table = nt; ix.src = nullptr; ix.perm = nullptr; ix.nrows = (int64_t)m;
    ix.image = simg; ix.hash.clear(); ix.row_slots.clear();
}

}  // namespace cpb
