// The evaluation cache of sc_set_eval_cache: stored results of sc_predict* leaves, keyed on the packed leaf exactly as
// the device kernels read it (the 544-byte sc_position row) and its ep byte.  An output of predict_launch is a pure
// function of that key, so a stored result is bit-identical to a fresh evaluation.
//
// The table: n_buckets buckets of CACHE_WAYS entries.  Per entry a 64-bit hash of its key (0 = empty), a stamp (the
// number of the last call that hit it or claimed it) and the entry itself.  A call is two kernels around the network:
//   cache_probe_kernel  sorts the n leaves into hits, in-call duplicates and misses, compacts the misses and claims
//                       their insert targets (never an entry a hit of the same call reads);
//   cache_finish_kernel assembles the n-row outputs from the entries, the misses' results and the duplicates' owners,
//                       then stores the misses' results into their claimed entries.
#include <climits>

#include "common.cuh"

namespace scb {

namespace {

constexpr int KEY_WORDS = sizeof(sc_position) / 8;  // 68
static_assert(sizeof(sc_position) == KEY_WORDS * 8, "sc_position is read as 64-bit words");
constexpr int PROBE_THREADS = 1024;
constexpr int PROBE_WARPS = PROBE_THREADS / 32;
constexpr int FINISH_WARPS = 8;

struct CacheEntry {
    uint64_t key[KEY_WORDS];  // the sc_position row
    int32_t cnt, term;
    float value;
    int32_t ep;  // the ep byte (-1 for none)
    uint32_t moves[SC_MAX_MOVES];  // sc_move bytes; the first min(cnt, SC_MAX_MOVES) are stored
    float priors[SC_MAX_MOVES];
};

__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// a key's words as lane `lane` of a warp holds them: words lane, lane + 32 and (lanes 0..3) lane + 64
struct KeyPart {
    uint64_t w[3];
};

__device__ __forceinline__ KeyPart load_key(const uint64_t *row, int lane)
{
    KeyPart k;
    k.w[0] = row[lane];
    k.w[1] = row[lane + 32];
    k.w[2] = lane + 64 < KEY_WORDS ? row[lane + 64] : 0;
    return k;
}

// a nonzero 64-bit hash of (key, ep), the same in every lane: each word is mixed with its index and the mixes summed
__device__ __forceinline__ uint64_t warp_hash(const KeyPart &k, int ep, int lane)
{
    constexpr uint64_t G = 0x9e3779b97f4a7c15ull;
    uint64_t h = mix64(k.w[0] + G * (lane + 1)) + mix64(k.w[1] + G * (lane + 33));
    if (lane + 64 < KEY_WORDS) h += mix64(k.w[2] + G * (lane + 65));
    for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
    return (h + mix64((uint64_t)(uint32_t)ep + G * (KEY_WORDS + 1))) | 1ull;
}

__device__ __forceinline__ bool warp_equal(const KeyPart &k, const uint64_t *row, int lane)
{
    bool eq = k.w[0] == row[lane] && k.w[1] == row[lane + 32];
    if (lane + 64 < KEY_WORDS) eq = eq && k.w[2] == row[lane + 64];
    return __all_sync(0xffffffffu, eq);
}

__device__ __forceinline__ int leaf_ep(const int8_t *ep, int i) { return ep ? ep[i] : -1; }

// the first entry of the bucket of hash h.  Bit 0 of every hash is 1 (0 marks an empty entry), so the bucket comes from
// the other 63 bits: with an even bucket count, h itself would reach only the odd buckets
__device__ __forceinline__ int64_t bucket_of(uint64_t h, int64_t n_buckets)
{
    return (int64_t)((h >> 1) % (uint64_t)n_buckets) * CACHE_WAYS;
}

__device__ __forceinline__ int dedup_slot(uint64_t h, int mask) { return (int)((h ^ (h >> 29)) & (uint64_t)mask); }

struct ProbeArgs {
    const sc_position *pos;
    const int8_t *ep;
    int n;
    const CacheEntry *ent;
    uint64_t *hash;
    unsigned long long *stamp;
    int64_t n_buckets;
    unsigned long long call;  // this call's stamp
    uint64_t *row_hash;
    int32_t *row_src, *row_owner, *miss_row, *claim;
    unsigned long long *dedup_key;
    int32_t *dedup_row;
    uint64_t *miss_pos;
    int8_t *miss_ep;
    int32_t *counts;  // pinned: misses, hits, duplicates, inserts, evictions
};

// One CTA.  row_owner[i]: -1 for a hit, else the lowest row with the same key (i itself for a miss).  row_src[i]: the
// miss index j of a miss or a duplicate (its owner is miss j), -(entry + 1) for a hit.  The misses' rows, positions and
// ep bytes go to miss_row / miss_pos / miss_ep in row order, each miss's insert target (or -1) to claim.
__global__ void __launch_bounds__(PROBE_THREADS) cache_probe_kernel(ProbeArgs a)
{
    __shared__ int s_cnt[4];  // hits, duplicates, inserts, evictions
    __shared__ int s_scan[PROBE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n = a.n;
    int dmask = 1;
    while (dmask < 2 * n) dmask <<= 1;
    dmask -= 1;
    for (int t = threadIdx.x; t <= dmask; t += PROBE_THREADS) {
        a.dedup_key[t] = 0;
        a.dedup_row[t] = INT_MAX;
    }
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    __syncthreads();

    // 1. hash every leaf and probe its bucket, confirming a way whose hash matches on all 545 bytes.  A hit stamps its
    //    entry with this call, which keeps the entry from being claimed in step 4; the other leaves enter the in-call
    //    table, which keeps per hash the lowest row
    for (int i = warp; i < n; i += PROBE_WARPS) {
        const KeyPart k = load_key(reinterpret_cast<const uint64_t *>(a.pos + i), lane);
        const int ep = leaf_ep(a.ep, i);
        const uint64_t h = warp_hash(k, ep, lane);
        const int64_t b = bucket_of(h, a.n_buckets);
        const uint64_t wh = lane < CACHE_WAYS ? a.hash[b + lane] : 0;
        unsigned cand = __ballot_sync(0xffffffffu, lane < CACHE_WAYS && wh == h);
        int hit = -1;
        while (cand && hit < 0) {
            const int64_t e = b + __ffs(cand) - 1;
            cand &= cand - 1;
            if (warp_equal(k, a.ent[e].key, lane) && a.ent[e].ep == ep) hit = (int)e;
        }
        if (lane == 0) {
            a.row_hash[i] = h;
            a.row_owner[i] = hit >= 0 ? -1 : i;
            if (hit >= 0) {
                a.row_src[i] = -(hit + 1);
                a.stamp[hit] = a.call;
                atomicAdd(&s_cnt[0], 1);
            } else {
                for (int s = dedup_slot(h, dmask);; s = (s + 1) & dmask) {
                    const unsigned long long prev = atomicCAS(a.dedup_key + s, 0ull, (unsigned long long)h);
                    if (prev == 0 || prev == h) {
                        atomicMin(a.dedup_row + s, i);
                        break;
                    }
                }
            }
        }
    }
    __syncthreads();

    // 2. a leaf that is not a hit duplicates the lowest row of its hash if their keys are equal; else it is a miss (a
    //    64-bit hash collision costs an evaluation, never a wrong answer)
    for (int i = warp; i < n; i += PROBE_WARPS) {
        if (a.row_owner[i] < 0) continue;
        const uint64_t h = a.row_hash[i];
        int first = i;
        if (lane == 0) {
            int s = dedup_slot(h, dmask);
            while (a.dedup_key[s] != h) s = (s + 1) & dmask;
            first = a.dedup_row[s];
        }
        first = __shfl_sync(0xffffffffu, first, 0);
        if (first == i) continue;
        const KeyPart k = load_key(reinterpret_cast<const uint64_t *>(a.pos + i), lane);
        if (warp_equal(k, reinterpret_cast<const uint64_t *>(a.pos + first), lane) &&
            leaf_ep(a.ep, i) == leaf_ep(a.ep, first) && lane == 0)
            a.row_owner[i] = first;
    }
    __syncthreads();

    // 3. the misses in row order: thread t takes rows [t * per, (t + 1) * per), an exclusive scan gives its first index
    const int per = (n + PROBE_THREADS - 1) / PROBE_THREADS, r0 = min(n, (int)threadIdx.x * per), r1 = min(n, r0 + per);
    int mine = 0;
    for (int i = r0; i < r1; i++) mine += a.row_owner[i] == i;
    int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_scan[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_scan[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += v;
        }
        s_scan[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int m = s_scan[PROBE_WARPS - 1];
    for (int i = r0, j = (warp ? s_scan[warp - 1] : 0) + incl - mine; i < r1; i++) {
        if (a.row_owner[i] != i) continue;
        a.miss_row[j] = i;
        a.row_src[i] = j++;
    }
    __syncthreads();

    // 4. duplicates take their owner's miss index; each miss copies its leaf and claims an insert target in its bucket:
    //    an empty way first, else the least recently used, never one stamped with this call (a hit of this call reads
    //    it, or another miss claimed it).  If every way is, the result is not stored
    for (int i = threadIdx.x; i < n; i += PROBE_THREADS) {
        const int o = a.row_owner[i];
        if (o < 0 || o == i) continue;
        a.row_src[i] = a.row_src[o];
        atomicAdd(&s_cnt[1], 1);
    }
    for (int j = warp; j < m; j += PROBE_WARPS) {
        const int i = a.miss_row[j];
        const uint64_t *src = reinterpret_cast<const uint64_t *>(a.pos + i);
        for (int w = lane; w < KEY_WORDS; w += 32) a.miss_pos[(size_t)j * KEY_WORDS + w] = src[w];
        if (lane != 0) continue;
        if (a.ep) a.miss_ep[j] = a.ep[i];
        const int64_t b = bucket_of(a.row_hash[i], a.n_buckets);
        volatile unsigned long long *stamp = a.stamp + b;
        volatile uint64_t *hash = a.hash + b;
        int got = -1;
        for (;;) {
            int best = -1;
            bool best_empty = false;
            unsigned long long best_stamp = 0;
            for (int w = 0; w < CACHE_WAYS; w++) {
                const unsigned long long s = stamp[w];
                if (s == a.call) continue;
                const bool empty = hash[w] == 0;
                if (best < 0 || (empty && !best_empty) || (empty == best_empty && s < best_stamp)) {
                    best = w;
                    best_empty = empty;
                    best_stamp = s;
                }
            }
            if (best < 0) break;
            if (atomicCAS(a.stamp + b + best, best_stamp, a.call) == best_stamp) {
                got = (int)(b + best);
                hash[best] = 0;  // invalid until the finish kernel has stored the new result
                atomicAdd(&s_cnt[2], 1);
                if (!best_empty) atomicAdd(&s_cnt[3], 1);
                break;
            }
        }
        a.claim[j] = got;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a.counts[0] = m;
        for (int c = 0; c < 4; c++) a.counts[1 + c] = s_cnt[c];
    }
}

struct FinishArgs {
    int n, m;
    CacheEntry *ent;
    uint64_t *hash;
    const uint64_t *row_hash;
    const int32_t *row_src, *miss_row, *claim;
    const uint64_t *miss_pos;
    const int8_t *miss_ep;
    const uint8_t *miss_out;  // the misses' moves [m][SC_MAX_MOVES], counts [m], termination codes [m]
    const float *miss_priors, *miss_value;
    uint8_t *out;  // the same layout for the n leaves
    float *priors, *value;
};

// one warp per leaf: its row of the outputs, then, for a miss with an insert target, the stored entry
__global__ void __launch_bounds__(FINISH_WARPS * 32) cache_finish_kernel(FinishArgs a)
{
    const int lane = threadIdx.x & 31, i = blockIdx.x * FINISH_WARPS + (threadIdx.x >> 5);
    if (i >= a.n) return;
    const uint32_t *miss_mv = reinterpret_cast<const uint32_t *>(a.miss_out);
    const int32_t *miss_cnt = reinterpret_cast<const int32_t *>(a.miss_out + sizeof(sc_move) * SC_MAX_MOVES * (size_t)a.m);
    uint32_t *out_mv = reinterpret_cast<uint32_t *>(a.out);
    int32_t *out_cnt = reinterpret_cast<int32_t *>(a.out + sizeof(sc_move) * SC_MAX_MOVES * (size_t)a.n);
    const int src = a.row_src[i];
    const uint32_t *mv;
    const float *pr;
    int cnt, term, ep = -1;
    float val;
    if (src >= 0) {
        mv = miss_mv + (size_t)src * SC_MAX_MOVES;
        pr = a.miss_priors + (size_t)src * SC_MAX_MOVES;
        cnt = miss_cnt[src];
        term = miss_cnt[a.m + src];
        val = a.miss_value[src];
    } else {
        const CacheEntry &E = a.ent[-src - 1];
        mv = E.moves;
        pr = E.priors;
        cnt = E.cnt;
        term = E.term;
        val = E.value;
    }
    const int c = min(max(cnt, 0), SC_MAX_MOVES);
    for (int k = lane; k < c; k += 32) {
        out_mv[(size_t)i * SC_MAX_MOVES + k] = mv[k];
        a.priors[(size_t)i * SC_MAX_MOVES + k] = pr[k];
    }
    if (lane == 0) {
        out_cnt[i] = cnt;
        out_cnt[a.n + i] = term;
        a.value[i] = val;
    }
    if (src < 0 || a.miss_row[src] != i || a.claim[src] < 0) return;
    const int e = a.claim[src];
    CacheEntry &E = a.ent[e];
    for (int w = lane; w < KEY_WORDS; w += 32) E.key[w] = a.miss_pos[(size_t)src * KEY_WORDS + w];
    for (int k = lane; k < c; k += 32) {
        E.moves[k] = mv[k];
        E.priors[k] = pr[k];
    }
    if (a.miss_ep) ep = a.miss_ep[src];
    if (lane == 0) {
        E.cnt = cnt;
        E.term = term;
        E.value = val;
        E.ep = ep;
        a.hash[e] = a.row_hash[i];
    }
}

}  // namespace

size_t eval_cache_entry_bytes() { return sizeof(CacheEntry); }

int eval_cache_create(EvalCache *c, int64_t entries, int max_batch, cudaStream_t st)
{
    const int64_t n_buckets = (entries + CACHE_WAYS - 1) / CACHE_WAYS, cap = n_buckets * CACHE_WAYS;
    int dedup = 1;
    while (dedup < 2 * max_batch) dedup <<= 1;
    const size_t rows = (size_t)max_batch;
    auto alloc = [](auto **p, size_t count) {
        *p = nullptr;
        return cudaMalloc(reinterpret_cast<void **>(p), count * sizeof(**p));
    };
    SCB_CUDA(cudaMalloc(&c->ent, sizeof(CacheEntry) * (size_t)cap));
    SCB_CUDA(alloc(&c->hash, (size_t)cap));
    SCB_CUDA(alloc(&c->stamp, (size_t)cap));
    SCB_CUDA(cudaMemsetAsync(c->hash, 0, sizeof(uint64_t) * (size_t)cap, st));
    SCB_CUDA(cudaMemsetAsync(c->stamp, 0, sizeof(unsigned long long) * (size_t)cap, st));
    SCB_CUDA(alloc(&c->row_hash, rows));
    SCB_CUDA(alloc(&c->row_src, rows));
    SCB_CUDA(alloc(&c->row_owner, rows));
    SCB_CUDA(alloc(&c->miss_row, rows));
    SCB_CUDA(alloc(&c->claim, rows));
    SCB_CUDA(alloc(&c->dedup_key, (size_t)dedup));
    SCB_CUDA(alloc(&c->dedup_row, (size_t)dedup));
    SCB_CUDA(alloc(&c->miss_pos, rows));
    SCB_CUDA(alloc(&c->miss_ep, rows));
    SCB_CUDA(alloc(&c->miss_out, rows * (sizeof(sc_move) * SC_MAX_MOVES + 2 * sizeof(int32_t))));
    SCB_CUDA(alloc(&c->miss_priors, rows * SC_MAX_MOVES));
    SCB_CUDA(alloc(&c->miss_value, rows));
    SCB_CUDA(cudaMallocHost(&c->h_counts, sizeof(int32_t) * 5));
    SCB_CUDA(cudaStreamSynchronize(st));
    c->n_buckets = n_buckets;
    c->entries = cap;
    c->calls = 0;
    return SC_OK;
}

void eval_cache_release(EvalCache *c)
{
    for (void *p : {(void *)c->ent, (void *)c->hash, (void *)c->stamp, (void *)c->row_hash, (void *)c->row_src,
                    (void *)c->row_owner, (void *)c->miss_row, (void *)c->claim, (void *)c->dedup_key,
                    (void *)c->dedup_row, (void *)c->miss_pos, (void *)c->miss_ep, (void *)c->miss_out,
                    (void *)c->miss_priors, (void *)c->miss_value})
        if (p) cudaFree(p);
    if (c->h_counts) cudaFreeHost(c->h_counts);
    *c = EvalCache{};
}

int launch_cache_probe(EvalCache *c, const sc_position *d_pos, const int8_t *d_ep, int n, cudaStream_t st)
{
    ProbeArgs a{d_pos, d_ep, n, static_cast<const CacheEntry *>(c->ent), c->hash, c->stamp, c->n_buckets, ++c->calls,
                c->row_hash, c->row_src, c->row_owner, c->miss_row, c->claim, c->dedup_key, c->dedup_row,
                reinterpret_cast<uint64_t *>(c->miss_pos), c->miss_ep, c->h_counts};
    cache_probe_kernel<<<1, PROBE_THREADS, 0, st>>>(a);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_cache_finish(const EvalCache *c, int n, int m, bool ep, uint8_t *d_out, float *d_priors, float *d_value,
                        cudaStream_t st)
{
    FinishArgs a{n, m, static_cast<CacheEntry *>(c->ent), c->hash, c->row_hash, c->row_src, c->miss_row, c->claim,
                 reinterpret_cast<const uint64_t *>(c->miss_pos), ep ? c->miss_ep : nullptr, c->miss_out,
                 c->miss_priors, c->miss_value, d_out, d_priors, d_value};
    cache_finish_kernel<<<(n + FINISH_WARPS - 1) / FINISH_WARPS, FINISH_WARPS * 32, 0, st>>>(a);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

}  // namespace scb
