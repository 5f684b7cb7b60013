// Occupancy loss (loss/occupancy_loss.py:102-149 of the reference with the shipped configs' options): weighted
// cross-entropy + Lovász-softmax over ONE pooled set of B*N points, forward value and gradient w.r.t. the logits
// (or probabilities), with no host synchronisation.  Semantics: include/gf_b200.h (gf_occ_loss_desc); design and
// measurements: DESIGN.md §4.6.
//
// Pipeline (all on the caller's stream; every launch geometry depends on the shape only, never on the data):
//   occ_rows      per 1024-row CTA: CE partial sums (fp64), Lovász-set size, per-class foreground counts, status bits
//   occ_setup     1 CTA: scan of the set sizes -> compaction offsets and M; foreground totals g[c] -> present classes;
//                 CE numerator / denominator in a fixed order; status word
//   occ_compact   stable compaction of the Lovász set; one 30-bit key per (present class, element):
//                 0x3F800000 - bits(e) sorts the errors e in [0, 1] in descending order; payload = index | fg << 31
//   3 x (occ_sort_hist, occ_sort_scan, occ_sort_scatter)
//                 stable LSD radix sort, 10 bits per pass, every present class one segment of M keys
//   occ_lov_count / occ_lov_scan
//                 foreground counts per sorted tile, then the closed-form Lovász gradient per sorted position,
//                 e * dJ summed in fp64 per tile, dL/dq scattered to a class-major [C, M] buffer
//   occ_final     1 CTA: [total, ce, lovasz] and the two gradient scales
//   occ_grad      dL/dpred per row (softmax Jacobian product + CE gradient, or the probability-mode terms)
#include <cstdint>

#include "common.cuh"

namespace gf {

namespace {

constexpr int kRowThreads = 256;
constexpr int kRowsPerCta = 1024;          // occ_rows / occ_compact: 4 rounds of 256 rows
constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortTile = 4096;            // keys per sort CTA: 8 warps x 512 consecutive keys
constexpr int kPerWarp = kSortTile / kSortWarps;
constexpr int kRadixBits = 10;
constexpr int kBins = 1 << kRadixBits;
constexpr int kLovTile = 4096;             // sorted keys per occ_lov_* CTA: 256 threads x 16
constexpr int kLovPerThread = kLovTile / kRowThreads;
constexpr int kMaxC = 32;
constexpr uint32_t kOne = 0x3F800000u;     // bits of 1.0f
constexpr uint32_t kFgBit = 0x80000000u;

struct OccGlobals {
    int32_t M;                 // size of the Lovász set
    int32_t npresent;
    int32_t present[kMaxC];
    int32_t g[kMaxC];          // foreground count per class
    double ce_num, ce_den;     // sum w[y] * nll, sum w[y]
    double ce_scale;           // ce_weight / ce_den
    double lov_scale;          // lovasz_weight / npresent (0 without a present class)
};

struct OccPlan {
    long long T;               // B * N rows
    int row_ctas;
    int sort_tiles;            // key tiles per segment for M = T (upper bound; CTAs past M exit)
    int lov_tiles;
    double *cta_ce;            // [row_ctas, 2]
    int32_t *cta_cnt;          // [row_ctas]   Lovász-set rows; overwritten with the exclusive offsets by occ_setup
    uint32_t *cta_flags;       // [row_ctas]
    int32_t *cta_fg;           // [row_ctas, C]
    OccGlobals *glob;
    int32_t *midx;             // [T] compacted index, -1 outside the set
    uint32_t *keys[2], *vals[2];   // [C, T] each (segment c at c * M)
    uint32_t *hist;            // [C, sort_tiles, kBins]
    int32_t *lov_fg;           // [C, lov_tiles]
    double *lov_part;          // [C, lov_tiles]
    float *gq;                 // [C, M] dL/dq, aliases keys[0]/vals[0] (free once the sort has finished in keys[1])
    size_t bytes;
};

size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

OccPlan plan(const gf_occ_loss_desc &d, void *base) {
    OccPlan p{};
    p.T = static_cast<long long>(d.B) * d.N;
    const long long T = p.T > 0 ? p.T : 1;
    const int C = d.C;
    p.row_ctas = static_cast<int>((T + kRowsPerCta - 1) / kRowsPerCta);
    p.sort_tiles = static_cast<int>((T + kSortTile - 1) / kSortTile);
    p.lov_tiles = static_cast<int>((T + kLovTile - 1) / kLovTile);
    size_t off = 0;
    char *b = static_cast<char *>(base);
    auto take = [&](size_t bytes) { void *ptr = b ? b + off : nullptr; off += align256(bytes); return ptr; };
    p.cta_ce = static_cast<double *>(take(sizeof(double) * 2 * p.row_ctas));
    p.cta_cnt = static_cast<int32_t *>(take(sizeof(int32_t) * p.row_ctas));
    p.cta_flags = static_cast<uint32_t *>(take(sizeof(uint32_t) * p.row_ctas));
    p.cta_fg = static_cast<int32_t *>(take(sizeof(int32_t) * p.row_ctas * C));
    p.glob = static_cast<OccGlobals *>(take(sizeof(OccGlobals)));
    if (d.lovasz) {
        p.midx = static_cast<int32_t *>(take(sizeof(int32_t) * T));
        for (int i = 0; i < 2; ++i) {
            p.keys[i] = static_cast<uint32_t *>(take(sizeof(uint32_t) * C * T));
            p.vals[i] = static_cast<uint32_t *>(take(sizeof(uint32_t) * C * T));
        }
        p.hist = static_cast<uint32_t *>(take(sizeof(uint32_t) * C * static_cast<size_t>(p.sort_tiles) * kBins));
        p.lov_fg = static_cast<int32_t *>(take(sizeof(int32_t) * C * p.lov_tiles));
        p.lov_part = static_cast<double *>(take(sizeof(double) * C * p.lov_tiles));
        p.gq = reinterpret_cast<float *>(p.keys[0]);
    }
    p.bytes = off;
    return p;
}

struct RowArgs {
    const float *pred;        // [T, C]
    const uint8_t *labels;    // [T]
    const uint8_t *mask;      // [T] or NULL
    const float *weights;     // [C] or NULL (ones)
    int C;
    int use_softmax, ignore_index, lovasz_ignore, ignore_empty, empty_label, lovasz;
    long long T;
};

// what one row contributes: CE (y valid, != ignore_index) and / or the Lovász set
struct RowClass {
    bool ce, in_set, bad;
};

__device__ __forceinline__ RowClass classify(const RowArgs &a, long long row, int y) {
    RowClass r{false, false, false};
    const bool active = (a.mask == nullptr || a.mask[row] != 0) && !(a.ignore_empty && y == a.empty_label);
    if (!active) return r;
    const bool in_range = y < a.C;
    r.bad = !in_range && y != a.ignore_index;
    r.ce = in_range && y != a.ignore_index;
    r.in_set = a.lovasz && (in_range || y == a.ignore_index) && y != a.lovasz_ignore;
    return r;
}

__device__ __forceinline__ float class_weight(const RowArgs &a, int y) { return a.weights ? a.weights[y] : 1.f; }

// coalesced load of rows [row0, row0 + n) into shared memory (row-major, C floats per row)
__device__ __forceinline__ void stage_rows(float *sm, const float *pred, long long row0, int n, int C) {
    const float *src = pred + row0 * C;
    for (int i = threadIdx.x; i < n * C; i += blockDim.x) sm[i] = src[i];
}

// q = softmax(z) (use_softmax) or q = z; returns the log-sum-exp of z (softmax only)
template <int C>
__device__ __forceinline__ float row_probs(const float *z, float *q, bool softmax) {
    if (!softmax) {
#pragma unroll
        for (int c = 0; c < C; ++c) q[c] = z[c];
        return 0.f;
    }
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        q[c] = expf(z[c] - m);
        s += q[c];
    }
    const float inv = 1.f / s;
#pragma unroll
    for (int c = 0; c < C; ++c) q[c] *= inv;
    return m + logf(s);
}

__device__ __forceinline__ float clamp_p(float p) { return fminf(fmaxf(p, 1e-6f), 1.f - 1e-6f); }

template <class Tv>
__device__ __forceinline__ Tv warp_sum(Tv v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// fixed-order block sum (result valid in thread 0); `sm` holds >= blockDim.x / 32 entries
template <class Tv>
__device__ __forceinline__ Tv block_sum(Tv v, Tv *sm) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) sm[w] = v;
    __syncthreads();
    Tv s = 0;
    if (threadIdx.x == 0)
        for (int i = 0; i < nw; ++i) s += sm[i];
    return s;
}

// exclusive block scan of ints; *total receives the block sum (all threads).  `sm`: >= 33 ints
__device__ __forceinline__ int block_exclusive_scan(int v, int *sm, int *total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    __syncthreads();
    if (lane == 31) sm[w] = incl;
    __syncthreads();
    if (w == 0) {
        int x = lane < nw ? sm[lane] : 0;
        int xi = x;
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, xi, o);
            if (lane >= o) xi += n;
        }
        if (lane < nw) sm[lane] = xi - x;
        if (lane == 31) sm[32] = xi;
    }
    __syncthreads();
    const int r = sm[w] + incl - v;
    *total = sm[32];
    return r;
}

// ---------------------------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kRowThreads) occ_rows(RowArgs a, OccPlan p) {
    __shared__ float rows[kRowThreads * C];
    __shared__ int fg[kMaxC];
    __shared__ double red[kRowThreads / 32];
    __shared__ uint32_t flags;
    if (threadIdx.x < kMaxC) fg[threadIdx.x] = 0;
    if (threadIdx.x == 0) flags = 0;
    double num = 0.0, den = 0.0;
    int cnt = 0;
    uint32_t bad = 0;
    const long long cta0 = static_cast<long long>(blockIdx.x) * kRowsPerCta;
    __syncthreads();
    for (int r = 0; r < kRowsPerCta / kRowThreads; ++r) {
        const long long row0 = cta0 + r * kRowThreads;
        if (row0 >= a.T) break;
        const int n = static_cast<int>((a.T - row0 < kRowThreads ? a.T - row0 : kRowThreads));
        __syncthreads();
        stage_rows(rows, a.pred, row0, n, C);
        __syncthreads();
        if (threadIdx.x < n) {
            const long long row = row0 + threadIdx.x;
            const int y = a.labels[row];
            const RowClass k = classify(a, row, y);
            bad |= k.bad ? GF_OCC_LABEL_OUT_OF_RANGE : 0u;
            if (k.in_set) {
                ++cnt;
                if (y < C) atomicAdd(&fg[y], 1);
            }
            if (k.ce) {
                const float *z = rows + threadIdx.x * C;
                float nll;
                if (a.use_softmax) {
                    float q[C];
                    nll = row_probs<C>(z, q, true) - z[y];
                } else {
                    nll = -logf(clamp_p(z[y]));
                }
                const float w = class_weight(a, y);
                num += static_cast<double>(w) * static_cast<double>(nll);
                den += static_cast<double>(w);
            }
        }
    }
    if (bad) atomicOr(&flags, bad);
    const double snum = block_sum(num, red);
    const double sden = block_sum(den, red);
    const int scnt = static_cast<int>(block_sum(static_cast<double>(cnt), red));
    __syncthreads();
    if (threadIdx.x == 0) {
        p.cta_ce[2 * blockIdx.x] = snum;
        p.cta_ce[2 * blockIdx.x + 1] = sden;
        p.cta_cnt[blockIdx.x] = scnt;
        p.cta_flags[blockIdx.x] = flags;
    }
    if (threadIdx.x < C) p.cta_fg[static_cast<long long>(blockIdx.x) * C + threadIdx.x] = fg[threadIdx.x];
}

__global__ void __launch_bounds__(1024) occ_setup(OccPlan p, int C, int nct, int lovasz, uint32_t *status) {
    __shared__ int sm[33];
    __shared__ double dred[32];
    __shared__ int fg[kMaxC];
    __shared__ uint32_t flags;
    if (threadIdx.x < kMaxC) fg[threadIdx.x] = 0;
    if (threadIdx.x == 0) flags = 0;
    __syncthreads();
    // contiguous chunk of CTAs per thread: sums in a fixed order
    const int per = (nct + blockDim.x - 1) / blockDim.x;
    const int i0 = min(nct, static_cast<int>(threadIdx.x) * per), i1 = min(nct, i0 + per);
    int cnt = 0;
    double num = 0.0, den = 0.0;
    uint32_t bad = 0;
    for (int i = i0; i < i1; ++i) {
        cnt += p.cta_cnt[i];
        num += p.cta_ce[2 * i];
        den += p.cta_ce[2 * i + 1];
        bad |= p.cta_flags[i];
    }
    for (int c = 0; c < C; ++c) {
        int s = 0;
        for (int i = i0; i < i1; ++i) s += p.cta_fg[static_cast<long long>(i) * C + c];
        if (s) atomicAdd(&fg[c], s);
    }
    if (bad) atomicOr(&flags, bad);
    int M = 0;
    int off = block_exclusive_scan(cnt, sm, &M);
    for (int i = i0; i < i1; ++i) {   // the set sizes become the compaction offsets
        const int v = p.cta_cnt[i];
        p.cta_cnt[i] = off;
        off += v;
    }
    const double snum = block_sum(num, dred);
    const double sden = block_sum(den, dred);
    __syncthreads();
    OccGlobals *g = p.glob;
    if (threadIdx.x == 0) {
        int np = 0;
        for (int c = 0; c < kMaxC; ++c) {
            const int gc = c < C && lovasz ? fg[c] : 0;
            g->g[c] = gc;
            g->present[c] = gc > 0;
            np += gc > 0;
        }
        g->M = lovasz ? M : 0;
        g->npresent = np;
        g->ce_num = snum;
        g->ce_den = sden;
        if (status) *status = flags;
    }
}

template <int C>
__global__ void __launch_bounds__(kRowThreads) occ_compact(RowArgs a, OccPlan p) {
    __shared__ float rows[kRowThreads * C];
    __shared__ int sm[33];
    const OccGlobals *g = p.glob;
    const int M = g->M;
    int base = p.cta_cnt[blockIdx.x];
    const long long cta0 = static_cast<long long>(blockIdx.x) * kRowsPerCta;
    for (int r = 0; r < kRowsPerCta / kRowThreads; ++r) {
        const long long row0 = cta0 + r * kRowThreads;
        if (row0 >= a.T) break;
        const int n = static_cast<int>((a.T - row0 < kRowThreads ? a.T - row0 : kRowThreads));
        __syncthreads();
        stage_rows(rows, a.pred, row0, n, C);
        __syncthreads();
        const long long row = row0 + threadIdx.x;
        int y = 0;
        bool in_set = false;
        if (threadIdx.x < n) {
            y = a.labels[row];
            in_set = classify(a, row, y).in_set;
        }
        int total = 0;
        const int rank = block_exclusive_scan(in_set ? 1 : 0, sm, &total);
        if (threadIdx.x < n) {
            const int m = in_set ? base + rank : -1;
            p.midx[row] = m;
            if (in_set) {
                float q[C];
                row_probs<C>(rows + threadIdx.x * C, q, a.use_softmax != 0);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    if (!g->present[c]) continue;
                    const bool fgc = y == c;
                    const float e = fabsf((fgc ? 1.f : 0.f) - q[c]);
                    const uint32_t key = kOne - __float_as_uint(fminf(e, 1.f));
                    const size_t at = static_cast<size_t>(c) * M + m;
                    p.keys[0][at] = key;
                    p.vals[0][at] = static_cast<uint32_t>(m) | (fgc ? kFgBit : 0u);
                }
            }
        }
        base += total;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// stable LSD radix sort of the C segments [c * M, (c + 1) * M) of present classes
__global__ void __launch_bounds__(kSortThreads) occ_sort_hist(const uint32_t *keys, OccPlan p, int shift) {
    __shared__ uint32_t h[kBins];
    const int c = blockIdx.y, tile = blockIdx.x;
    const int M = p.glob->M;
    if (!p.glob->present[c] || static_cast<long long>(tile) * kSortTile >= M) return;
    for (int i = threadIdx.x; i < kBins; i += kSortThreads) h[i] = 0;
    __syncthreads();
    const uint32_t *k = keys + static_cast<size_t>(c) * M;
    const int end = min(M, (tile + 1) * kSortTile);
    for (int i = tile * kSortTile + threadIdx.x; i < end; i += kSortThreads) atomicAdd(&h[(k[i] >> shift) & (kBins - 1)], 1u);
    __syncthreads();
    uint32_t *out = p.hist + (static_cast<size_t>(c) * p.sort_tiles + tile) * kBins;
    for (int i = threadIdx.x; i < kBins; i += kSortThreads) out[i] = h[i];
}

// per segment: hist[c][t][d] <- offset of the first key of digit d from tile t within the sorted segment
__global__ void __launch_bounds__(kBins) occ_sort_scan(OccPlan p) {
    __shared__ int sm[33];
    const int c = blockIdx.x;
    const int M = p.glob->M;
    if (!p.glob->present[c]) return;
    const int nt = (M + kSortTile - 1) / kSortTile;
    uint32_t *h = p.hist + static_cast<size_t>(c) * p.sort_tiles * kBins + threadIdx.x;
    int tot = 0;
    for (int t = 0; t < nt; ++t) tot += h[static_cast<size_t>(t) * kBins];
    int all = 0;
    int base = block_exclusive_scan(tot, sm, &all);
    for (int t = 0; t < nt; ++t) {
        const uint32_t v = h[static_cast<size_t>(t) * kBins];
        h[static_cast<size_t>(t) * kBins] = base;
        base += v;
    }
}

// Each warp owns 512 consecutive keys of the tile; per-warp digit offsets make the scatter stable: a key goes after
// every equal digit of earlier tiles, earlier warps, earlier 32-key steps and lower lanes.
__global__ void __launch_bounds__(kSortThreads) occ_sort_scatter(const uint32_t *kin, const uint32_t *vin, uint32_t *kout,
                                                                 uint32_t *vout, OccPlan p, int shift) {
    __shared__ uint32_t wh[kSortWarps][kBins];
    const int c = blockIdx.y, tile = blockIdx.x;
    const int M = p.glob->M;
    if (!p.glob->present[c] || static_cast<long long>(tile) * kSortTile >= M) return;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < kSortWarps * kBins; i += kSortThreads) (&wh[0][0])[i] = 0;
    __syncthreads();
    const size_t seg = static_cast<size_t>(c) * M;
    const int w0 = tile * kSortTile + w * kPerWarp;
    for (int s = 0; s < kPerWarp; s += 32) {
        const int i = w0 + s + lane;
        if (i < M) atomicAdd(&wh[w][(kin[seg + i] >> shift) & (kBins - 1)], 1u);
    }
    __syncthreads();
    const uint32_t *h = p.hist + (static_cast<size_t>(c) * p.sort_tiles + tile) * kBins;
    for (int d = threadIdx.x; d < kBins; d += kSortThreads) {
        uint32_t base = h[d];
        for (int j = 0; j < kSortWarps; ++j) {
            const uint32_t v = wh[j][d];
            wh[j][d] = base;
            base += v;
        }
    }
    __syncthreads();
    const unsigned lt = (1u << lane) - 1u;
    for (int s = 0; s < kPerWarp; s += 32) {
        const int i = w0 + s + lane;
        const bool ok = i < M;
        const uint32_t key = ok ? kin[seg + i] : 0u;
        const uint32_t val = ok ? vin[seg + i] : 0u;
        const uint32_t d = ok ? (key >> shift) & (kBins - 1) : kBins;   // kBins: a group of its own for idle lanes
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const uint32_t pos = ok ? wh[w][d] + __popc(peers & lt) : 0u;
        __syncwarp();
        if (ok && (__ffs(peers) - 1) == lane) wh[w][d] += __popc(peers);
        __syncwarp();
        if (ok) {
            kout[seg + pos] = key;
            vout[seg + pos] = val;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRowThreads) occ_lov_count(const uint32_t *vals, OccPlan p) {
    __shared__ double red[kRowThreads / 32];
    const int c = blockIdx.y, tile = blockIdx.x;
    const int M = p.glob->M;
    if (!p.glob->present[c] || static_cast<long long>(tile) * kLovTile >= M) return;
    const uint32_t *v = vals + static_cast<size_t>(c) * M;
    const int end = min(M, (tile + 1) * kLovTile);
    int n = 0;
    for (int i = tile * kLovTile + threadIdx.x; i < end; i += kRowThreads) n += v[i] >> 31;
    const int s = static_cast<int>(block_sum(static_cast<double>(n), red));
    if (threadIdx.x == 0) p.lov_fg[static_cast<size_t>(c) * p.lov_tiles + tile] = s;
}

// Closed-form Lovász gradient of the Jaccard index at sorted position i (g foreground elements in the class, F of them
// before i, B background elements up to and including i):  foreground 1 / (g + B),  background (g - F) / ((g+B-1)(g+B)).
__global__ void __launch_bounds__(kRowThreads) occ_lov_scan(const uint32_t *keys, const uint32_t *vals, OccPlan p,
                                                            int want_grad) {
    __shared__ int sm[33];
    __shared__ double red[kRowThreads / 32];
    const int c = blockIdx.y, tile = blockIdx.x;
    const int M = p.glob->M;
    if (!p.glob->present[c] || static_cast<long long>(tile) * kLovTile >= M) return;
    const size_t seg = static_cast<size_t>(c) * M;
    const double gc = p.glob->g[c];
    int before = 0;   // foreground elements in earlier tiles
    for (int t = threadIdx.x; t < tile; t += kRowThreads) before += p.lov_fg[static_cast<size_t>(c) * p.lov_tiles + t];
    before = static_cast<int>(block_sum(static_cast<double>(before), red));
    __syncthreads();
    if (threadIdx.x == 0) sm[32] = before;   // broadcast through the scan's scratch below
    __syncthreads();
    before = sm[32];
    const int i0 = tile * kLovTile + threadIdx.x * kLovPerThread;
    const int i1 = min(M, i0 + kLovPerThread);
    int mine = 0;
    for (int i = i0; i < i1; ++i) mine += vals[seg + i] >> 31;
    int total = 0;
    int F = before + block_exclusive_scan(mine, sm, &total);
    double acc = 0.0;
    for (int i = i0; i < i1; ++i) {
        const uint32_t v = vals[seg + i];
        const bool fg = v >> 31;
        const double Bc = static_cast<double>(i + 1 - F - (fg ? 1 : 0));
        const double dj = fg ? 1.0 / (gc + Bc) : (gc - F) / ((gc + Bc - 1.0) * (gc + Bc));
        const float e = __uint_as_float(kOne - keys[seg + i]);
        acc += static_cast<double>(e) * dj;
        if (want_grad) {
            // e = |fg - q|: de/dq = -1 (fg) or +1 (background), 0 where e == 0 (torch's abs'(0) = 0)
            const float gqv = e == 0.f ? 0.f : static_cast<float>(fg ? -dj : dj);
            p.gq[seg + (v & ~kFgBit)] = gqv;
        }
        F += fg;
    }
    const double s = block_sum(acc, red);
    if (threadIdx.x == 0) p.lov_part[static_cast<size_t>(c) * p.lov_tiles + tile] = s;
}

__global__ void __launch_bounds__(1024) occ_final(OccPlan p, int C, float ce_weight, float lovasz_weight, float *loss3) {
    __shared__ double cls[kMaxC];
    OccGlobals *g = p.glob;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int M = g->M;
    const int nt = (M + kLovTile - 1) / kLovTile;
    if (w < C) {   // one warp per class, fixed order
        double s = 0.0;
        if (g->present[w])
            for (int t = lane; t < nt; t += 32) s += p.lov_part == nullptr ? 0.0 : p.lov_part[static_cast<size_t>(w) * p.lov_tiles + t];
        s = warp_sum(s);
        if (lane == 0) cls[w] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double lov = 0.0;
        for (int c = 0; c < C; ++c)
            if (g->present[c]) lov += cls[c];
        const int np = g->npresent;
        lov = np > 0 ? lov / np : 0.0;
        const double ce = g->ce_num / g->ce_den;   // 0 / 0 = NaN when no point is left, as in torch
        const double ce_w = static_cast<double>(ce_weight) * ce;
        const double lov_w = static_cast<double>(lovasz_weight) * lov;
        loss3[0] = static_cast<float>(ce_w + lov_w);
        loss3[1] = static_cast<float>(ce_w);
        loss3[2] = static_cast<float>(lov_w);
        g->ce_scale = static_cast<double>(ce_weight) / g->ce_den;
        g->lov_scale = np > 0 ? static_cast<double>(lovasz_weight) / np : 0.0;
    }
}

template <int C>
__global__ void __launch_bounds__(kRowThreads) occ_grad(RowArgs a, OccPlan p, float *grad) {
    __shared__ float rows[kRowThreads * C];
    const long long row0 = static_cast<long long>(blockIdx.x) * kRowThreads;
    const int n = static_cast<int>((a.T - row0 < kRowThreads ? a.T - row0 : kRowThreads));
    stage_rows(rows, a.pred, row0, n, C);
    __syncthreads();
    const OccGlobals *g = p.glob;
    if (threadIdx.x < n) {
        const long long row = row0 + threadIdx.x;
        const int y = a.labels[row];
        const RowClass k = classify(a, row, y);
        float *z = rows + threadIdx.x * C;   // overwritten in place with the gradient row
        const float zy = k.ce ? z[y] : 0.f;   // the probability of the label in probability mode
        float q[C], gl[C];
        row_probs<C>(z, q, a.use_softmax != 0);
        const int m = a.lovasz && k.in_set ? p.midx[row] : -1;
        const float ls = static_cast<float>(g->lov_scale);
        const int M = g->M;
#pragma unroll
        for (int c = 0; c < C; ++c) gl[c] = (m >= 0 && g->present[c]) ? ls * p.gq[static_cast<size_t>(c) * M + m] : 0.f;
        const float cs = k.ce ? static_cast<float>(g->ce_scale * class_weight(a, y)) : 0.f;
        if (a.use_softmax) {
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) dot += q[c] * gl[c];
#pragma unroll
            for (int c = 0; c < C; ++c)
                z[c] = q[c] * (gl[c] - dot) + (k.ce ? cs * (q[c] - (c == y ? 1.f : 0.f)) : 0.f);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = gl[c];
            if (k.ce && zy >= 1e-6f && zy <= 1.f - 1e-6f) z[y] += -cs / zy;   // clamp passes the gradient on [lo, hi]
        }
        if (!(k.ce || k.in_set))
            for (int c = 0; c < C; ++c) z[c] = 0.f;
    }
    __syncthreads();
    float *dst = grad + row0 * C;
    for (int i = threadIdx.x; i < n * C; i += blockDim.x) dst[i] = rows[i];
}

template <int C>
int launch_all(const gf_occ_loss_desc &d, const RowArgs &a, const OccPlan &p, float *loss3, float *grad,
               uint32_t *status, cudaStream_t stream) {
    const int nct = p.T > 0 ? p.row_ctas : 0;
    if (nct > 0) occ_rows<C><<<nct, kRowThreads, 0, stream>>>(a, p);
    occ_setup<<<1, 1024, 0, stream>>>(p, d.C, nct, d.lovasz != 0, status);
    if (d.lovasz && nct > 0) {
        occ_compact<C><<<nct, kRowThreads, 0, stream>>>(a, p);
        const dim3 sgrid(p.sort_tiles, d.C);
        for (int pass = 0; pass < 3; ++pass) {
            const int src = pass & 1, shift = pass * kRadixBits;
            occ_sort_hist<<<sgrid, kSortThreads, 0, stream>>>(p.keys[src], p, shift);
            occ_sort_scan<<<d.C, kBins, 0, stream>>>(p);
            occ_sort_scatter<<<sgrid, kSortThreads, 0, stream>>>(p.keys[src], p.vals[src], p.keys[src ^ 1],
                                                                  p.vals[src ^ 1], p, shift);
        }
        const dim3 lgrid(p.lov_tiles, d.C);   // sorted keys are in buffer 1 after three passes
        occ_lov_count<<<lgrid, kRowThreads, 0, stream>>>(p.vals[1], p);
        occ_lov_scan<<<lgrid, kRowThreads, 0, stream>>>(p.keys[1], p.vals[1], p, grad != nullptr);
    }
    occ_final<<<1, 1024, 0, stream>>>(p, d.C, d.ce_weight, d.lovasz_weight, loss3);
    if (grad && nct > 0)
        occ_grad<C><<<static_cast<int>((p.T + kRowThreads - 1) / kRowThreads), kRowThreads, 0, stream>>>(a, p, grad);
    GF_CUDA_TRY(cudaGetLastError());
    return GF_OK;
}

}  // namespace

int occ_loss_check(const gf_occ_loss_desc *d) {
    GF_REQUIRE(d != nullptr, GF_ERR_INVALID_ARG, "occ_loss: desc is NULL");
    GF_REQUIRE(d->B >= 0 && d->N >= 0, GF_ERR_INVALID_ARG, "occ_loss: negative B or N");
    GF_REQUIRE(d->C >= 16 && d->C <= 20, GF_ERR_UNSUPPORTED, "occ_loss: class count C=%d outside the compiled range 16..20", d->C);
    GF_REQUIRE(static_cast<long long>(d->B) * d->N * d->C < (1ll << 31), GF_ERR_UNSUPPORTED, "occ_loss: B x N x C >= 2^31");
    GF_REQUIRE(d->ignore_index >= 0 && d->ignore_index <= 255, GF_ERR_INVALID_ARG, "occ_loss: ignore_index outside 0..255");
    return GF_OK;
}

size_t occ_loss_workspace_bytes(const gf_occ_loss_desc &d) { return plan(d, nullptr).bytes; }

int occ_loss_forward(const gf_occ_loss_desc &d, const float *pred, const uint8_t *labels, const uint8_t *mask,
                     const float *weights, float *loss3, float *grad, uint32_t *status, void *ws, cudaStream_t stream) {
    OccPlan p = plan(d, ws);
    RowArgs a{pred, labels, mask, weights, d.C, d.use_softmax, d.ignore_index, d.lovasz_ignore, d.ignore_empty,
              d.empty_label, d.lovasz != 0, p.T};
    switch (d.C) {
        case 16: return launch_all<16>(d, a, p, loss3, grad, status, stream);
        case 17: return launch_all<17>(d, a, p, loss3, grad, status, stream);
        case 18: return launch_all<18>(d, a, p, loss3, grad, status, stream);
        case 19: return launch_all<19>(d, a, p, loss3, grad, status, stream);
        case 20: return launch_all<20>(d, a, p, loss3, grad, status, stream);
        default: break;
    }
    GF_REQUIRE(false, GF_ERR_UNSUPPORTED, "occ_loss: class count C=%d is not compiled in", d.C);
}

}  // namespace gf
