// Geometry distortion metric on the device (SURVEY 8f-3): exact nearest neighbour of every query point in a reference
// cloud, the kernel under the D1 (point-to-point) / D2 (point-to-plane) PSNR that the reference obtains from the MPEG
// `pc_error` subprocess (lib/metrics/pc_error_wrapper.py:40-106, called from lib/evaluators.py:49-124).
// Brute force in integer arithmetic: exact squared distances, lowest reference index among equal distances.
// Bound: CUDA-core integer ALU (3 subtractions + 3 multiply-adds + compare/select per pair); reference points are
// staged once per CTA tile in shared memory and broadcast, so HBM/L2 traffic is nr*16 B per CTA.
//
// Exact batched K nearest neighbours on a uniform cell grid (fpcc_knn_search, DESIGN 3.6): the search under
// lib/knn3d/src/knn3d.cu (KNearestNeighborKernelV0/V2) and, at K = 1, under metrics.pc_error.  O(N*K) for voxel
// clouds instead of the O(N^2) of the brute force above, which stays as the workspace-free entry point and as the
// on-device reference of the tests.
//
// All-ties nearest neighbour with attribute sums (fpcc_nn_tie_attr, DESIGN 3.7): the same grid and ring walk with a
// collector that keeps every reference row at the least distance, for recolouring and pc_error's colour figures.
#include <cub/cub.cuh>

#include "common.cuh"

namespace fpcc {

constexpr int NN_THREADS = 256;
constexpr int NN_QPT = 4;       // queries per thread (registers)
constexpr int NN_TILE = 1024;   // reference points per shared-memory tile (16 KB)

template <typename D>  // D = uint32_t when 3 * 4^coord_bits fits 32 bits, else uint64_t
__global__ void __launch_bounds__(NN_THREADS) nn_kernel(const int32_t *__restrict__ query, int nq, int q_ld, int q_col,
                                                        const int32_t *__restrict__ ref, int nr, int r_ld, int r_col,
                                                        int64_t *__restrict__ d2_out, int32_t *__restrict__ idx_out) {
    __shared__ int4 tile[NN_TILE];
    int qx[NN_QPT], qy[NN_QPT], qz[NN_QPT], bi[NN_QPT];
    D best[NN_QPT];
    const int q0 = blockIdx.x * (NN_THREADS * NN_QPT) + threadIdx.x;
#pragma unroll
    for (int j = 0; j < NN_QPT; ++j) {
        const int q = q0 + j * NN_THREADS;
        const int32_t *p = query + (int64_t)min(q, nq - 1) * q_ld + q_col;
        qx[j] = p[0]; qy[j] = p[1]; qz[j] = p[2];
        best[j] = ~(D)0; bi[j] = -1;
    }
    for (int base = 0; base < nr; base += NN_TILE) {
        const int cnt = min(NN_TILE, nr - base);
        __syncthreads();
        for (int t = threadIdx.x; t < cnt; t += NN_THREADS) {
            const int32_t *p = ref + (int64_t)(base + t) * r_ld + r_col;
            tile[t] = make_int4(p[0], p[1], p[2], 0);
        }
        __syncthreads();
#pragma unroll 4
        for (int t = 0; t < cnt; ++t) {
            const int4 r = tile[t];
#pragma unroll
            for (int j = 0; j < NN_QPT; ++j) {
                const int dx = qx[j] - r.x, dy = qy[j] - r.y, dz = qz[j] - r.z;
                D d;
                if (sizeof(D) == 4) d = (D)((uint32_t)(dx * dx) + (uint32_t)(dy * dy) + (uint32_t)(dz * dz));
                else d = (D)((uint64_t)((int64_t)dx * dx) + (uint64_t)((int64_t)dy * dy) + (uint64_t)((int64_t)dz * dz));
                if (d < best[j]) { best[j] = d; bi[j] = base + t; }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NN_QPT; ++j) {
        const int q = q0 + j * NN_THREADS;
        if (q < nq) {
            d2_out[q] = (int64_t)best[j];
            if (idx_out) idx_out[q] = bi[j];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K nearest neighbours on a cell grid.
//
// Build (reference rows, all on the device): per-batch bounding box and count -> base cell edge 2^e0 per batch (the
// smallest power of two, >= 1 for int32, for which the batch spans < 2^18 base cells per axis) -> sort by
// (batch, Morton code of the base cell) -> count, per level l, the distinct cells of edge 2^(e0+l) (Morton order nests
// the levels, so every cell of every level is one contiguous run of the sorted order) -> per batch the smallest level
// with at least `target` points per occupied cell -> one hash entry (pack_key(b, cx, cy, cz) -> [start, end)) per
// occupied cell and a packed copy of the sorted points.
//
// Cell assignment is floor(x * 2^-e0) in double: exact for int32 and float32 inputs alike, so every point lies inside
// the closed box of its cell and the pruning bound below needs no slack.
//
// Search (one thread per query): Chebyshev rings of cells around the query's cell, the K best (distance, row) pairs
// sorted in registers.  After ring r every unvisited point lies outside the box of cells [qc - r, qc + r] on some
// axis, hence at distance >= g along that axis, g = the least gap from the query to a face of that box behind which
// the batch still has cells.  The search stops when K candidates are held and g^2 > the K-th distance (strictly: an
// equal distance at a lower row would still win), when no such face is left, or after KNN_RING_CAP rings; the last
// case restarts the query as a scan of its whole batch.  Batches of at most KNN_SCAN_MAX points are scanned directly.
// float32: the gap is rounded down and squared with the distance's own rounding, and fp rounding is monotone, so the
// computed distance of any point outside the box is >= the computed bound: the stop test is conservative.
constexpr int KNN_LEVELS = 19;      // cell levels 0..18 above the base cell (18 bits per axis)
constexpr int KNN_RING_CAP = 6;     // rings 0..6: at most 13^3 cell probes before the batch scan
constexpr int KNN_SCAN_MAX = 64;    // batches this small are scanned
constexpr int KNN_THREADS = 128;
constexpr int KNN_CHUNK = 16;       // rows per thread in the reduction passes

struct KnnBatch {
    uint32_t lo[3], hi[3];          // order-preserving images of the per-axis min / max
    int32_t count;                  // reference rows of the batch
    int32_t start;                  // its first row in the sorted order
    int32_t e0;                     // base cell edge 2^e0
    int32_t level;                  // search cell edge 2^(e0 + level)
    long long minc[3];              // base cell of the box corner: floor(min * 2^-e0)
    int32_t ncell[3];               // base cells spanned (after the build: search cells per axis)
    int32_t hist[KNN_LEVELS];       // hist[l]: sorted neighbours whose base cells first share a cell at level l + 1
};

template <typename T> struct KnnT;
template <> struct KnnT<int32_t> {
    typedef unsigned long long D;
    typedef int4 P;
    static constexpr bool is_int = true;
    static __device__ __forceinline__ uint32_t order(int32_t v) { return (uint32_t)v ^ 0x80000000u; }
    static __device__ __forceinline__ double unorder(uint32_t u) { return (double)(int32_t)(u ^ 0x80000000u); }
    static __device__ __forceinline__ int batch(int32_t v, int nb) { return (v >= 0 && v < nb) ? v : -1; }
    static __device__ __forceinline__ P pack(int32_t x, int32_t y, int32_t z, int row) { return make_int4(x, y, z, row); }
    static __device__ __forceinline__ int row(const P &p) { return p.w; }
    static __device__ __forceinline__ D far() { return ~0ull; }
    static __device__ __forceinline__ D dist(int32_t x, int32_t y, int32_t z, const P &p) {
        const long long dx = (long long)x - p.x, dy = (long long)y - p.y, dz = (long long)z - p.z;
        return (D)(dx * dx) + (D)(dy * dy) + (D)(dz * dz);  // |c| < 2^30: < 3 * 2^62, exact
    }
    static __device__ __forceinline__ D bound(double g) {  // g: an exact integer gap
        return g >= 4294967296.0 ? ~0ull : (D)g * (D)g;
    }
};
template <> struct KnnT<float> {
    typedef float D;
    typedef float4 P;
    static constexpr bool is_int = false;
    static __device__ __forceinline__ uint32_t order(float f) {
        const uint32_t u = __float_as_uint(f);
        return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    }
    static __device__ __forceinline__ double unorder(uint32_t k) {
        return (double)__uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
    }
    static __device__ __forceinline__ int batch(float v, int nb) {
        return (v >= 0.f && v < (float)nb && v == floorf(v)) ? (int)v : -1;
    }
    static __device__ __forceinline__ P pack(float x, float y, float z, int row) { return make_float4(x, y, z, __int_as_float(row)); }
    static __device__ __forceinline__ int row(const P &p) { return __float_as_int(p.w); }
    static __device__ __forceinline__ D far() { return __int_as_float(0x7f800000); }
    static __device__ __forceinline__ D dist(float x, float y, float z, const P &p) {
        // ((dx*dx + dy*dy) + dz*dz), one rounding per operation, no FMA contraction: numpy float32's own result
        const float dx = __fsub_rn(x, p.x), dy = __fsub_rn(y, p.y), dz = __fsub_rn(z, p.z);
        return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    }
    static __device__ __forceinline__ D bound(double g) {
        const float gf = __double2float_rd(g);
        return __fmul_rn(gf, gf);
    }
};

__device__ __forceinline__ unsigned long long knn_spread3(uint32_t v) {
    unsigned long long x = v & 0x3ffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
__device__ __forceinline__ uint32_t knn_compact3(unsigned long long x) {
    x &= 0x1249249249249249ull;
    x = (x ^ (x >> 2)) & 0x10c30c30c30c30c3ull;
    x = (x ^ (x >> 4)) & 0x100f00f00f00f00full;
    x = (x ^ (x >> 8)) & 0x1f0000ff0000ffull;
    x = (x ^ (x >> 16)) & 0x1f00000000ffffull;
    x = (x ^ (x >> 32)) & 0x1fffffull;
    return (uint32_t)x;
}
// 2^e for |e| <= 1022, exact (cell edges are powers of two; ldexp is a library call)
__device__ __forceinline__ double knn_pow2(int e) { return __longlong_as_double((long long)(1023 + e) << 52); }
constexpr unsigned long long KNN_CELL_MASK = (1ull << 54) - 1;
constexpr unsigned long long KNN_NO_KEY = ~0ull;  // rows outside [0, n_batch): sorted last, never matched

template <typename T>
__device__ __forceinline__ int knn_row_batch(const T *row, int bcol, int nb) {
    return bcol < 0 ? 0 : KnnT<T>::batch(row[bcol], nb);
}

__global__ void knn_init_kernel(KnnBatch *bt, int nb) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    KnnBatch z = {};
    for (int a = 0; a < 3; ++a) z.lo[a] = 0xffffffffu;
    bt[b] = z;
}

// per-batch bounding box and count; each thread folds KNN_CHUNK consecutive rows and flushes on a batch change
template <typename T>
__global__ void __launch_bounds__(256) knn_bbox_kernel(const T *ref, int nr, int ld, int col, int bcol, int nb, KnnBatch *bt) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * KNN_CHUNK;
    int cur = -1, cnt = 0;
    uint32_t lo[3], hi[3];
    for (int64_t i = i0; i < i0 + KNN_CHUNK && i < nr; ++i) {
        const T *p = ref + i * ld;
        const int b = knn_row_batch(p, bcol, nb);
        if (b < 0) continue;
        if (b != cur) {
            if (cur >= 0) {
                for (int a = 0; a < 3; ++a) { atomicMin(&bt[cur].lo[a], lo[a]); atomicMax(&bt[cur].hi[a], hi[a]); }
                atomicAdd(&bt[cur].count, cnt);
            }
            cur = b; cnt = 0;
            for (int a = 0; a < 3; ++a) { lo[a] = 0xffffffffu; hi[a] = 0; }
        }
        ++cnt;
        for (int a = 0; a < 3; ++a) {
            const uint32_t o = KnnT<T>::order(p[col + a]);
            lo[a] = min(lo[a], o); hi[a] = max(hi[a], o);
        }
    }
    if (cur >= 0) {
        for (int a = 0; a < 3; ++a) { atomicMin(&bt[cur].lo[a], lo[a]); atomicMax(&bt[cur].hi[a], hi[a]); }
        atomicAdd(&bt[cur].count, cnt);
    }
}

// one block: batch start offsets, base cell edge and corner per batch
template <typename T>
__global__ void __launch_bounds__(1024) knn_setup_kernel(KnnBatch *bt, int nb) {
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        KnnBatch &B = bt[b];
        if (B.count == 0) continue;
        double lo[3], hi[3], ext = 0.0, mabs = 0.0;
        for (int a = 0; a < 3; ++a) {
            lo[a] = KnnT<T>::unorder(B.lo[a]); hi[a] = KnnT<T>::unorder(B.hi[a]);
            ext = fmax(ext, hi[a] - lo[a]);
            mabs = fmax(mabs, fmax(fabs(lo[a]), fabs(hi[a])));
        }
        int e0 = KnnT<T>::is_int ? 0 : -2000;
        if (ext > 0.0) e0 = max(e0, ilogb(ext) - 16);   // span < 2^17 base cells
        if (mabs > 0.0) e0 = max(e0, ilogb(mabs) - 50); // |x| * 2^-e0 < 2^51: cell bounds exact in double
        if (e0 == -2000) e0 = 0;                         // all points at the origin
        for (;;) {  // the span test is exact; at most a step or two beyond the estimate
            const double s = knn_pow2(-e0);
            bool ok = true;
            for (int a = 0; a < 3; ++a) ok &= floor(hi[a] * s) - floor(lo[a] * s) < 262144.0;
            if (ok) break;
            ++e0;
        }
        const double s = knn_pow2(-e0);
        B.e0 = e0;
        for (int a = 0; a < 3; ++a) {
            B.minc[a] = (long long)floor(lo[a] * s);
            B.ncell[a] = (int)((long long)floor(hi[a] * s) - B.minc[a]) + 1;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int b = 0; b < nb; ++b) { bt[b].start = s; s += bt[b].count; }
    }
}

template <typename T>
__device__ __forceinline__ void knn_base_cell(const T *xyz, const KnnBatch &B, int64_t c[3]) {
    const double s = knn_pow2(-B.e0);
    for (int a = 0; a < 3; ++a) c[a] = (long long)floor((double)xyz[a] * s) - B.minc[a];
}

template <typename T>
__global__ void __launch_bounds__(256) knn_key_kernel(const T *ref, int nr, int ld, int col, int bcol, int nb, const KnnBatch *bt,
                                                      unsigned long long *keys, int32_t *rows) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nr) return;
    const T *p = ref + (int64_t)i * ld;
    const int b = knn_row_batch(p, bcol, nb);
    unsigned long long key = KNN_NO_KEY;
    if (b >= 0) {
        int64_t c[3];
        knn_base_cell(p + col, bt[b], c);
        key = ((unsigned long long)b << 54) | knn_spread3((uint32_t)c[0]) << 2 | knn_spread3((uint32_t)c[1]) << 1 |
              knn_spread3((uint32_t)c[2]);
    }
    keys[i] = key;
    rows[i] = i;
}

// distinct-cell counts per level: sorted neighbours i-1, i of one batch first share a cell at level hb/3 + 1
__global__ void __launch_bounds__(256) knn_hist_kernel(const unsigned long long *keys, int nr, KnnBatch *bt) {
    __shared__ int h[KNN_LEVELS];
    __shared__ unsigned long long b0;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (threadIdx.x < KNN_LEVELS) h[threadIdx.x] = 0;
    if (threadIdx.x == 0) b0 = keys[blockIdx.x * blockDim.x] >> 54;
    __syncthreads();
    if (i > 0 && i < nr) {
        const unsigned long long k = keys[i], x = k ^ keys[i - 1];
        if (k != KNN_NO_KEY && x != 0 && (x >> 54) == 0) {
            const int l = (63 - __clzll((long long)x)) / 3;
            if ((k >> 54) == b0) atomicAdd(&h[l], 1);
            else atomicAdd(&bt[k >> 54].hist[l], 1);
        }
    }
    __syncthreads();
    if (threadIdx.x < KNN_LEVELS && h[threadIdx.x] && b0 < 1023) atomicAdd(&bt[b0].hist[threadIdx.x], h[threadIdx.x]);
}

// smallest level with >= target points per occupied cell
__global__ void __launch_bounds__(1024) knn_level_kernel(KnnBatch *bt, int nb, int target) {
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        KnnBatch &B = bt[b];
        if (B.count == 0) continue;
        int distinct = 1, level = KNN_LEVELS - 1;
        for (int l = KNN_LEVELS - 1; l >= 0; --l) {  // distinct(l) = 1 + sum_{j >= l} hist[j]
            distinct += B.hist[l];
            if (B.count >= target * distinct) level = l;
            else break;
        }
        B.level = level;
        for (int a = 0; a < 3; ++a) B.ncell[a] = ((B.ncell[a] - 1) >> level) + 1;
    }
}

__device__ __forceinline__ uint32_t knn_hash_find(const unsigned long long *__restrict__ keys, uint32_t capacity,
                                                  unsigned long long key) {
    uint32_t slot = hash_slot(key, capacity);
    while (true) {
        const unsigned long long cur = __ldg(&keys[slot]);
        if (cur == key) return slot;
        if (cur == 0ull) return 0xffffffffu;
        slot = slot + 1 == capacity ? 0 : slot + 1;
    }
}

// packed sorted points; the first and the last row of every cell run register the run in the hash table
template <typename T>
__global__ void __launch_bounds__(256) knn_cell_kernel(const T *ref, int nr, int ld, int col, const unsigned long long *keys,
                                                       const int32_t *rows, const KnnBatch *bt, typename KnnT<T>::P *pts,
                                                       unsigned long long *hkeys, int32_t *hlo, int32_t *hhi, uint32_t cap) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nr) return;
    const unsigned long long k = keys[i];
    if (k == KNN_NO_KEY) return;
    const int row = rows[i];
    const T *p = ref + (int64_t)row * ld + col;
    pts[i] = KnnT<T>::pack(p[0], p[1], p[2], row);
    const int b = (int)(k >> 54);
    const int sh = 3 * bt[b].level;  // a batch change sets bits >= 54 >= sh of the xor
    const bool first = i == 0 || ((k ^ keys[i - 1]) >> sh) != 0;
    const bool last = i == nr - 1 || ((k ^ keys[i + 1]) >> sh) != 0;
    if (!first && !last) return;
    const unsigned long long c = k & KNN_CELL_MASK;
    const int lv = bt[b].level;
    const unsigned long long key = pack_key(b, knn_compact3(c >> 2) >> lv, knn_compact3(c >> 1) >> lv, knn_compact3(c) >> lv);
    uint32_t slot = hash_slot(key, cap);
    while (true) {
        const unsigned long long prev = atomicCAS(&hkeys[slot], 0ull, key);
        if (prev == 0ull || prev == key) break;
        slot = slot + 1 == cap ? 0 : slot + 1;
    }
    if (first) hlo[slot] = i;
    if (last) hhi[slot] = i + 1;
}

// Collectors of the ring walk: begin (bind the outputs, empty), reset (empty), offer(distance, packed point),
// settled(bound, k)
// (every unvisited point is at distance >= bound: may the walk stop?), store(query, k).
template <typename T, int KB>
struct KnnList {  // the K best (distance, row) pairs, sorted in registers
    typedef typename KnnT<T>::D D;
    struct Out {
        D *dist;
        int32_t *idx;
    };
    static constexpr int min_blocks = KB >= 16 ? 2 : 4;
    D d[KB];
    int r[KB];
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int j = 0; j < KB; ++j) { d[j] = KnnT<T>::far(); r[j] = INT_MAX; }
    }
    __device__ __forceinline__ void begin(const Out &) { reset(); }
    static __device__ __forceinline__ bool better(D da, int ra, D db, int rb) { return da < db || (da == db && ra < rb); }
    __device__ __forceinline__ void offer(D nd, const typename KnnT<T>::P &p) {
        const int nr = KnnT<T>::row(p);
        if (!better(nd, nr, d[KB - 1], r[KB - 1])) return;
#pragma unroll
        for (int j = KB - 1; j > 0; --j) {  // j > slot: shift down, j == slot: insert, j < slot: keep
            const bool sh = better(nd, nr, d[j - 1], r[j - 1]);
            const bool here = !sh && better(nd, nr, d[j], r[j]);
            d[j] = sh ? d[j - 1] : (here ? nd : d[j]);
            r[j] = sh ? r[j - 1] : (here ? nr : r[j]);
        }
        if (better(nd, nr, d[0], r[0])) { d[0] = nd; r[0] = nr; }
    }
    // K held and the bound strictly beyond the K-th distance: an equal distance at a lower row would still win
    __device__ __forceinline__ bool settled(D bnd, int k) const {
        D kd = d[0];  // the k-th best so far (the list is sorted: the last of the first k)
        int kr = r[0];
#pragma unroll
        for (int j = 1; j < KB; ++j) {
            kd = j < k ? d[j] : kd;
            kr = j < k ? r[j] : kr;
        }
        return kr != INT_MAX && bnd > kd;
    }
    __device__ __forceinline__ void store(const Out &o, int q, int k) const {
#pragma unroll
        for (int j = 0; j < KB; ++j) {
            if (j < k) {
                const bool hit = r[j] != INT_MAX;
                o.dist[(int64_t)q * k + j] = hit ? d[j] : (D)0;
                o.idx[(int64_t)q * k + j] = hit ? r[j] : -1;
            }
        }
    }
};

// every reference row at the least distance (int32 rows): that distance, their number and the sums of their uint8
// RGB rows.  Integer sums: the result does not depend on the order of the visit.
struct KnnTie {
    typedef unsigned long long D;
    struct Out {
        const uint8_t *rgb;
        int64_t *d2;
        int32_t *count;
        int64_t *sum;
    };
    static constexpr int min_blocks = 4;
    const uint8_t *__restrict__ rgb;
    D best;
    int n;
    long long s0, s1, s2;
    __device__ __forceinline__ void reset() { best = ~0ull; n = 0; s0 = s1 = s2 = 0; }
    __device__ __forceinline__ void begin(const Out &o) { rgb = o.rgb; reset(); }
    __device__ __forceinline__ void offer(D d, const int4 &p) {
        if (d > best) return;
        const int row = p.w;
        if (d < best) { best = d; n = 0; s0 = s1 = s2 = 0; }
        const uint8_t *c = rgb + 3 * (int64_t)row;
        ++n; s0 += __ldg(c); s1 += __ldg(c + 1); s2 += __ldg(c + 2);
    }
    // strictly beyond: a point at exactly `best` may still be unvisited
    __device__ __forceinline__ bool settled(D bnd, int) const { return n > 0 && bnd > best; }
    __device__ __forceinline__ void store(const Out &o, int q, int) const {
        o.d2[q] = n ? (int64_t)best : 0;
        o.count[q] = n;
        o.sum[3 * (int64_t)q] = s0; o.sum[3 * (int64_t)q + 1] = s1; o.sum[3 * (int64_t)q + 2] = s2;
    }
};

// The ring walk of one query (x, y, z) of batch b (b >= 0) over the grid, feeding every visited row to L.  rings false:
// go straight to the scan of the whole batch.  Returns false when the walk ended in that scan, true when the rings
// settled (or the rings visited every cell of the batch).
template <typename T, typename Coll>
__device__ __forceinline__ bool knn_walk(Coll &L, T qx, T qy, T qz, int b, int k, bool rings, const KnnBatch *__restrict__ bt,
                                         const typename KnnT<T>::P *__restrict__ pts, const unsigned long long *__restrict__ hkeys,
                                         const int32_t *__restrict__ hlo, const int32_t *__restrict__ hhi, uint32_t cap) {
    typedef KnnT<T> C;
    const int count = bt[b].count, start = bt[b].start;
    if (rings && count > KNN_SCAN_MAX) {
        const int lv = bt[b].level, e0 = bt[b].e0;
        int64_t qc[3];
        int nc[3];
        double qd[3] = {(double)qx, (double)qy, (double)qz}, lo0[3];
        const double s = knn_pow2(-e0);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const long long m = bt[b].minc[a];
            // clamped far outside the grid: the gaps below stay valid bounds for such a query
            const double rel = fmin(fmax(floor(qd[a] * s) - (double)m, -1099511627776.0), 1099511627776.0);
            qc[a] = (int64_t)rel >> lv;
            nc[a] = bt[b].ncell[a];
            lo0[a] = (double)m;
        }
        const int64_t step = (int64_t)1 << lv;  // base cells per search cell
        const double e0p = knn_pow2(e0);        // base cell edge
        for (int r = 0; r <= KNN_RING_CAP; ++r) {
            const int64_t x0 = max(qc[0] - r, (int64_t)0), x1 = min(qc[0] + r, (int64_t)nc[0] - 1);
            const int64_t y0 = max(qc[1] - r, (int64_t)0), y1 = min(qc[1] + r, (int64_t)nc[1] - 1);
            const int64_t z0 = max(qc[2] - r, (int64_t)0), z1 = min(qc[2] + r, (int64_t)nc[2] - 1);
            for (int64_t x = x0; x <= x1; ++x) {
                for (int64_t y = y0; y <= y1; ++y) {
                    // shell columns on an x or y face: every z; inner columns (r >= 1): the two z faces
                    const bool face = x == qc[0] - r || x == qc[0] + r || y == qc[1] - r || y == qc[1] + r;
                    const int64_t zs = face ? 1 : 2 * r;
                    for (int64_t z = face ? z0 : qc[2] - r; z <= (face ? z1 : qc[2] + r); z += zs) {
                        if (z < z0 || z > z1) continue;
                        const uint32_t slot = knn_hash_find(hkeys, cap, pack_key(b, (int)x, (int)y, (int)z));
                        if (slot == 0xffffffffu) continue;
                        const int e = __ldg(&hhi[slot]);
                        for (int j = __ldg(&hlo[slot]); j < e; ++j) {
                            const typename C::P p = pts[j];
                            L.offer(C::dist(qx, qy, qz, p), p);
                        }
                    }
                }
            }
            // least gap to a face of the visited box that still has cells behind it
            double g = INFINITY;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (qc[a] - r > 0) g = fmin(g, __dsub_rd(qd[a], (lo0[a] + (double)((qc[a] - r) * step)) * e0p));
                if (qc[a] + r < nc[a] - 1) g = fmin(g, __dsub_rd((lo0[a] + (double)((qc[a] + r + 1) * step)) * e0p, qd[a]));
            }
            if (g == INFINITY) return true;  // every cell of the batch visited
            if (L.settled(C::bound(g), k)) return true;
        }
    }
    // small batch, or a query the rings did not settle: every point of the batch
    L.reset();
    for (int j = start; j < start + count; ++j) {
        const typename C::P p = pts[j];
        L.offer(C::dist(qx, qy, qz, p), p);
    }
    return false;
}

template <typename T, typename Coll>
__global__ void __launch_bounds__(KNN_THREADS, Coll::min_blocks) knn_grid_search_kernel(
    const T *__restrict__ query, int nq, int ld, int col, int bcol, int nb, int k, const KnnBatch *__restrict__ bt,
    const typename KnnT<T>::P *__restrict__ pts, const unsigned long long *__restrict__ hkeys, const int32_t *__restrict__ hlo,
    const int32_t *__restrict__ hhi, uint32_t cap, const typename Coll::Out out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const T *qp = query + (int64_t)q * ld;
    const int b = knn_row_batch(qp, bcol, nb);
    Coll L;
    L.begin(out);
    if (b >= 0 && bt[b].count > 0) knn_walk<T, Coll>(L, qp[col], qp[col + 1], qp[col + 2], b, k, true, bt, pts, hkeys, hlo, hhi, cap);
    L.store(out, q, k);
}

// ---------------------------------------------------------------------------------------------------------------
// Point normals from all-ties K-neighbourhoods (fpcc_knn_normals, DESIGN 3.8), int32 rows, the query set = the
// reference set.  Per query p: d_K = the K-th least squared distance to the rows of its own batch (KnnList walk);
// N(p) = every row at distance <= d_K (KnnMoments walk); M = n sum d d^T - (sum d)(sum d)^T over the offsets d of N(p),
// exact in 128-bit integers and rounded once to double; the normal = the unit eigenvector of M's least eigenvalue
// (cyclic Jacobi in double), zero when n < 3 or rank M <= 1.
// Bound: |c| < 2^30 (the search's own).  Then |d| < 2^31, every product d_i d_j < 2^62 fits int64, and with n < 2^31
// rows sum d < 2^62, sum d_i d_j < 2^93, n sum d_i d_j and (sum d_i)(sum d_j) < 2^124: M fits signed 128 bits.
typedef __int128 i128;
typedef unsigned __int128 u128;

// every row at distance <= lim: their number, the sums of their offsets and of the offsets' products
struct KnnMoments {
    typedef unsigned long long D;
    static constexpr int min_blocks = 2;
    int qx, qy, qz;
    D lim;
    int n;
    long long s[3];
    i128 m[6];  // xx, yy, zz, xy, xz, yz
    __device__ __forceinline__ void reset() {
        n = 0;
        s[0] = s[1] = s[2] = 0;
#pragma unroll
        for (int j = 0; j < 6; ++j) m[j] = 0;
    }
    __device__ __forceinline__ void offer(D d, const int4 &p) {
        if (d > lim) return;
        const long long dx = (long long)p.x - qx, dy = (long long)p.y - qy, dz = (long long)p.z - qz;
        ++n; s[0] += dx; s[1] += dy; s[2] += dz;
        m[0] += dx * dx; m[1] += dy * dy; m[2] += dz * dz; m[3] += dx * dy; m[4] += dx * dz; m[5] += dy * dz;
    }
    // strictly beyond: a row at exactly lim may still be unvisited
    __device__ __forceinline__ bool settled(D bnd, int) const { return bnd > lim; }
};

// round-to-nearest-even conversion of a 128-bit integer (one rounding: the bits below the top 64 fold into a sticky
// bit, which sits below the rounding position of a 64-bit value of more than 53 significant bits)
__device__ __forceinline__ double knn_i128_to_double(i128 v) {
    const bool neg = v < 0;
    u128 u = neg ? (u128)0 - (u128)v : (u128)v;
    const unsigned long long hi = (unsigned long long)(u >> 64);
    double r;
    if (hi == 0) {
        r = __ull2double_rn((unsigned long long)u);
    } else {
        const int sh = 64 - __clzll((long long)hi);  // 1..64: u >> sh fits 64 bits
        const u128 low = u & (((u128)1 << sh) - 1);
        r = __ull2double_rn((unsigned long long)(u >> sh) | (low != 0)) * knn_pow2(sh);
    }
    return neg ? -r : r;
}

// a * b == c * c for 0 <= a, b, |c| < 2^127, in 256 bits
__device__ __forceinline__ void knn_mul256(u128 a, u128 b, u128 &hi, u128 &lo) {
    const unsigned long long a0 = (unsigned long long)a, a1 = (unsigned long long)(a >> 64);
    const unsigned long long b0 = (unsigned long long)b, b1 = (unsigned long long)(b >> 64);
    const u128 p00 = (u128)a0 * b0, p01 = (u128)a0 * b1, p10 = (u128)a1 * b0, p11 = (u128)a1 * b1;
    const u128 mid = (p00 >> 64) + (unsigned long long)p01 + (unsigned long long)p10;  // < 3 * 2^64
    lo = (u128)(unsigned long long)p00 | (mid << 64);
    hi = p11 + (p01 >> 64) + (p10 >> 64) + (mid >> 64);
}
__device__ __forceinline__ bool knn_minor_zero(i128 a, i128 b, i128 c) {
    const u128 uc = c < 0 ? (u128)0 - (u128)c : (u128)c;
    u128 h1, l1, h2, l2;
    knn_mul256((u128)a, (u128)b, h1, l1);
    knn_mul256(uc, uc, h2, l2);
    return h1 == h2 && l1 == l2;
}

constexpr int KNN_JACOBI_SWEEPS = 16;  // a cap: convergence is quadratic, a 3 x 3 matrix is expected to stop well before

// eigenvector of the least eigenvalue of the symmetric a (xx, yy, zz, xy, xz, yz), cyclic Jacobi; unit length
__device__ __forceinline__ void knn_least_eigvec(const double a[6], double &vx, double &vy, double &vz) {
    double A[3][3] = {{a[0], a[3], a[4]}, {a[3], a[1], a[5]}, {a[4], a[5], a[2]}};
    double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < KNN_JACOBI_SWEEPS; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int P = pq == 2 ? 1 : 0, Q = pq == 0 ? 1 : 2;
            const double apq = A[P][Q];
            // negligible against both diagonal entries (relative to the eigenvalues they converge to)
            if (fabs(apq) <= 1e-18 * sqrt(fabs(A[P][P]) * fabs(A[Q][Q])) || apq == 0.0) continue;
            rotated = true;
            const double theta = (A[Q][Q] - A[P][P]) / (2.0 * apq);
            const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
            const int R = 3 - P - Q;
            const double arp = A[R][P], arq = A[R][Q];
            A[P][P] -= t * apq;
            A[Q][Q] += t * apq;
            A[P][Q] = A[Q][P] = 0.0;
            A[R][P] = A[P][R] = c * arp - sn * arq;
            A[R][Q] = A[Q][R] = sn * arp + c * arq;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const double vp = V[i][P], vq = V[i][Q];
                V[i][P] = c * vp - sn * vq;
                V[i][Q] = sn * vp + c * vq;
            }
        }
        if (!rotated) break;
    }
    // the least diagonal entry, the lowest index on a tie (selects, not a run-time index: the arrays stay in registers)
    const bool m1 = A[1][1] < A[0][0];
    const double l01 = m1 ? A[1][1] : A[0][0];
    const bool m2 = A[2][2] < l01;
    const double x = m2 ? V[0][2] : (m1 ? V[0][1] : V[0][0]);
    const double y = m2 ? V[1][2] : (m1 ? V[1][1] : V[1][0]);
    const double z = m2 ? V[2][2] : (m1 ? V[2][1] : V[2][0]);
    const double inv = 1.0 / sqrt(x * x + y * y + z * z);
    vx = x * inv; vy = y * inv; vz = z * inv;
}

struct KnnView {  // the orientation reference: use = 0 -> the largest component positive
    double x, y, z;
    int use;
};

template <int KB>
__global__ void __launch_bounds__(KNN_THREADS, 2) knn_normals_kernel(
    const int32_t *__restrict__ rows, int n, int ld, int col, int bcol, int nb, int k, const KnnBatch *__restrict__ bt,
    const int4 *__restrict__ pts, const unsigned long long *__restrict__ hkeys, const int32_t *__restrict__ hlo,
    const int32_t *__restrict__ hhi, uint32_t cap, KnnView view, float *__restrict__ normal_out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int32_t *qp = rows + (int64_t)q * ld;
    const int b = knn_row_batch(qp, bcol, nb);
    const int qx = qp[col], qy = qp[col + 1], qz = qp[col + 2];
    float *o = normal_out + 3 * (int64_t)q;
    double nx = 0.0, ny = 0.0, nz = 0.0;
    if (b >= 0) {  // the query is a row of its own batch: count >= 1
        // phase 1: d_K (far when the batch has fewer than k rows: N(p) is then the whole batch)
        KnnList<int32_t, KB> L;
        L.reset();
        const bool rings = knn_walk<int32_t>(L, qx, qy, qz, b, k, true, bt, pts, hkeys, hlo, hhi, cap);
        unsigned long long dk = L.d[0];
        int rk = L.r[0];
#pragma unroll
        for (int j = 1; j < KB; ++j) {
            dk = j < k ? L.d[j] : dk;
            rk = j < k ? L.r[j] : rk;
        }
        // phase 2: every row at <= d_K; a query whose phase 1 ended in the batch scan scans again
        KnnMoments S;
        S.qx = qx; S.qy = qy; S.qz = qz;
        S.lim = rk == INT_MAX ? ~0ull : dk;
        S.reset();
        knn_walk<int32_t>(S, qx, qy, qz, b, k, rings, bt, pts, hkeys, hlo, hhi, cap);
        if (S.n >= 3) {
            const i128 nn = S.n;
            i128 M[6];
            M[0] = nn * S.m[0] - (i128)S.s[0] * S.s[0];
            M[1] = nn * S.m[1] - (i128)S.s[1] * S.s[1];
            M[2] = nn * S.m[2] - (i128)S.s[2] * S.s[2];
            M[3] = nn * S.m[3] - (i128)S.s[0] * S.s[1];
            M[4] = nn * S.m[4] - (i128)S.s[0] * S.s[2];
            M[5] = nn * S.m[5] - (i128)S.s[1] * S.s[2];
            // M is positive semidefinite: rank <= 1 exactly when every 2 x 2 principal minor vanishes
            const bool flat = knn_minor_zero(M[0], M[1], M[3]) && knn_minor_zero(M[0], M[2], M[4]) &&
                              knn_minor_zero(M[1], M[2], M[5]);
            if (!flat) {
                double a[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) a[j] = knn_i128_to_double(M[j]);
                knn_least_eigvec(a, nx, ny, nz);
                bool flip;
                if (view.use) {
                    const double dot = nx * (view.x - (double)qx) + ny * (view.y - (double)qy) + nz * (view.z - (double)qz);
                    flip = dot < 0.0;
                } else {  // the component of largest magnitude positive, the lowest axis on a tie
                    const bool y1 = fabs(ny) > fabs(nx);
                    const double top = y1 ? ny : nx;
                    flip = (fabs(nz) > fabs(top) ? nz : top) < 0.0;
                }
                if (flip) { nx = -nx; ny = -ny; nz = -nz; }
            }
        }
    }
    o[0] = (float)nx; o[1] = (float)ny; o[2] = (float)nz;
}

static inline size_t knn_a256(size_t b) { return (b + 255) & ~(size_t)255; }
static inline uint32_t knn_capacity(int64_t n_ref) { return (uint32_t)(2 * n_ref + 64); }

struct KnnGrid {  // the cell grid of the reference rows, in the workspace
    KnnBatch *bt;
    void *pts;
    unsigned long long *hkeys;
    int32_t *hlo, *hhi;
    uint32_t cap;
};

// target: points per occupied cell (knn_level_kernel)
template <typename T>
static int knn_build(int target, int nb, const T *ref, int nr, int r_ld, int r_col, int r_bcol, void *workspace,
                     size_t workspace_bytes, cudaStream_t s, KnnGrid &g) {
    char *w = (char *)workspace;
    const uint32_t cap = knn_capacity(nr);
    KnnBatch *bt = (KnnBatch *)w; w += knn_a256((size_t)nb * sizeof(KnnBatch));
    unsigned long long *keys = (unsigned long long *)w; w += knn_a256((size_t)(nr > 0 ? nr : 1) * 8);
    unsigned long long *keys_s = (unsigned long long *)w; w += knn_a256((size_t)(nr > 0 ? nr : 1) * 8);
    int32_t *rows = (int32_t *)w; w += knn_a256((size_t)(nr > 0 ? nr : 1) * 4);
    int32_t *rows_s = (int32_t *)w; w += knn_a256((size_t)(nr > 0 ? nr : 1) * 4);
    void *pts = w; w += knn_a256((size_t)(nr > 0 ? nr : 1) * 16);
    unsigned long long *hkeys = (unsigned long long *)w; w += knn_a256((size_t)cap * 8);
    int32_t *hlo = (int32_t *)w; w += knn_a256((size_t)cap * 4);
    int32_t *hhi = (int32_t *)w; w += knn_a256((size_t)cap * 4);
    size_t tmp_bytes = workspace_bytes - (size_t)(w - (char *)workspace);
    g = KnnGrid{bt, pts, hkeys, hlo, hhi, cap};
    knn_init_kernel<<<ceil_div(nb, 256), 256, 0, s>>>(bt, nb);
    FPCC_LAUNCH_CHECK();
    if (nr > 0) {
        FPCC_CUDA(cudaMemsetAsync(hkeys, 0, (size_t)cap * 8, s));
        knn_bbox_kernel<T><<<ceil_div(ceil_div(nr, KNN_CHUNK), 256), 256, 0, s>>>(ref, nr, r_ld, r_col, r_bcol, nb, bt);
        knn_setup_kernel<T><<<1, 1024, 0, s>>>(bt, nb);
        knn_key_kernel<T><<<ceil_div(nr, 256), 256, 0, s>>>(ref, nr, r_ld, r_col, r_bcol, nb, bt, keys, rows);
        FPCC_LAUNCH_CHECK();
        FPCC_CUDA(cub::DeviceRadixSort::SortPairs(w, tmp_bytes, keys, keys_s, rows, rows_s, nr, 0, 64, s));
        knn_hist_kernel<<<ceil_div(nr, 256), 256, 0, s>>>(keys_s, nr, bt);
        knn_level_kernel<<<1, 1024, 0, s>>>(bt, nb, target);
        knn_cell_kernel<T><<<ceil_div(nr, 256), 256, 0, s>>>(ref, nr, r_ld, r_col, keys_s, rows_s, bt,
                                                             (typename KnnT<T>::P *)pts, hkeys, hlo, hhi, cap);
        FPCC_LAUNCH_CHECK();
    }
    return FPCC_OK;
}

template <typename T, typename Coll>
static int knn_launch(const T *query, int nq, int ld, int col, int bcol, int nb, int k, const KnnGrid &g,
                      const typename Coll::Out &out, cudaStream_t s) {
    if (nq == 0) return FPCC_OK;
    knn_grid_search_kernel<T, Coll><<<ceil_div(nq, KNN_THREADS), KNN_THREADS, 0, s>>>(
        query, nq, ld, col, bcol, nb, k, g.bt, (const typename KnnT<T>::P *)g.pts, g.hkeys, g.hlo, g.hhi, g.cap, out);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

// cell size of the K-NN search: a few points per occupied cell for small K, about K/2 for large K (the 27 cells around
// a query then hold several times K points)
static inline int knn_target(int k) { return k / 2 > 4 ? k / 2 : 4; }

template <typename T>
static int knn_run(int k, int nb, const T *query, int nq, int q_ld, int q_col, int q_bcol, const T *ref, int nr, int r_ld,
                   int r_col, int r_bcol, void *dist, int32_t *idx, void *workspace, size_t workspace_bytes, cudaStream_t s) {
    KnnGrid g;
    const int rc = knn_build<T>(knn_target(k), nb, ref, nr, r_ld, r_col, r_bcol, workspace, workspace_bytes, s, g);
    if (rc != FPCC_OK) return rc;
    typedef typename KnnT<T>::D D;
#define FPCC_KNN_CASE(KB)                                                                                                   \
    return knn_launch<T, KnnList<T, KB>>(query, nq, q_ld, q_col, q_bcol, nb, k, g, {(D *)dist, idx}, s)
    if (k <= 1) FPCC_KNN_CASE(1);
    else if (k <= 2) FPCC_KNN_CASE(2);
    else if (k <= 4) FPCC_KNN_CASE(4);
    else if (k <= 8) FPCC_KNN_CASE(8);
    else if (k <= 16) FPCC_KNN_CASE(16);
    else FPCC_KNN_CASE(32);
#undef FPCC_KNN_CASE
}

static int knn_normals_run(int k, int nb, const int32_t *rows, int n, int ld, int col, int bcol, const KnnView &view,
                           float *normal_out, void *workspace, size_t workspace_bytes, cudaStream_t s) {
    KnnGrid g;
    const int rc = knn_build<int32_t>(knn_target(k), nb, rows, n, ld, col, bcol, workspace, workspace_bytes, s, g);
    if (rc != FPCC_OK) return rc;
    if (n == 0) return FPCC_OK;
#define FPCC_NORMALS_CASE(KB)                                                                                               \
    knn_normals_kernel<KB><<<ceil_div(n, KNN_THREADS), KNN_THREADS, 0, s>>>(rows, n, ld, col, bcol, nb, k, g.bt,           \
                                                                           (const int4 *)g.pts, g.hkeys, g.hlo, g.hhi,     \
                                                                           g.cap, view, normal_out)
    if (k <= 4) FPCC_NORMALS_CASE(4);
    else if (k <= 8) FPCC_NORMALS_CASE(8);
    else if (k <= 16) FPCC_NORMALS_CASE(16);
    else FPCC_NORMALS_CASE(32);
#undef FPCC_NORMALS_CASE
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

static bool knn_layout_ok(int ld, int col, int bcol) {
    if (col < 0 || ld < col + 3) return false;
    if (bcol < 0) return true;
    return bcol < ld && (bcol < col || bcol >= col + 3);
}


}  // namespace fpcc

using namespace fpcc;

extern "C" int fpcc_nn_search(const int32_t *query, int nq, int q_ld, int q_col, const int32_t *ref, int nr, int r_ld,
                              int r_col, int coord_bits, int64_t *d2_out, int32_t *idx_out, void *stream) {
    FPCC_REQUIRE(query && ref && d2_out, "nn_search: NULL pointer");
    FPCC_REQUIRE(nq > 0 && nr > 0, "nn_search: empty cloud (nq=%d nr=%d)", nq, nr);
    FPCC_REQUIRE(q_ld >= 3 + q_col && r_ld >= 3 + r_col && q_col >= 0 && r_col >= 0, "nn_search: bad row layout");
    FPCC_REQUIRE(coord_bits >= 1 && coord_bits <= 30, "nn_search: coord_bits must be in 1..30");
    const int grid = ceil_div(nq, NN_THREADS * NN_QPT);
    cudaStream_t s = (cudaStream_t)stream;
    if (coord_bits <= 14)  // |d| < 2^15 per axis with signed slack: 3 * 2^30 < 2^32
        nn_kernel<uint32_t><<<grid, NN_THREADS, 0, s>>>(query, nq, q_ld, q_col, ref, nr, r_ld, r_col, d2_out, idx_out);
    else
        nn_kernel<uint64_t><<<grid, NN_THREADS, 0, s>>>(query, nq, q_ld, q_col, ref, nr, r_ld, r_col, d2_out, idx_out);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

extern "C" size_t fpcc_knn_workspace(int64_t n_ref, int n_batch) {
    if (n_ref < 1) n_ref = 1;
    if (n_batch < 1) n_batch = 1;
    size_t sort_tmp = 0;
    cub::DeviceRadixSort::SortPairs((void *)nullptr, sort_tmp, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, (int)n_ref, 0, 64);
    const size_t cap = knn_capacity(n_ref);
    return knn_a256((size_t)n_batch * sizeof(KnnBatch)) + 2 * knn_a256((size_t)n_ref * 8) + 2 * knn_a256((size_t)n_ref * 4) +
           knn_a256((size_t)n_ref * 16) + knn_a256(cap * 8) + 2 * knn_a256(cap * 4) + knn_a256(sort_tmp);
}

// the row checks of fpcc_knn_search and fpcc_nn_tie_attr, messages prefixed with the entry point's name
static int knn_check_rows(const char *who, int n_batch, int64_t nq, int q_ld, int q_col, int q_batch_col, int64_t nr,
                          int r_ld, int r_col, int r_batch_col) {
    FPCC_REQUIRE(n_batch >= 1 && n_batch <= 1023, "%s: n_batch must be in 1..1023 (10-bit batch field of the cell keys), got %d",
                 who, n_batch);
    FPCC_REQUIRE(nq >= 0 && nr >= 0 && nq < ((int64_t)1 << 31) && nr < ((int64_t)1 << 31),
                 "%s: row counts must be in 0..2^31-1 (nq=%lld nr=%lld)", who, (long long)nq, (long long)nr);
    FPCC_REQUIRE((q_batch_col < 0) == (r_batch_col < 0), "%s: a batch column is needed on both sides or on neither", who);
    FPCC_REQUIRE(q_batch_col >= 0 || n_batch == 1, "%s: one cloud (no batch column) needs n_batch = 1", who);
    FPCC_REQUIRE(knn_layout_ok(q_ld, q_col, q_batch_col) && knn_layout_ok(r_ld, r_col, r_batch_col),
                 "%s: bad row layout (q: ld %d col %d batch col %d, ref: ld %d col %d batch col %d)", who, q_ld, q_col,
                 q_batch_col, r_ld, r_col, r_batch_col);
    return FPCC_OK;
}

static int knn_check_workspace(const char *who, const void *workspace, size_t workspace_bytes, int64_t nr, int n_batch) {
    FPCC_REQUIRE(((uintptr_t)workspace & 15) == 0, "%s: workspace must be 16-byte aligned", who);
    const size_t need = fpcc_knn_workspace(nr, n_batch);
    FPCC_REQUIRE(workspace_bytes >= need, "%s: workspace too small (%zu < %zu bytes)", who, workspace_bytes, need);
    return FPCC_OK;
}

extern "C" int fpcc_knn_search(int coord_type, int k, int n_batch, const void *query, int64_t nq, int q_ld, int q_col,
                               int q_batch_col, const void *ref, int64_t nr, int r_ld, int r_col, int r_batch_col,
                               void *dist_out, int32_t *idx_out, void *workspace, size_t workspace_bytes, void *stream) {
    FPCC_REQUIRE(coord_type == 0 || coord_type == 1, "knn_search: coord_type must be 0 (int32) or 1 (float32), got %d", coord_type);
    FPCC_REQUIRE(k >= 1 && k <= 32, "knn_search: k must be in 1..32, got %d", k);
    int rc = knn_check_rows("knn_search", n_batch, nq, q_ld, q_col, q_batch_col, nr, r_ld, r_col, r_batch_col);
    if (rc != FPCC_OK) return rc;
    FPCC_REQUIRE(workspace && (nq == 0 || (query && dist_out && idx_out)) && (nr == 0 || ref), "knn_search: NULL pointer");
    rc = knn_check_workspace("knn_search", workspace, workspace_bytes, nr, n_batch);
    if (rc != FPCC_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (coord_type == 0)
        return knn_run<int32_t>(k, n_batch, (const int32_t *)query, (int)nq, q_ld, q_col, q_batch_col, (const int32_t *)ref,
                                (int)nr, r_ld, r_col, r_batch_col, dist_out, idx_out, workspace, workspace_bytes, s);
    return knn_run<float>(k, n_batch, (const float *)query, (int)nq, q_ld, q_col, q_batch_col, (const float *)ref, (int)nr,
                          r_ld, r_col, r_batch_col, dist_out, idx_out, workspace, workspace_bytes, s);
}

extern "C" int fpcc_nn_tie_attr(int n_batch, const int32_t *query, int64_t nq, int q_ld, int q_col, int q_batch_col,
                                const int32_t *ref, int64_t nr, int r_ld, int r_col, int r_batch_col, const uint8_t *ref_rgb,
                                int64_t *d2_out, int32_t *count_out, int64_t *sum_out, void *workspace,
                                size_t workspace_bytes, void *stream) {
    int rc = knn_check_rows("nn_tie_attr", n_batch, nq, q_ld, q_col, q_batch_col, nr, r_ld, r_col, r_batch_col);
    if (rc != FPCC_OK) return rc;
    FPCC_REQUIRE(workspace && (nq == 0 || (query && d2_out && count_out && sum_out)) && (nr == 0 || (ref && ref_rgb)),
                 "nn_tie_attr: NULL pointer");
    rc = knn_check_workspace("nn_tie_attr", workspace, workspace_bytes, nr, n_batch);
    if (rc != FPCC_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    KnnGrid g;
    rc = knn_build<int32_t>(4, n_batch, ref, (int)nr, r_ld, r_col, r_batch_col, workspace, workspace_bytes, s, g);  // the K = 1 cells
    if (rc != FPCC_OK) return rc;
    return knn_launch<int32_t, KnnTie>(query, (int)nq, q_ld, q_col, q_batch_col, n_batch, 1, g,
                                       {ref_rgb, d2_out, count_out, sum_out}, s);
}

extern "C" int fpcc_knn_normals(int k, int n_batch, const int32_t *pts, int64_t n, int ld, int col, int batch_col,
                                const double *viewpoint, float *normal_out, void *workspace, size_t workspace_bytes,
                                void *stream) {
    FPCC_REQUIRE(k >= 3 && k <= 32, "knn_normals: k must be in 3..32, got %d", k);
    int rc = knn_check_rows("knn_normals", n_batch, n, ld, col, batch_col, n, ld, col, batch_col);
    if (rc != FPCC_OK) return rc;
    FPCC_REQUIRE(workspace && (n == 0 || (pts && normal_out)), "knn_normals: NULL pointer");
    rc = knn_check_workspace("knn_normals", workspace, workspace_bytes, n, n_batch);
    if (rc != FPCC_OK) return rc;
    KnnView view = {0.0, 0.0, 0.0, 0};
    if (viewpoint) {
        FPCC_REQUIRE(isfinite(viewpoint[0]) && isfinite(viewpoint[1]) && isfinite(viewpoint[2]),
                     "knn_normals: viewpoint must be three finite numbers");
        view = KnnView{viewpoint[0], viewpoint[1], viewpoint[2], 1};
    }
    return knn_normals_run(k, n_batch, pts, (int)n, ld, col, batch_col, view, normal_out, workspace, workspace_bytes,
                           (cudaStream_t)stream);
}
