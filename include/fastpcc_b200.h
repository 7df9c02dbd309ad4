/*
 * fastpcc_b200.h -- C ABI of the B200-native (sm_100a) sparse-convolution codec hot path.
 *
 * Drop-in boundary for FastPCC's operator layer (SURVEY.md 8b).  Every entry point takes plain
 * device/host pointers, sizes and a CUDA stream (cudaStream_t passed as void*); none takes a torch
 * type.  All functions return 0 on success and a negative code otherwise; fpcc_last_error() returns
 * the message of the last failure on the calling thread (the Python shim raises RuntimeError with it,
 * mirroring the reference's TORCH_CHECK behaviour).  Nothing synchronises the device unless stated.
 *
 * Reference interfaces replaced (file:line under pengpeng-yu/FastPCC):
 *   lib/int_sparse_conv/src/binding.cu:114-145            pybind11 module `int_sparse_conv_ext`
 *   lib/int_sparse_conv/src/hashmap/hashmap_cuda.cuh      GPUHashTable::{insert_coords,lookup_coords}
 *   lib/int_sparse_conv/src/gather_gemm_scatter.cu:157    cutlass_gather_gemm_scatter_int8
 *   lib/int_sparse_conv/src/gemm.cu:140                   cutlass_gemm_int8
 *   lib/int_sparse_conv/src/element_wise/*.cu             {,bias_,prelu_,bias_prelu_}requant_to_int{8,16,32}, prelu
 *   lib/int_sparse_conv/src/softmax.cu:119                softmax_int32
 *   lib/space_filling_curves/src/morton3d.cu:39           morton3d_encode_magicbits
 *   models/convolutional/lossy_coord_v3/rans_coder/simple_rans_wrapper.cpp:272-286   RansEncoder / RansDecoder
 *   lib/entropy_models/rans_coder/rans_wrapper.cpp:430-451  IndexedRansCoder / BinaryRansCoder / batched_pmf_to_quantized_cdf
 *   models/convolutional/lossl_coord_int/model.py:261-295, 344-353, 81-91   get_bin / batch_quantize_pmf_torch / child generation
 *   lib/knn3d/src/knn3d.cu:25,75                        KNearestNeighborKernelV0/V2 (fpcc_knn_search)
 *   lib/entropy_models/distributions/deep_factorized.py   NoisyDeepFactorized likelihood (fpcc_factorized_*; not a verified drop-in)
 *   lib/entropy_models/distributions/ (noisy normal), continuous_indexed.py   Gaussian conditional likelihood and indexed
 *                                                       tables (fpcc_gaussian_*; not a verified drop-in)
 */
#ifndef FASTPCC_B200_H_
#define FASTPCC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FPCC_OK 0
#define FPCC_ERR_INVALID (-1) /* bad argument (shape, alignment, range)            */
#define FPCC_ERR_CUDA (-2)    /* a CUDA runtime call or launch failed               */
#define FPCC_ERR_UNSUPPORTED (-3)

/* output element types of the requant epilogues */
#define FPCC_OUT_I8 0
#define FPCC_OUT_I16 1
#define FPCC_OUT_I32 2

const char *fpcc_last_error(void);
int fpcc_version(void);
/* Fills major/minor/SM count of the current device; fails unless it is an sm_100 part. */
int fpcc_device_check(int *cc_major, int *cc_minor, int *sm_count);

/* ------------------------------------------------------------------------------------------------
 * Coordinates, hashing, kernel maps.  Coordinates are int32 [n,4].  `layout` = 0 for the model-side
 * order (batch,x,y,z) and 1 for the permuted order (x,y,z,batch) that the reference passes to its
 * hash table (cuda_ops.py:120).  0 <= x,y,z < 2^18, 0 <= batch < 1023 (rows outside that range are
 * not inserted and never match).
 * The table is the caller's pair of zero-initialised arrays (int64 keys[cap], int32 vals[cap]) exactly
 * as in cuda_ops.py:117-119; 0 marks an empty slot; values are row index + 1.
 * ---------------------------------------------------------------------------------------------- */

/* replaces GPUHashTable::insert_coords (hashmap_cuda.cuh:171-191, 286-303) */
int fpcc_hash_insert_coords(int64_t *keys, int32_t *vals, int capacity,
                            const int32_t *coords, int n, int layout, void *stream);

/* replaces GPUHashTable::lookup_coords (hashmap_cuda.cuh:221-275, 339-348).
 * For every output coordinate o and kernel index k: neighbour = o*stride + offset(k), offsets
 * enumerated as in the reference (odd kernel volume: x fastest, even: z fastest; per-axis offset
 * k%ks - (ks-1)/2).  Writes row index + 1 or 0.
 * k_major = 1 writes table[k*ld + o] (ld >= n_out), k_major = 0 writes table[o*kvol + k] (the
 * reference's layout).  Every entry of the addressed region is written (no pre-zeroing needed).
 * convention 0 = the torchsparse-derived rule above (compact per-level coordinates).  convention 1 =
 * MinkowskiEngine HYPER_CUBE (lib/minkowski_sparse_conv_layers.py; offsets as minkowski_expand_coord_2x :401-408):
 * absolute coordinates, neighbour = o + offset(k) * s, x fastest for every kernel, odd kernels centred, even
 * kernels 0..k-1, with s = the input tensor stride. */
int fpcc_kmap_lookup(const int64_t *keys, const int32_t *vals, int capacity,
                     const int32_t *out_coords, int n_out, int layout,
                     int ksx, int ksy, int ksz, int sx, int sy, int sz, int convention,
                     int32_t *table, int k_major, int64_t ld, void *stream);

/* replaces the host-synchronising compaction at cuda_ops.py:132-151.  table is k-major [kvol, ld].
 * Produces offset-major pair lists (output index ascending inside each offset): in_map/out_map hold
 * sum(counts) entries, offsets[k] = start of offset k, offsets[kvol] = total.  `omit_k` (or -1) is
 * skipped (its count is 0).  workspace: fpcc_kmap_compact_workspace(kvol, n_out) bytes. */
size_t fpcc_kmap_compact_workspace(int kvol, int n_out);
int fpcc_kmap_compact(const int32_t *table, int kvol, int n_out, int64_t ld, int omit_k,
                      int32_t *in_map, int32_t *out_map, int32_t *offsets /* [kvol+1] */,
                      void *workspace, size_t workspace_bytes, void *stream);

/* 3x3x3, stride-1 neighbour table of a pyramid level from the table of its PARENT level (octree neighbour finding)
 * instead of hash probes: same values as fpcc_kmap_lookup(ks = 3, stride = 1) on the level's coordinates (the
 * reference rebuilds a hash table per level, hashmap_cuda.cuh:171-275).  coarse_table: k-major [27, ld_coarse] of
 * the parent level; coarse_occ[j] bit 7-s = child slot s = 4x+2y+z of parent j exists; child_base[j] = row of its
 * first child (children stored in slot order); parent / slot: per fine node. */
int fpcc_kmap_from_parent(const int32_t *coarse_table, int64_t ld_coarse, int n_coarse, const uint8_t *coarse_occ,
                          const int32_t *child_base, const int32_t *parent, const uint8_t *slot, int n_fine,
                          int32_t *table, int64_t ld, void *stream);

/* Row grouping for fpcc_spconv_*: masks[o] = OR_k (table[k*ld+o] != 0) << min(k,31) (non-negative int32, the sort
 * key), and out[k*ld_out + j] = table[k*ld + perm[j]] for a permutation `perm` of the output rows (e.g. the
 * argsort of the masks).  No reference counterpart: the reference runs one GEMM per offset on pair lists
 * (cuda_ops.py:132-169); this is the equivalent compaction for the output-stationary kernel. */
int fpcc_kmap_row_masks(const int32_t *table, int kvol, int n_out, int64_t ld, int32_t *masks, void *stream);
int fpcc_kmap_permute(const int32_t *table, int kvol, int n_out, int64_t ld, const int32_t *perm, int32_t *out,
                      int64_t ld_out, void *stream);

/* replaces Model.get_bin (lossl_coord_int/model.py:261-295): coords must be sorted so that the 8
 * children of a parent are contiguous (x-major Morton order, batch-major).  Writes parent coords
 * (coords>>1, unique_consecutive), the 8-bit child occupancy of each parent
 * (bit 7-k set <=> child k = 4*(x&1)+2*(y&1)+(z&1) present, so oct symbol = occ-1), the parent row of
 * every child and its slot k (both optional).  *n_out_dev (device int32) receives the parent count.
 * Buffers sized for n rows.  workspace: fpcc_scan_workspace(n) bytes. */
size_t fpcc_scan_workspace(int n);
int fpcc_downsample(const int32_t *coords, int n, int32_t *out_coords, uint8_t *out_occ,
                    int32_t *parent_of_child, uint8_t *slot_of_child, int32_t *n_out_dev,
                    void *workspace, size_t workspace_bytes, void *stream);

/* replaces `(C<<1 + unfold_kernel)[cur_bin]` (model.py:86-91,186-190,499-507): children (z fastest) of
 * every parent whose occupancy bit is set.  child_parent[j] = parent row, child_slot[j] = k (0..7).
 * *n_child_dev (device int32) receives the child count; child buffers sized for 8*n rows.
 * `shift_add`: xyz offset added to every child (the final coord_offset), may be NULL. */
int fpcc_upsample(const int32_t *coords, const uint8_t *occ, int n,
                  int32_t *child_coords, int32_t *child_parent, uint8_t *child_slot, int32_t *n_child_dev,
                  const int32_t *shift_add, void *workspace, size_t workspace_bytes, void *stream);

/* occ byte <-> the reference's [n,8] 0/1 feature layout (channel k <-> bit 7-k) */
int fpcc_occ_to_bits(const uint8_t *occ, int n, int32_t *bits_i32 /* [n,8] */, void *stream);

/* replaces morton3d_encode_magicbits (morton3d.cu:19-37).  xyz int32 [n,3] with row stride `ld` ints
 * (ld=4 and xyz pointing at column 1 encodes (b,x,y,z) rows).  msb_axis: 0 -> x most significant
 * (the reference's inverse=True / 'zyx'), 2 -> z most significant ('xyz').  63-bit codes. */
int fpcc_morton_encode(const int32_t *xyz, int64_t ld, int n, int msb_axis, int64_t *codes, void *stream);
/* dst[i] = src[idx[i]] for n rows of 16 bytes (int32 (batch,x,y,z) coordinates): applies the sort permutation
 * `xyz = xyz[order]` of models/convolutional/lossl_coord_int/model.py:396-398 (idx: int64 as torch.argsort returns). */
int fpcc_gather_rows16(const void *src, const int64_t *idx, int64_t n, void *dst, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Front end (SURVEY 8f-1): the step immediately before the codec.
 *
 * fpcc_voxelize_f32 replaces the host NumPy of lib/datasets/KITTIOdometry/dataset.py:96-102 followed by the
 * Morton argsort of dataset.py:117-118 / lossl_coord_int/model.py:398:
 *     org = xyz.min(0); xyz -= org; xyz *= scale; xyz = np.unique(xyz.round().astype(int32), axis=0); Morton sort
 * points: float32 rows of `ld` floats (x,y,z first; KITTI .bin rows have ld = 4).  Arithmetic is float32 with one
 * rounding per operation and round-half-to-even, exactly as NumPy evaluates the in-place ops.  Output: unique voxels
 * as int32 (batch,x,y,z) rows in Morton order (msb_axis as fpcc_morton_encode), min_xyz_dev[3] = org (the
 * inv_transform origin), *n_out_dev = voxel count, or -1 if a quantised coordinate does not fit `coord_bits`
 * (1..21) bits.  out_coords sized for n rows.  workspace: fpcc_voxelize_workspace(n) bytes. */
size_t fpcc_voxelize_workspace(int64_t n);
int fpcc_voxelize_f32(const float *points, int64_t n, int ld, float scale, int coord_bits, int msb_axis, int batch,
                      int32_t *out_coords, float *min_xyz_dev, int32_t *n_out_dev, void *workspace,
                      size_t workspace_bytes, void *stream);

/* One node of _kd_tree_partition (lib/data_utils.py:196-205): axis = argmax of the coordinate variance,
 * split value = kthvalue(n/2) of that axis, left = rows <= value, right = the rest, both in their input order.
 * coords / out_coords int32 [n,4] (batch,x,y,z), coordinates in [0, 2^coord_bits).  out_coords = left rows then
 * right rows; info_dev[3] (device int32) = {axis, split value, number of left rows}.  The caller recurses
 * (fastpcc_b200/frontend.py).  workspace: fpcc_kd_split_workspace(n, coord_bits) bytes. */
size_t fpcc_kd_split_workspace(int64_t n, int coord_bits);
int fpcc_kd_split(const int32_t *coords, int64_t n, int coord_bits, int32_t *out_coords, int32_t *info_dev,
                  void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Bitstream containers (SURVEY 8f-2), host memory only: the byte layouts needed to exchange streams with the
 * reference decoder.  The int64 functions return a byte count, or -1 with fpcc_last_error() set.
 *
 * frame header: lossl_coord_int/model.py:447-452 / 466-473 -- three uint16 LE coord offsets, uint16 LE bottom
 * point count; the rANS payload follows. */
int fpcc_frame_header_write(const int32_t coord_offset[3], int bottom_points, uint8_t out[8]);
int fpcc_frame_header_read(const uint8_t *data, int64_t len, int32_t coord_offset[3], int *bottom_points);
/* partition container: compress_partitions / decompress_partitions (model.py:455-463, 510-521): a 3-byte LE
 * length before every partition stream.  pack: out == NULL returns the size.  index: returns the partition
 * count (offsets / lens may be NULL to count only), -1 on a truncated container. */
int64_t fpcc_partitions_pack(const uint8_t *const *items, const int64_t *lens, int n, uint8_t *out, int64_t out_cap);
int fpcc_partitions_index(const uint8_t *data, int64_t len, int max_n, int64_t *offsets, int64_t *lens);
/* BytesListUtils.concat_bytes_list / split_bytes_list
 * (lib/entropy_models/hyperprior/noisy_deep_factorized/utils.py:8-45, 47-76): bit-packed head with the byte width
 * of every length, the LE lengths, the payloads.  concat: n >= 2 as the reference asserts, out == NULL returns
 * the size.  split: the caller knows n (as in the reference); returns the bytes consumed. */
int64_t fpcc_bytes_list_concat(const uint8_t *const *items, const int64_t *lens, int n, uint8_t *out, int64_t out_cap);
int64_t fpcc_bytes_list_split(const uint8_t *data, int64_t len, int n, int64_t *offsets, int64_t *lens);

/* ------------------------------------------------------------------------------------------------
 * Distortion metric (SURVEY 8f-3): exact nearest neighbour, the kernel under D1 / D2 PSNR.  Replaces the MPEG
 * `pc_error` subprocess of lib/metrics/pc_error_wrapper.py:40-106 (lib/evaluators.py:49-124) for geometry.
 * query / ref: int32 rows of q_ld / r_ld ints, xyz starting at column q_col / r_col ((batch,x,y,z) rows: ld 4,
 * col 1); |coordinates| < 2^coord_bits.  d2_out[nq] = exact squared distance to the nearest reference point,
 * idx_out[nq] (optional) = its row, the lowest row among equidistant ones. */
int fpcc_nn_search(const int32_t *query, int nq, int q_ld, int q_col, const int32_t *ref, int nr, int r_ld, int r_col,
                   int coord_bits, int64_t *d2_out, int32_t *idx_out, void *stream);

/* Exact K nearest neighbours, batched, on a uniform cell grid built on the reference rows inside the call (device
 * reductions, cub radix sort, open-addressing cell table; no host round trip).  Replaces lib/knn3d/src/knn3d.cu
 * (KNearestNeighborKernelV0/V2, brute force, float32, D = 3) and the search under pc_error
 * (lib/metrics/pc_error_wrapper.py:40-106); metrics.pc_error runs on it with k = 1.
 * coord_type 0: int32 coordinates, |c| < 2^30, dist_out int64 exact squared distances.  coord_type 1: finite float32
 * coordinates, dist_out float32 = ((dx*dx + dy*dy) + dz*dz) with one rounding per operation (no FMA), so NumPy float32
 * evaluating that expression gives the same bits.  Rows of q_ld / r_ld elements, xyz at column q_col / r_col.
 * Batches: q_batch_col = r_batch_col = -1 is one cloud (n_batch must be 1); otherwise both columns hold the batch id
 * (an int32, or for coord_type 1 a float32 holding an integer), queries match references of their own batch only,
 * 1 <= n_batch <= 1023, and rows whose id lies outside [0, n_batch) are ignored (as queries they get padding).
 * Output [nq, k] row-major, ascending by (distance, reference row): the lowest row wins among equal distances.
 * idx_out holds reference rows of the call (not per-batch indices); slots beyond the batch's point count get idx -1,
 * distance 0.  1 <= k <= 32; nq, nr < 2^31 (either may be 0).
 * workspace: fpcc_knn_workspace(nr, n_batch) bytes (16-byte aligned or better). */
size_t fpcc_knn_workspace(int64_t n_ref, int n_batch);
int fpcc_knn_search(int coord_type, int k, int n_batch,
                    const void *query, int64_t nq, int q_ld, int q_col, int q_batch_col,
                    const void *ref, int64_t nr, int r_ld, int r_col, int r_batch_col,
                    void *dist_out, int32_t *idx_out, void *workspace, size_t workspace_bytes, void *stream);

/* All-ties nearest neighbour with attribute sums, on the cell grid of fpcc_knn_search (same build at its k = 1 cell
 * size, same workspace: fpcc_knn_workspace(nr, n_batch)).  int32 rows as coord_type 0 of fpcc_knn_search, |c| < 2^30,
 * the same batch rules.  For every query row: d2_out[nq] int64 = d*, the least squared distance to a reference row of
 * its batch; count_out[nq] int32 = the reference rows at exactly d*; sum_out[nq,3] int64 = the per-channel sums of
 * their ref_rgb[nr,3] uint8 rows.  Integer sums: exact, independent of the visiting order.  A query whose batch has no
 * reference row gets d2 0, count 0, sums 0.  Replaces the colour neighbour search of pc_error
 * (lib/metrics/pc_error_wrapper.py:40-106) and the KNN recolour of
 * models/convolutional/lossy_coord_lossy_color/layers.py:269-333 (metrics.pc_error colours, attributes.recolor). */
int fpcc_nn_tie_attr(int n_batch, const int32_t *query, int64_t nq, int q_ld, int q_col, int q_batch_col,
                     const int32_t *ref, int64_t nr, int r_ld, int r_col, int r_batch_col, const uint8_t *ref_rgb,
                     int64_t *d2_out, int32_t *count_out, int64_t *sum_out, void *workspace, size_t workspace_bytes,
                     void *stream);

/* Point normals from all-ties K-neighbourhoods (DESIGN 3.8), on the cell grid of fpcc_knn_search (same build at its
 * k cell size, same workspace: fpcc_knn_workspace(n, n_batch)).  One set of int32 rows is both the query and the
 * reference set: n rows of ld elements, xyz at column col, |c| < 2^30, batch id at batch_col (-1: one cloud, n_batch
 * must be 1), the batch rules of fpcc_knn_search.  For every row p: d_K = the k-th least squared distance to the rows
 * of its batch (p itself counts, at 0); N(p) = every row of the batch at distance <= d_K (the whole batch when it has
 * fewer than k rows); M = n sum d d^T - (sum d)(sum d)^T over the offsets d of N(p), n = |N(p)|, exact in integers
 * and rounded once to double; normal_out[n,3] float32 = the unit eigenvector of M's least eigenvalue, solved in
 * double.  Zero vector when n < 3, when M has rank <= 1 (decided exactly), or when the batch id lies outside
 * [0, n_batch).  Orientation: viewpoint NULL: the component of largest magnitude positive, the lowest axis on a tie;
 * otherwise (three finite doubles in host memory, read during the call) normal . (viewpoint - p) >= 0.  The result
 * is a function of the point set alone, not of the row order.  3 <= k <= 32; n < 2^31. */
int fpcc_knn_normals(int k, int n_batch, const int32_t *pts, int64_t n, int ld, int col, int batch_col,
                     const double *viewpoint, float *normal_out, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * int8 GEMMs.  A [M,K] int8 row-major, B [N,K] int8 row-major (= one kernel offset's weight
 * C_out x C_in), int32 accumulation (exact; wraps, never saturates at the sizes in use).
 * ---------------------------------------------------------------------------------------------- */

/* replaces cutlass_gemm_int8 (gemm.cu): D = A*B^T + C.  c_mode 0: no C, 1: C is (N,) bias, 2: C is (M,N). */
int fpcc_gemm_i8(const int8_t *A, const int8_t *B, const int32_t *C, int c_mode, int32_t *D,
                 int M, int N, int K, void *stream);

/* replaces cutlass_gather_gemm_scatter_int8 with C == D (cuda_ops.py:163-166):
 * D[scatter[i],:] += A[gather[i],:] * B^T for i < L.  scatter indices must be distinct. */
int fpcc_gather_gemm_scatter_i8(const int8_t *A, const int8_t *B, int32_t *D,
                                const int32_t *gather_idx, const int32_t *scatter_idx,
                                int L, int N, int K, void *stream);

/* Epilogue description shared by the fused kernels and the element-wise entry points.
 * v = acc + bias[ch]; if (slope && v<0) v = rha(v*slope, 25); p = v*mul[ch] + zero_point;
 * o = clamp(rha(p, shift));  rha = round-half-away arithmetic shift (bias_prelu_requant.cu:6-37).
 * residual/post_slope (fused kernels only, out_type I32): o = prelu32(wrap32(o + residual), post_slope)
 * i.e. the tail of SparseResBlockIn32W8Out32.forward (cuda_ops.py:90).
 * row_bias/row_idx (fused linear only) fold the 8 occupancy-bit input channels of `cat(F, bin << 23)` ->
 * Linear(C+8 -> C) (model.py:63-64) into a 256-entry per-row bias table: the contraction keeps K = C. */
typedef struct {
    const int32_t *bias;         /* [ch] or NULL                                    */
    const int32_t *slope;        /* device [1] Q6.25 or NULL                        */
    const uint32_t *requant_mul; /* [ch], or [1] when mul_is_scalar                 */
    const int64_t *zero_point;   /* device [1]                                      */
    int32_t shift;               /* >= 0                                            */
    int32_t out_type;            /* FPCC_OUT_*                                      */
    int32_t mul_is_scalar;
    const int32_t *residual;     /* [rows, ch] int32 or NULL                        */
    const int32_t *post_slope;   /* device [1] Q6.25 or NULL                        */
    const int32_t *row_bias;     /* fused kernels: [256, ch] table or NULL: v += row_bias[row_idx[row]][ch] */
    const uint8_t *row_idx;      /* [rows] table row of every output row            */
    int32_t row_bias_bound;      /* max |entry| of the row_bias table if the caller knows it, else 0: lets the fused
                                  * kernels prove that acc + row_bias + bias stays inside int32 (32-bit epilogue)  */
    /* Fused second stage (tensor-core kernels, out_type FPCC_OUT_I32 only): when post_requant_mul is set the finished
     * int32 (Q8.23) value y is not stored; instead the consumer's PReLUIn32Out32 (optional, prelu.cu:6-21) and
     * RequantFxpToScaledInt8 (cuda_ops.py:473-509) run in the same epilogue and `out` receives int8 rows:
     *     out = sat8(rha(prelu(y) * post_requant_mul + post_zero_point, post_shift))
     * i.e. exactly what fpcc_prelu_i32 + fpcc_requant would produce from the int32 tensor. */
    const uint32_t *post_requant_mul;   /* device [1] or NULL */
    const int64_t *post_zero_point;     /* device [1]         */
    int32_t post_shift;                 /* 0 .. 62            */
    const int32_t *post_requant_slope;  /* device [1] Q6.25 or NULL */
    /* Dual output: with post_requant_mul AND aux_out set the int32 (Q8.23) rows are stored to `out` as usual and the second
     * stage's int8 rows go to aux_out ([rows, ch] int8) as well -- an int32 tensor with two consumers (the residual input of
     * SparseResBlockIn32W8Out32 and its input_requant, cuda_ops.py:82-92; a block output and the Requant that opens the next
     * predictor step, lossl_coord_int/model.py:147-172) leaves its producer once in each form and the stand-alone requant
     * pass over it disappears. */
    int8_t *aux_out;                    /* device [rows, ch] or NULL */
    /* int8 outputs of the fused kernels (FPCC_OUT_I8, or int32 + fused second stage without aux_out): row pitch of `out` in
     * elements, 0 = dense.  Lets a producer write the first C columns of the [rows, C + 16] buffer that the next
     * Linear(cat(F, occupancy bits)) (lossl_coord_int/model.py:63-64) contracts over -- the concatenation costs no copy. */
    int64_t out_ld;
} fpcc_epilogue;

/* replaces the 12 requant entry points of binding.cu:118-129 */
int fpcc_requant(const int32_t *in, int64_t rows, int ch, const fpcc_epilogue *ep, void *out, void *stream);
/* The same for RequantFxpToScaledInt8 (one multiplier, no bias, int8 output) with an output row pitch: row r goes to
 * out + r * out_ld (bytes; ch, out_ld % 16 == 0).  Lets the two requants in front of `Linear(cat(F, embed))`
 * (models/convolutional/lossl_coord_int/model.py:199-201) write the two column halves of ONE [rows, 2C] int8 buffer: the
 * concatenation costs no copy. */
int fpcc_requant_ld(const int32_t *in, int64_t rows, int ch, const fpcc_epilogue *ep, void *out, int64_t out_ld, void *stream);
/* replaces prelu (prelu.cu) */
int fpcc_prelu_i32(const int32_t *in, int64_t numel, const int32_t *slope, int32_t *out, void *stream);

/* Fused sparse convolution = sparse_conv_in8w8out32 (cuda_ops.py:95-169) + its epilogue
 * (cuda_ops.py:383-403) in one output-stationary kernel, driven by the k-major neighbour table of
 * fpcc_kmap_lookup (no pair lists, no atomics, no int32 round trip through HBM).
 * in_feats [n_in,c_in] int8, weight [kvol,c_out,c_in] int8, out [n_out,c_out] (ep->out_type).
 * zp_comp: optional int32 [kvol,c_out] zero-point compensation rows (cuda_ops.py:157-162).
 * row_perm: NULL, or int32 [n_out] when the table's columns were regrouped with fpcc_kmap_row_masks /
 * fpcc_kmap_permute: column j then describes output row row_perm[j] (results are identical; the kernel skips an
 * offset per 128-row tile, so tiles of equal neighbour patterns do ~2x less work on LiDAR levels). */
int fpcc_spconv_i8(const int8_t *in_feats, int n_in, int c_in,
                   const int8_t *weight, int kvol, int c_out,
                   const int32_t *nbr_table, int64_t ld, int n_out, const int32_t *row_perm,
                   const int32_t *zp_comp, const fpcc_epilogue *ep, void *out, void *stream);

/* Fused LinearIn8W8.forward (cuda_ops.py:609-635): out = epilogue(A*W^T), bias inside the epilogue.
 * Optional selection computes only chosen (row, output-block) pairs -- the "occupied children only"
 * form of Linear(C->8C) followed by the child mask (model.py:64-66): W is [n_groups*n, k]; the pairs are
 * grouped by output block g (sel_offsets[g] .. sel_offsets[g+1], device array of n_groups+1 entries, e.g.
 * from fpcc_kmap_compact over the child-slot table) and
 *     out[sel_out[i], :] = epilogue(A[sel_row[i], :] * W[g*n .. g*n+n, :]^T)   with bias/mul at g*n + col.
 * sel_row == NULL -> plain dense linear over all m rows. */
int fpcc_linear_i8(const int8_t *A, int m, int k, const int8_t *W, int n,
                   const int32_t *sel_row, const int32_t *sel_out, const int32_t *sel_offsets, int n_groups, int n_sel,
                   const fpcc_epilogue *ep, void *out, void *stream);

/* im2col for thin inputs (C_in = 1 or 8): patches[o, k*c + j] = feats[table[k*ld + o] - 1, j], 0 where the
 * table holds 0.  patches is [n_out, kp] int8 with kp >= kvol*c; columns >= kvol*c are left untouched (zero them
 * once).  A sparse conv then becomes fpcc_linear_i8 over K = kp with the weight reshaped to [C_out, kp]. */
int fpcc_gather_patches(const int8_t *feats, int c, const int32_t *table, int64_t ld, int kvol, int n_out,
                        int8_t *patches, int kp, void *stream);

/* k-major table for the selection above: table[g*ld + j] = child_parent[j]+1 if child_slot[j]==g else 0 */
/* The 8 occupancy-bit channels of `cat(F, bin << 23)` after RequantFxpToScaledInt8 (lossl_coord_int/model.py:63-64): byte k
 * (k = 0..7) of row r is q1 when bit 7-k of occ[r] is set, else q0 (the int8 images of the Q8.23 values 1.0 and 0); bytes 8..15
 * are zero.  16 bytes per row at out + r * out_ld: the tail columns of the [rows, C + 16] buffer of fpcc_epilogue::out_ld. */
int fpcc_occ_bits_q8(const uint8_t *occ, int64_t n, int q0, int q1, int8_t *out, int64_t out_ld, void *stream);
int fpcc_slot_table(const int32_t *child_parent, const uint8_t *child_slot, int n_child, int32_t *table, int64_t ld,
                    void *stream);

/* Selects the GEMM engine of fpcc_spconv_i8 / fpcc_linear_i8: 1 (default) = tcgen05 tensor-core kernels
 * wherever the shape allows (C_in % 16 == 0, C_in >= 32, C_out >= 16, kernel volume <= 32), 0 = the CUDA-core
 * (dp4a) kernels for every shape.  Both produce identical integers; the switch exists for A/B verification. */
int fpcc_set_tc_mode(int mode);
/* Persistent GEMM kernels occupy one whole SM per CTA.  When serial range-coder kernels of another CUDA stream
 * should run beside them, cap the GEMM grids at `sms` SMs (0 = all SMs) so that the coder blocks find free SMs. */
int fpcc_set_sm_budget(int sms);
/* Waiting host threads sleep instead of spinning (cudaDeviceScheduleBlockingSync) on `device`; call before the first
 * CUDA work of the process.  One process per GPU with several launching threads otherwise burns 2-3 cores per rank. */
int fpcc_set_blocking_sync(int device);
/* fp16 / bf16 twins of fpcc_spconv_i8 / fpcc_linear_i8 on tcgen05.mma.kind::f16 with fp32 accumulation in TMEM,
 * for the float layer API (MinkowskiEngine blocks of lib/minkowski_sparse_conv_layers.py:31-280, torchsparse
 * spnn.Conv3d of lossl_coord/model.py:34-46).  dtype: 0 fp16, 1 bf16 (features and weights); weight is
 * [kvol, c_out, c_in] (the layer keeps ME's [kvol, c_in, c_out] parameter and caches this transposed copy).
 * Epilogue: v = acc + bias; v = act(v); [v += residual; v = post_act(v)]; cast to out_type (0 fp16, 1 bf16, 2 fp32).
 * act codes: 0 none, 1 ReLU, 2 LeakyReLU / single-slope PReLU.  Accumulation order is fixed (offset-major, K
 * ascending), so encoder and decoder of a float codec see identical bits run to run.  c_in % 8 == 0, >= 16. */
int fpcc_spconv_f16(const void *feats, int dtype, int n_in, int c_in, const void *weight, int kvol, int c_out,
                    const int32_t *nbr_table, int64_t ld, int n_out, const int32_t *row_perm, const float *bias, int act, float slope,
                    const void *residual, int post_act, float post_slope, void *out, int out_type, void *stream);
/* Weight gradient of fpcc_spconv_f16 on the tensor cores (training; the wgrad product of MinkowskiEngine's /
 * torchsparse's backward: per kernel offset dW[k] = X[in_k]^T * dY[out_k], reference call sites train.py:359-404 via
 * loss.backward()).  x [*, c_in_p], dy [*, c_out_p] fp16 (dtype 0) / bf16 (1) rows padded to c_in_p in {128, 256} and
 * c_out_p a multiple of 64 (<= 256); in_idx / out_idx are the compacted pair lists of fpcc_kmap_compact; tiles holds
 * n_tiles int32 quadruples (offset k, first pair, end pair, 0), each at most 2048 pairs (none allowed) of ONE offset; dw is the fp32
 * [kvol, c_in, c_out] gradient, ACCUMULATED into (zero it first).  Contraction over the gathered rows: tcgen05.mma with
 * both operands MN-major; partial sums of the tiles of an offset meet in dw through fp32 atomics. */
int fpcc_spconv_wgrad_f16(const void *x, const void *dy, int dtype, int c_in_p, int c_out_p, const int32_t *in_idx,
                          const int32_t *out_idx, const int32_t *tiles, int n_tiles, float *dw, int c_in, int c_out,
                          void *stream);
/* Transposed neighbour table for the dgrad of fpcc_spconv_f16 (MinkowskiEngine's backward runs the same gather-GEMM-
 * scatter on the transposed kernel map; the training step of lossy_coord_v2 / lossy_coord_lossy_color, train.py:359-404,
 * reaches it through loss.backward()).  table: k-major [kvol, ld] with table[k, m] = input row + 1 of output row m (0 =
 * none), n_out columns used.  tt: k-major [kvol, ld_t], n_in columns written: tt[k, j] = m + 1 where table[k, m] == j + 1,
 * 0 elsewhere.  Precondition: every (k, input row) pair has at most one output row -- true for stride-1 and strided
 * HYPER_CUBE maps, maps onto an explicit target key, and the child-slot table of fpcc_slot_table -- so the result is
 * deterministic without atomics.  Entries outside 1..n_in are ignored. */
int fpcc_kmap_transpose(const int32_t *table, int kvol, int n_out, int64_t ld, int n_in, int32_t *tt, int64_t ld_t,
                        void *stream);
/* Backward of an activation fused into the fpcc_spconv_f16 / fpcc_linear_f16 epilogue, one pass over [n, c]:
 *   dz[r, j] = dy[r, j] * act'(y[r, j])  rounded once to dz_type (0 fp16, 1 bf16), rows of c_pad columns with zeros
 *              in c <= j < c_pad (the operand width of the dgrad / wgrad kernels);
 *   dbias[j] = sum_r of the unrounded products (fp32 result; NULL = not wanted).
 * dy / y: element types 0 fp16, 1 bf16, 2 fp32, row pitches ld_dy / ld_y; y is the forward OUTPUT.  act: 0 none (y may be
 * NULL), 1 ReLU, 2 LeakyReLU with slope >= 0 -- for these act'(y) is read from y alone (y > 0 ? 1 : slope).  dbias is
 * reduced from fp64 per-CTA partials in a fixed order (no float atomics), so it is reproducible bit for bit.
 * workspace: fpcc_act_grad_workspace(n, c) bytes when dbias is wanted. */
size_t fpcc_act_grad_workspace(int64_t n, int c);
int fpcc_act_grad_f16(const void *dy, int dy_type, int64_t ld_dy, const void *y, int y_type, int64_t ld_y, int64_t n, int c,
                      int act, float slope, void *dz, int dz_type, int c_pad, float *dbias, void *workspace,
                      size_t workspace_bytes, void *stream);
int fpcc_linear_f16(const void *A, int dtype, int m, int k, const void *W, int n, const int32_t *sel_row,
                    const int32_t *sel_out, const int32_t *sel_offsets, int n_groups, int n_sel, const float *bias,
                    int act, float slope, const void *residual, int post_act, float post_slope, void *out,
                    int out_type, void *stream);

/* Measures the kind::i8 tensor-pipe ceiling of the current device: every SM issues `iters` x 4 back-to-back
 * tcgen05.mma (M=128, N=n, K=32) on resident shared-memory tiles.  Synchronises.  *tops_out = int8 TOP/s. */
int fpcc_mma_i8_peak(int iters, int n, double *tops_out, void *stream);
/* 1 if a GEMM with contraction k, n output channels and `kvol` offsets runs on the tensor cores, else 0 */
int fpcc_gemm_engine(int k, int n, int kvol, int has_zp_comp);

/* ------------------------------------------------------------------------------------------------
 * Entropy head
 * ---------------------------------------------------------------------------------------------- */

/* replaces softmax_int32 (softmax.cu:41-144): int32 Q15.16 [rows,c] -> uint32 Q0.32 */
int fpcc_softmax_i32(const int32_t *in, int64_t rows, int c, uint32_t *out, void *stream);

/* replaces Model.batch_quantize_pmf_torch (model.py:344-353) without the D2H copy:
 * logits Q8.23 [rows,s] (row pitch `logits_ld` >= s elements, so a padded linear output is read in place)
 * -> inclusive uint16 CDF rows (entry s-1 = 65535) with a row pitch of `ld` >= s entries; pad entries are
 * 0xFFFF.  ld = 256 with 16-byte aligned rows selects the decoder's fast path. */
int fpcc_quantize_cdf(const int32_t *logits, int64_t logits_ld, int64_t rows, int s, uint16_t *cdf, int ld, void *stream);

/* Encoder-side fusion of the above with the symbol lookup of RansEncoder::encode
 * (simple_rans_wrapper.cpp:86-90): ranges[i] = start | (freq-1)<<16 of symbols[i] under row i.
 * Device-side symbol arrays are int32 throughout this ABI (values 0..s-1). */
int fpcc_cdf_symbol_ranges(const int32_t *logits, int64_t logits_ld, int64_t rows, int s, const int32_t *symbols,
                           uint32_t *ranges, void *stream);
/* same lookup for an explicit uint16 CDF table ([n_cdf,s], n_cdf == rows or 1) */
int fpcc_table_symbol_ranges(const uint16_t *cdf, int64_t n_cdf, int s, const int32_t *symbols, int64_t rows,
                             uint32_t *ranges, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Range coders (32-bit rANS, byte renormalisation, L = 2^23; rans_byte.h:66-165).  One independent
 * stream per frame / partition; streams are coded concurrently, each stream serially (byte-identical
 * output forbids splitting a stream).
 * ---------------------------------------------------------------------------------------------- */

/* Encodes n_streams streams.  Stream b consumes ranges[rng_off[b] .. rng_off[b+1]) -- packed
 * (start | (freq-1)<<16 | scale_bits-flag in a side array when needed) -- in REVERSE array order, i.e.
 * the array is laid out in DECODE order.  bits[i] (may be NULL = all 16) is the scale_bits of entry i
 * (16, or 1 for the Elias-gamma escape bits of IndexedRansCoder).  Output bytes of stream b end at
 * out + (b+1)*out_stride; out_len[b] receives the byte count (4-byte state header included), or -1 if
 * out_stride was too small.
 * state_io (optional, uint32 [n_streams,2] = {state x, bytes written}; initialise to {1<<23, 0}) lets a
 * stream stay open across calls exactly like RansEncoder between encode() calls: with do_flush = 0 the
 * state is stored back and out_len reports the bytes so far; do_flush = 1 writes the 4-byte state header
 * (RansEncoder::flush, simple_rans_wrapper.cpp:126-134). */
int fpcc_rans_encode(const uint32_t *ranges, const uint8_t *bits, const int64_t *rng_off, int n_streams,
                     int64_t total_entries /* = rng_off[n_streams], as a host value */,
                     uint8_t *out, int64_t out_stride, int32_t *out_len, uint32_t *state_io, int do_flush,
                     void *workspace, size_t workspace_bytes /* >= 16 * total_entries */, void *stream);

/* Decoder state of one stream (device resident, 16 bytes) */
typedef struct {
    uint32_t x;
    uint32_t pos;  /* read offset into the stream's bytes */
    uint32_t len;  /* byte count                          */
    uint32_t err;  /* nonzero once a read ran past len    */
} fpcc_rans_dec_state;

/* RansDecoder::flush (simple_rans_wrapper.cpp:139-145) for n_streams streams stored at
 * bytes + byte_off[b] with byte_len[b] bytes.  The buffer must stay readable for 512 bytes past the end of
 * the last stream (the decoders read ahead through an aligned byte window; the extra bytes are never used). */
int fpcc_rans_dec_init(fpcc_rans_dec_state *st, const uint8_t *bytes, const int64_t *byte_off,
                       const int32_t *byte_len, int n_streams, void *stream);

/* RansDecoder::decode (simple_rans_wrapper.cpp:206-239): stream b decodes symbols
 * [row_off[b], row_off[b+1]) with CDF row i (one row per symbol), the single shared row when n_cdf == 1, or
 * row b (one table per stream, e.g. the per-frame bottom-coordinate histogram) when rows_per_stream != 0;
 * s_per_stream (optional, device) overrides the alphabet size s per stream. */
int fpcc_rans_decode(fpcc_rans_dec_state *st, const uint8_t *bytes, const int64_t *byte_off,
                     const uint16_t *cdf, int64_t n_cdf, int s, int ld, const int64_t *row_off, int n_streams,
                     int32_t *symbols, int rows_per_stream, const int32_t *s_per_stream, void *stream);

/* BinaryRansCoder (rans_wrapper.cpp:326-428): prob = P(1)*65536 in [1,65535], uint32 [n_streams, n]. */
/* total = n_streams * n symbols; ranges come out in decode order, stream after stream */
int fpcc_rans_binary_ranges(const uint8_t *symbols, const uint32_t *prob, int64_t total, uint32_t *ranges, void *stream);
/* *err_dev (device int32, caller-zeroed) is set to 1 if any stream ran past its bytes */
int fpcc_rans_binary_decode(const uint8_t *bytes, const int64_t *byte_off, const int32_t *byte_len,
                            const uint32_t *prob, int64_t n, int n_streams, uint8_t *symbols, int32_t *err_dev,
                            void *stream);

/* IndexedRansCoder (rans_wrapper.cpp:89-279): static tables, optional index array, optional
 * overflow (sign + Elias-gamma) escape.  Tables are flat uint32: cdf_flat[cdf_off[t] .. +cdf_len[t]).
 * Encoding is two calls: fpcc_indexed_ranges expands symbols into (range,bits) entries in decode order
 * (entry_off[b] = prefix of per-stream entry counts, computed by the call, workspace-backed), then
 * fpcc_rans_encode.  max_entries_per_symbol = 1 without overflow coding, 66 with. */
int fpcc_indexed_count(const uint32_t *cdf_flat, const int64_t *cdf_off, const int32_t *cdf_len, int n_tables,
                       const int32_t *offsets, int overflow, const int32_t *symbols, const int32_t *indexes,
                       int64_t n, int n_streams, int32_t *entries_per_symbol, void *stream);
int fpcc_indexed_ranges(const uint32_t *cdf_flat, const int64_t *cdf_off, const int32_t *cdf_len, int n_tables,
                        const int32_t *offsets, int overflow, const int32_t *symbols, const int32_t *indexes,
                        int64_t n, int n_streams, const int64_t *entry_pos /* exclusive scan of entries_per_symbol */,
                        uint32_t *ranges, uint8_t *bits, void *stream);
int fpcc_indexed_decode(const uint32_t *cdf_flat, const int64_t *cdf_off, const int32_t *cdf_len, int n_tables,
                        const int32_t *offsets, int overflow, const uint8_t *bytes, const int64_t *byte_off,
                        const int32_t *byte_len, const int32_t *indexes, int64_t n, int n_streams,
                        int32_t *symbols, int32_t *err_dev, void *stream);

/* replaces batched_pmf_to_quantized_cdf (cdf_ops.cpp:4-143): one thread per table, double arithmetic in the
 * reference's evaluation order.  pmf [n_tables,pmf_size] is overwritten by its prefix sums and `offsets` is
 * adjusted in overflow mode (both as in the reference).  cdf_out [n_tables, pmf_size+2]; cdf_len[t] = entries
 * of table t, or -1 when no frequency could be stolen. */
int fpcc_pmf_to_quantized_cdf(double *pmf, int n_tables, int pmf_size, int32_t *offsets, int overflow,
                              uint32_t *cdf_out, int32_t *cdf_len, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Deep-factorized entropy model (csrc/entropy_model.cu; DESIGN 3.10).  params fp32 [C, 43], one row per channel:
 *   H0[3x1] b0[3] a0[3] | H1[3x3] b1[3] a1[3] | H2[3x3] b2[3] a2[3] | H3[1x3] b3[1]    (H row-major [out][in])
 * f_c(x): v = x; per layer v <- softplus(H_i) v + b_i, and for i < 3 v <- v + tanh(a_i) * tanh(v) (monotone in x).
 * L_c(y) = |sigmoid(s u) - sigmoid(s l)|, u = f_c(y + 1/2), l = f_c(y - 1/2), s = -1 if u + l > 0 else +1.
 * bits = -log2(max(L, bound)), 0 < bound < 1.  The gradient at the bound follows compressai's LowerBound: it passes
 * where L >= bound or where it would raise L.  The parity of this definition with the reference is unpinned.
 * ---------------------------------------------------------------------------------------------- */

/* bits fp32 [n, C] (dense) of y fp32 [n, C] with row pitch ld_y >= C */
int fpcc_factorized_bits(const float *y, int64_t ld_y, int64_t n, int C, const float *params, float bound, float *bits,
                         void *stream);
/* dy fp32 [n, C] (dense) and dparams fp32 [C, 43] (with respect to the RAW params, through softplus / tanh) from the
 * upstream dbits [n, C] (row pitch ld_db).  The forward is recomputed; dparams is reduced from fp64 per-CTA partials
 * in a fixed order (no float atomics), so it is reproducible bit for bit.  workspace: fpcc_factorized_grad_workspace
 * bytes. */
size_t fpcc_factorized_grad_workspace(int64_t n, int C);
int fpcc_factorized_grad(const float *y, int64_t ld_y, const float *dbits, int64_t ld_db, int64_t n, int C,
                         const float *params, float bound, float *dy, float *dparams, void *workspace,
                         size_t workspace_bytes, void *stream);
/* pmf fp64 [C, n_sym]: pmf[c, k] = L_c(lo + k), unbounded, by the device function of fpcc_factorized_bits (the input
 * of fpcc_pmf_to_quantized_cdf) */
int fpcc_factorized_pmf(const float *params, int C, int lo, int n_sym, double *pmf, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Gaussian conditional entropy model (csrc/entropy_model.cu; DESIGN 3.11), after compressai's GaussianConditional.
 * All float inputs are fp32 rows [n, C] with a row pitch ld_* >= C (mu and sigma may be the two column halves of
 * one [n, 2C] tensor); mu may be NULL (mean 0).  Per element:
 *   v = |y - mu|, s = max(sigma, scale_bound), u = (1/2 - v) / s, l = (-1/2 - v) / s,
 *   L = Phi(u) - Phi(l), Phi(x) = erfc(-x / sqrt 2) / 2 (erfcf), bits = -log2(max(L, bound)), 0 < bound < 1.
 * Both lower bounds pass gradients as compressai's LowerBound: where the value is at or above the bound, or where the
 * step would raise it.  n == 0 is a no-op.  The parity of this definition with the reference is unpinned.
 * ---------------------------------------------------------------------------------------------- */

/* bits fp32 [n, C] (dense) */
int fpcc_gaussian_bits(const float *y, int64_t ld_y, const float *mu, int64_t ld_mu, const float *sigma, int64_t ld_s,
                       int64_t n, int C, float scale_bound, float bound, float *bits, void *stream);
/* dy, dmu (NULL: not written; needs mu) and dsigma fp32 [n, C] (dense) from the upstream dbits [n, C] (row pitch
 * ld_db); the forward is recomputed in registers.  Elementwise, no reduction: deterministic. */
int fpcc_gaussian_grad(const float *y, int64_t ld_y, const float *mu, int64_t ld_mu, const float *sigma, int64_t ld_s,
                       const float *dbits, int64_t ld_db, int64_t n, int C, float scale_bound, float bound, float *dy,
                       float *dmu, float *dsigma, void *stream);
/* m = -Phi^-1(tail_mass / 2) in double (NaN unless 0 < tail_mass < 1): the half-width factor of the tables */
double fpcc_gaussian_tail_multiplier(double tail_mass);
/* Tables of a strictly increasing, positive scale_table fp32 [T] (compressai's rule): center_t = ceil(scale_table[t] * m)
 * in double, pmf fp64 [T, S] row t = L(k) at mean 0, sigma = scale_table[t] for k = -center_t .. center_t, zero-padded;
 * offsets[t] = -center_t.  S = 2 max(center) + 1 holds every row (a longer row is cut at S).  The input of
 * fpcc_pmf_to_quantized_cdf with overflow coding. */
int fpcc_gaussian_pmf(const float *scale_table, int T, double tail_mass, int S, double *pmf, int32_t *offsets, void *stream);
/* idx int32 [n, C] (dense): the first t with scale_table[t] >= max(sigma, scale_bound), capped at T - 1 (compressai's
 * build_indexes: never a narrower table than the model).  With y (and sym), also sym int32 [n, C] = rint(y - mu)
 * (half to even; |y - mu| < 2^31 is the caller's to ensure).  The decoder passes y = sym = NULL and gets the same idx. */
int fpcc_gaussian_indexes(const float *y, int64_t ld_y, const float *mu, int64_t ld_mu, const float *sigma, int64_t ld_s,
                          int64_t n, int C, float scale_bound, const float *scale_table, int T, int32_t *sym,
                          int32_t *idx, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FASTPCC_B200_H_ */
