// Automatic mask generation: per-candidate mask statistics, bit-packed pairwise IoU and greedy mask NMS.
//
// Candidates are rows of mask logits (one row per prompt x multimask output).  psam_mask_stats_f32 turns a chunk of rows
// into bit-packed masks (bit j of word w = point 32w + j) plus area / stability / filter flag; everything after it works
// on the packed bits, so a candidate costs N/8 bytes instead of 4N and a pairwise intersection is AND + POPC per word.
// Semantics follow SAM's SamAutomaticMaskGenerator (see DESIGN.md, "Automatic mask generation").
#include "psam_common.cuh"
#include "../../include/psam_b200.h"

namespace psam {

constexpr int STATS_THREADS = 512;
constexpr int TILE = 64;          // candidates per side of a pairwise tile
constexpr int TILE_WORDS = 32;    // words of each row staged in shared memory per step
constexpr int TILE_THREADS = 256; // 16 x 16 threads, 4 x 4 pairs each
constexpr int NMS_MAX_K = 16384;
constexpr int SORT_THREADS = 1024;
constexpr int SCAN_THREADS = 1024;

// 8 bits -> bits 0, 4, 8, ..., 28
__device__ __forceinline__ uint32_t spread_nibbles(uint32_t b) {
    b = (b | (b << 12)) & 0x000F000Fu;
    b = (b | (b << 6)) & 0x03030303u;
    b = (b | (b << 3)) & 0x11111111u;
    return b;
}

// One CTA per candidate row.  Vector path (N % 4 == 0): a warp covers 128 points per step with one float4 per lane; the
// four component ballots hold the mask of lanes' points 4l + c, re-interleaved into the 4 words of the step.  Scalar
// path: one float per lane, the ballot is the word.
__global__ void __launch_bounds__(STATS_THREADS) mask_stats_kernel(const float* __restrict__ logits, const float* __restrict__ iou_pred,
                                                                   int N, int W, int vec4, float t, float t_hi, float t_lo,
                                                                   float iou_thresh, float stab_thresh, uint32_t* __restrict__ bits,
                                                                   int* __restrict__ area, float* __restrict__ stability,
                                                                   unsigned char* __restrict__ keep) {
    const int r = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = STATS_THREADS / 32;
    const float* row = logits + (size_t)r * N;
    uint32_t* brow = bits + (size_t)r * W;
    int c_in = 0, c_hi = 0, c_lo = 0;
    if (vec4) {
        const int steps = (N + 127) / 128;
        const float4* row4 = reinterpret_cast<const float4*>(row);
#pragma unroll 4
        for (int s = warp; s < steps; s += nwarps) {
            const int p = s * 128 + lane * 4;
            float4 v = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            if (p < N) v = __ldcs(row4 + (p >> 2));
            const float x[4] = {v.x, v.y, v.z, v.w};
            uint32_t word = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                c_in += x[c] > t;
                c_hi += x[c] > t_hi;
                c_lo += x[c] > t_lo;
                const uint32_t bal = __ballot_sync(0xffffffffu, x[c] > t);  // bit l = point 4l + c of the step
                if (lane < 4) word |= spread_nibbles((bal >> (8 * lane)) & 0xffu) << c;
            }
            const int w = s * 4 + lane;
            if (lane < 4 && w < W) brow[w] = word;
        }
    } else {
        for (int w = warp; w < W; w += nwarps) {
            const int p = w * 32 + lane;
            const float x = p < N ? row[p] : -INFINITY;
            c_in += x > t;
            c_hi += x > t_hi;
            c_lo += x > t_lo;
            const uint32_t bal = __ballot_sync(0xffffffffu, x > t);
            if (lane == 0) brow[w] = bal;
        }
    }
    __shared__ int red[3][STATS_THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c_in += __shfl_xor_sync(0xffffffffu, c_in, o);
        c_hi += __shfl_xor_sync(0xffffffffu, c_hi, o);
        c_lo += __shfl_xor_sync(0xffffffffu, c_lo, o);
    }
    if (lane == 0) {
        red[0][warp] = c_in;
        red[1][warp] = c_hi;
        red[2][warp] = c_lo;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0, hi = 0, lo = 0;
        for (int i = 0; i < nwarps; ++i) {
            a += red[0][i];
            hi += red[1][i];
            lo += red[2][i];
        }
        const float st = lo > 0 ? (float)hi / (float)lo : 0.0f;  // SAM's calculate_stability_score
        area[r] = a;
        stability[r] = st;
        keep[r] = (iou_pred[r] > iou_thresh && st >= stab_thresh && a > 0) ? 1 : 0;
    }
}

// Pairwise tile core: inter[a][b] = sum over words of popc(A_row(ty + 16a) & B_row(tx + 16b)).  Rows are given as pointers
// (NULL = outside the set: contributes zeros).  Words stream through shared memory TILE_WORDS at a time; rows are padded
// by one word so that the 16 rows a warp reads at one word index fall into distinct banks.
struct TileSmem {
    uint32_t a[TILE][TILE_WORDS + 1];
    uint32_t b[TILE][TILE_WORDS + 1];
    const uint32_t* ra[TILE];
    const uint32_t* rb[TILE];
};

__device__ __forceinline__ void tile_intersections(TileSmem& sm, int W, int (&inter)[4][4]) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) inter[i][j] = 0;
    for (int w0 = 0; w0 < W; w0 += TILE_WORDS) {
        __syncthreads();
        for (int e = threadIdx.x; e < TILE * TILE_WORDS; e += TILE_THREADS) {
            const int row = e / TILE_WORDS, k = e % TILE_WORDS;
            const int w = w0 + k;
            const uint32_t* pa = sm.ra[row];
            const uint32_t* pb = sm.rb[row];
            sm.a[row][k] = (pa && w < W) ? __ldg(pa + w) : 0u;
            sm.b[row][k] = (pb && w < W) ? __ldg(pb + w) : 0u;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < TILE_WORDS; ++k) {
            uint32_t va[4], vb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) va[i] = sm.a[ty + 16 * i][k];
#pragma unroll
            for (int j = 0; j < 4; ++j) vb[j] = sm.b[tx + 16 * j][k];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) inter[i][j] += __popc(va[i] & vb[j]);
        }
    }
}

__device__ __forceinline__ float iou_of(int inter, int area_a, int area_b) {
    const int uni = area_a + area_b - inter;
    return uni > 0 ? (float)inter / (float)uni : 0.0f;
}

// IoU matrix of two bit-mask sets.  Each CTA counts the areas of its own 64 + 64 rows before the tile loop.
__global__ void __launch_bounds__(TILE_THREADS) mask_iou_kernel(const uint32_t* __restrict__ a_bits, int Ka, const uint32_t* __restrict__ b_bits,
                                                                int Kb, int W, float* __restrict__ iou, int* __restrict__ inter_out) {
    __shared__ TileSmem sm;
    __shared__ int area_a[TILE], area_b[TILE];
    const int i0 = blockIdx.y * TILE, j0 = blockIdx.x * TILE;
    if (threadIdx.x < TILE) {
        const int i = i0 + threadIdx.x, j = j0 + threadIdx.x;
        sm.ra[threadIdx.x] = i < Ka ? a_bits + (size_t)i * W : nullptr;
        sm.rb[threadIdx.x] = j < Kb ? b_bits + (size_t)j * W : nullptr;
        int ca = 0, cb = 0;
        if (i < Ka)
            for (int w = 0; w < W; ++w) ca += __popc(a_bits[(size_t)i * W + w]);
        if (j < Kb)
            for (int w = 0; w < W; ++w) cb += __popc(b_bits[(size_t)j * W + w]);
        area_a[threadIdx.x] = ca;
        area_b[threadIdx.x] = cb;
    }
    int inter[4][4];
    tile_intersections(sm, W, inter);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
        const int i = i0 + ty + 16 * ii;
        if (i >= Ka) continue;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            const int j = j0 + tx + 16 * jj;
            if (j >= Kb) continue;
            const int x = inter[ii][jj];
            iou[(size_t)i * Kb + j] = iou_of(x, area_a[ty + 16 * ii], area_b[tx + 16 * jj]);
            if (inter_out) inter_out[(size_t)i * Kb + j] = x;
        }
    }
}

// Single CTA: stable descending sort of the candidates that passed the filter (key = ordered score bits, then the
// complement of the index so that ties go to the lower index), as a bitonic sort over a power-of-two shared array.
// Writes order[0..M) and *M.
__global__ void __launch_bounds__(SORT_THREADS) mask_sort_kernel(const float* __restrict__ score, const unsigned char* __restrict__ keep,
                                                                 int K, int Kp, int* __restrict__ order, int* __restrict__ count) {
    extern __shared__ unsigned long long keys[];
    __shared__ int n_pass;
    if (threadIdx.x == 0) n_pass = 0;
    __syncthreads();
    int local = 0;
    for (int i = threadIdx.x; i < Kp; i += SORT_THREADS) {
        unsigned long long key = 0ull;
        if (i < K && keep[i]) {
            uint32_t u = __float_as_uint(score[i] + 0.0f);  // -0 -> +0: equal scores compare equal
            u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
            key = ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
            ++local;
        }
        keys[i] = key;
    }
    atomicAdd(&n_pass, local);
    for (int size = 2; size <= Kp; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < Kp / 2; t += SORT_THREADS) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool desc = (lo & size) == 0;  // descending runs first: the whole array ends descending
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a < b) == desc) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
        }
    }
    __syncthreads();
    const int M = n_pass;
    for (int i = threadIdx.x; i < M; i += SORT_THREADS) order[i] = (int)(0xFFFFFFFFu - (uint32_t)(keys[i] & 0xFFFFFFFFull));
    if (threadIdx.x == 0) *count = M;
}

// Suppression bits of the upper triangle: sup[p][q / 64] bit (q % 64) = IoU(order[p], order[q]) > thresh, for q > p
// (positions in score order).  One CTA per 64 x 64 tile (tb >= ta); the grid covers K, tiles past the device-side
// count M exit before loading anything.
__global__ void __launch_bounds__(TILE_THREADS) mask_suppress_kernel(const uint32_t* __restrict__ bits, const int* __restrict__ area, int W,
                                                                     const int* __restrict__ order, const int* __restrict__ count, int T,
                                                                     float thresh, unsigned long long* __restrict__ sup) {
    __shared__ union {
        TileSmem t;
        int inter[TILE][TILE + 1];  // the tile's intersections, restaged for the divisions
    } sm;
    __shared__ int area_a[TILE], area_b[TILE];
    // tile index -> (ta, tb), tb >= ta, row-major over the upper triangle
    int t = blockIdx.x, ta = 0;
    while (t >= T - ta) {
        t -= T - ta;
        ++ta;
    }
    const int tb = ta + t;
    const int M = *count;
    if (tb * TILE >= M) return;  // ta <= tb
    if (threadIdx.x < TILE) {
        const int p = ta * TILE + threadIdx.x, q = tb * TILE + threadIdx.x;
        const int ci = p < M ? order[p] : -1, cj = q < M ? order[q] : -1;
        sm.t.ra[threadIdx.x] = ci >= 0 ? bits + (size_t)ci * W : nullptr;
        sm.t.rb[threadIdx.x] = cj >= 0 ? bits + (size_t)cj * W : nullptr;
        area_a[threadIdx.x] = ci >= 0 ? area[ci] : 0;
        area_b[threadIdx.x] = cj >= 0 ? area[cj] : 0;
    }
    int inter[4][4];
    tile_intersections(sm.t, W, inter);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    __syncthreads();
#pragma unroll
    for (int ii = 0; ii < 4; ++ii)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) sm.inter[ty + 16 * ii][tx + 16 * jj] = inter[ii][jj];
    __syncthreads();
    // 4 threads per row, 16 columns each; the row word is OR-combined across the 4 lanes
    const int pr = threadIdx.x >> 2, part = threadIdx.x & 3;
    const int p = ta * TILE + pr;
    unsigned long long m = 0ull;
    for (int c = part * 16; c < part * 16 + 16; ++c) {
        const int q = tb * TILE + c;
        if (p < M && q < M && q > p && iou_of(sm.inter[pr][c], area_a[pr], area_b[c]) > thresh) m |= 1ull << c;
    }
    m |= __shfl_xor_sync(0xffffffffu, m, 1);
    m |= __shfl_xor_sync(0xffffffffu, m, 2);
    if (part == 0 && p < M) sup[(size_t)p * T + tb] = m;
}

// Single CTA greedy scan, 64 rows per round: thread 0 resolves the round's rows in order from the diagonal block (a row
// is kept unless an earlier kept row of the round or of an earlier round suppressed it), then all threads OR the kept
// rows' suppression words into the pending masks of the later blocks.
__global__ void __launch_bounds__(SCAN_THREADS) mask_scan_kernel(const unsigned long long* __restrict__ sup, const int* __restrict__ order,
                                                                 const int* __restrict__ count, int K, int T, int* __restrict__ keep_idx,
                                                                 int* __restrict__ kept_count) {
    extern __shared__ unsigned long long removed[];  // [T]
    __shared__ unsigned long long kept_bits;
    __shared__ int n_kept;
    const int M = *count;
    const int TM = (M + TILE - 1) / TILE;
    for (int b = threadIdx.x; b < T; b += SCAN_THREADS) removed[b] = 0ull;
    if (threadIdx.x == 0) n_kept = 0;
    __syncthreads();
    for (int b = 0; b < TM; ++b) {
        if (threadIdx.x == 0) {
            const int rows = min(TILE, M - b * TILE);
            unsigned long long cur = removed[b], kept = 0ull;
            int n = n_kept;
            for (int r = 0; r < rows; ++r) {
                if ((cur >> r) & 1ull) continue;
                kept |= 1ull << r;
                cur |= sup[(size_t)(b * TILE + r) * T + b];
                keep_idx[n++] = order[b * TILE + r];
            }
            kept_bits = kept;
            n_kept = n;
        }
        __syncthreads();
        const unsigned long long kept = kept_bits;
        const int nc = TM - b - 1;
        if (kept && nc > 0) {
            for (int e = threadIdx.x; e < TILE * nc; e += SCAN_THREADS) {
                const int r = e / nc, c = b + 1 + e % nc;
                if ((kept >> r) & 1ull) {
                    const unsigned long long v = sup[(size_t)(b * TILE + r) * T + c];
                    if (v) atomicOr(&removed[c], v);
                }
            }
        }
        __syncthreads();
    }
    const int n = n_kept;
    for (int i = n + threadIdx.x; i < K; i += SCAN_THREADS) keep_idx[i] = -1;
    if (threadIdx.x == 0) *kept_count = n;
}

__global__ void mask_unpack_kernel(const uint32_t* __restrict__ bits, int W, const int* __restrict__ rows, int N,
                                   unsigned char* __restrict__ out) {
    const int k = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    const int r = rows ? rows[k] : k;
    out[(size_t)k * N + p] = (bits[(size_t)r * W + (p >> 5)] >> (p & 31)) & 1u;
}

}  // namespace psam

using namespace psam;

extern "C" int psam_mask_stats_f32(const float* logits, const float* iou_pred, int R, int N, float mask_threshold,
                                   float stability_offset, float pred_iou_thresh, float stability_thresh, unsigned int* bits,
                                   int* area, float* stability, unsigned char* keep, cudaStream_t stream) {
    if (!logits || !iou_pred || !bits || !area || !stability || !keep || R <= 0 || N <= 0) return PSAM_ERR_ARG;
    const int W = ceil_div(N, 32);
    const int vec4 = (N & 3) == 0 && ((uintptr_t)logits & 15) == 0;
    const float t_hi = mask_threshold + stability_offset, t_lo = mask_threshold - stability_offset;
    mask_stats_kernel<<<R, STATS_THREADS, 0, stream>>>(logits, iou_pred, N, W, vec4, mask_threshold, t_hi, t_lo, pred_iou_thresh,
                                                       stability_thresh, bits, area, stability, keep);
    PSAM_LAUNCH_CHECK();
    return PSAM_OK;
}

extern "C" int psam_mask_iou_u32(const unsigned int* a_bits, int Ka, const unsigned int* b_bits, int Kb, int W, float* iou,
                                 int* inter, cudaStream_t stream) {
    if (!a_bits || !b_bits || !iou || Ka <= 0 || Kb <= 0 || W <= 0) return PSAM_ERR_ARG;
    if (ceil_div(Ka, TILE) > 65535) return PSAM_ERR_UNSUPPORTED;
    mask_iou_kernel<<<dim3(ceil_div(Kb, TILE), ceil_div(Ka, TILE)), TILE_THREADS, 0, stream>>>(a_bits, Ka, b_bits, Kb, W, iou, inter);
    PSAM_LAUNCH_CHECK();
    return PSAM_OK;
}

static int nms_pow2(int K) {
    int p = 1;
    while (p < K) p <<= 1;
    return p < 2 ? 2 : p;
}

extern "C" size_t psam_mask_nms_workspace_bytes(int K, int W) {
    if (K <= 0 || W <= 0) return 0;
    const size_t T = (size_t)ceil_div(K, TILE);
    return 16 + (size_t)(K + 3) / 4 * 16 + (size_t)K * T * 8;  // count, order (16-byte padded), suppression bits
}

extern "C" int psam_mask_nms(const unsigned int* bits, const int* area, const float* score, const unsigned char* keep, int K, int W,
                             float nms_thresh, int* keep_idx, int* kept_count, void* workspace, cudaStream_t stream) {
    if (!bits || !area || !score || !keep || !keep_idx || !kept_count || !workspace || K <= 0 || W <= 0 ||
        ((uintptr_t)workspace & 15) != 0)
        return PSAM_ERR_ARG;
    if (K > NMS_MAX_K) return PSAM_ERR_UNSUPPORTED;
    const int T = ceil_div(K, TILE);
    char* ws = static_cast<char*>(workspace);
    int* count = reinterpret_cast<int*>(ws);
    int* order = reinterpret_cast<int*>(ws + 16);
    unsigned long long* sup = reinterpret_cast<unsigned long long*>(ws + 16 + (size_t)(K + 3) / 4 * 16);
    const int Kp = nms_pow2(K);
    const size_t sort_smem = (size_t)Kp * 8;
    if (sort_smem > 48 * 1024) PSAM_CUDA_TRY(cudaFuncSetAttribute(mask_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
    mask_sort_kernel<<<1, SORT_THREADS, sort_smem, stream>>>(score, keep, K, Kp, order, count);
    PSAM_LAUNCH_CHECK();
    mask_suppress_kernel<<<T * (T + 1) / 2, TILE_THREADS, 0, stream>>>(bits, area, W, order, count, T, nms_thresh, sup);
    PSAM_LAUNCH_CHECK();
    mask_scan_kernel<<<1, SCAN_THREADS, (size_t)T * 8, stream>>>(sup, order, count, K, T, keep_idx, kept_count);
    PSAM_LAUNCH_CHECK();
    return PSAM_OK;
}

extern "C" int psam_mask_unpack_u8(const unsigned int* bits, int W, const int* rows, int k, int N, unsigned char* out,
                                   cudaStream_t stream) {
    if (!bits || !out || k <= 0 || N <= 0 || W < ceil_div(N, 32)) return PSAM_ERR_ARG;
    if (k > 65535) return PSAM_ERR_UNSUPPORTED;
    mask_unpack_kernel<<<dim3(ceil_div(N, 256), k), 256, 0, stream>>>(bits, W, rows, N, out);
    PSAM_LAUNCH_CHECK();
    return PSAM_OK;
}
