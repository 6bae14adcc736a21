// Rotated BEV IoU, rotated NMS and the rescoring tail.
//
// Replaces iou3d_cuda.nms_gpu (mmdet/ops/iou3d/src/iou3d.cpp:73-120 +
// iou3d_kernel.cu:250-292) and the Python around it
// (ssd_rotate_head.py:487-533, iou3d_utils.py:47-60,114-128, bbox_nms.py:4-27).
//
// Differences in structure, not in arithmetic:
//  * only the tiles on/above the diagonal are evaluated (the reference computes
//    and discards the lower triangle, iou3d_kernel.cu:258);
//  * the greedy sweep runs on the device in one CTA per frame, 64 boxes at a
//    time (diagonal tile resolved from registers, the kept rows OR-ed into the
//    remaining columns in parallel) — no cudaMalloc/cudaFree, no blocking D2H
//    copy of the bitmask, no host loop (iou3d.cpp:87-116);
//  * score threshold, stable sort and BEV conversion are fused in front of it.
// The IoU itself is evaluated expression-for-expression like the reference's
// box_overlap/iou_bev (same fp32 operation order, same libm calls, same
// contraction opportunities) because the keep mask must match bit for bit.
#include "common.cuh"

namespace {

constexpr float kEps = 1e-8f;

struct P2 { float x, y; };

__device__ __forceinline__ float cross_o(const P2& p1, const P2& p2, const P2& p0) {
    return (p1.x - p0.x) * (p2.y - p0.y) - (p2.x - p0.x) * (p1.y - p0.y);
}

__device__ __forceinline__ float cross_v(const P2& a, const P2& b) { return a.x * b.y - a.y * b.x; }

__device__ __forceinline__ bool spans_overlap(const P2& p1, const P2& p2, const P2& q1, const P2& q2) {
    return fminf(p1.x, p2.x) <= fmaxf(q1.x, q2.x) && fminf(q1.x, q2.x) <= fmaxf(p1.x, p2.x) &&
           fminf(p1.y, p2.y) <= fmaxf(q1.y, q2.y) && fminf(q1.y, q2.y) <= fmaxf(p1.y, p2.y);
}

// is p inside the rotated rectangle `box` = (x1,y1,x2,y2,angle), margin 1e-5
__device__ __forceinline__ bool point_in_box(const float* box, const P2& p) {
    const float MARGIN = 1e-5f;
    float center_x = (box[0] + box[2]) / 2;
    float center_y = (box[1] + box[3]) / 2;
    float angle_cos = cosf(-box[4]), angle_sin = sinf(-box[4]);
    float rot_x = (p.x - center_x) * angle_cos + (p.y - center_y) * angle_sin + center_x;
    float rot_y = -(p.x - center_x) * angle_sin + (p.y - center_y) * angle_cos + center_y;
    return (rot_x > box[0] - MARGIN && rot_x < box[2] + MARGIN && rot_y > box[1] - MARGIN && rot_y < box[3] + MARGIN);
}

__device__ __forceinline__ bool edge_hit(const P2& p1, const P2& p0, const P2& q1, const P2& q0, P2& ans) {
    if (!spans_overlap(p0, p1, q0, q1)) return false;
    float s1 = cross_o(q0, p1, p0);
    float s2 = cross_o(p1, q1, p0);
    float s3 = cross_o(p0, q1, q0);
    float s4 = cross_o(q1, p1, q0);
    if (!(s1 * s2 > 0 && s3 * s4 > 0)) return false;
    float s5 = cross_o(q1, p1, p0);
    if (fabsf(s5 - s1) > kEps) {
        ans.x = (s5 * q0.x - s1 * q1.x) / (s5 - s1);
        ans.y = (s5 * q0.y - s1 * q1.y) / (s5 - s1);
    } else {
        float a0 = p0.y - p1.y, b0 = p1.x - p0.x, c0 = p0.x * p1.y - p1.x * p0.y;
        float a1 = q0.y - q1.y, b1 = q1.x - q0.x, c1 = q0.x * q1.y - q1.x * q0.y;
        float D = a0 * b1 - a1 * b0;
        ans.x = (b0 * c1 - b1 * c0) / D;
        ans.y = (a1 * c0 - a0 * c1) / D;
    }
    return true;
}

__device__ __forceinline__ void spin(const P2& center, float angle_cos, float angle_sin, P2& p) {
    float new_x = (p.x - center.x) * angle_cos + (p.y - center.y) * angle_sin + center.x;
    float new_y = -(p.x - center.x) * angle_sin + (p.y - center.y) * angle_cos + center.y;
    p.x = new_x;
    p.y = new_y;
}

__device__ float rotated_overlap(const float* box_a, const float* box_b) {
    float a_x1 = box_a[0], a_y1 = box_a[1], a_x2 = box_a[2], a_y2 = box_a[3], a_angle = box_a[4];
    float b_x1 = box_b[0], b_y1 = box_b[1], b_x2 = box_b[2], b_y2 = box_b[3], b_angle = box_b[4];
    P2 center_a{(a_x1 + a_x2) / 2, (a_y1 + a_y2) / 2};
    P2 center_b{(b_x1 + b_x2) / 2, (b_y1 + b_y2) / 2};
    P2 ca[5] = {{a_x1, a_y1}, {a_x2, a_y1}, {a_x2, a_y2}, {a_x1, a_y2}, {0.f, 0.f}};
    P2 cb[5] = {{b_x1, b_y1}, {b_x2, b_y1}, {b_x2, b_y2}, {b_x1, b_y2}, {0.f, 0.f}};
    float a_angle_cos = cosf(a_angle), a_angle_sin = sinf(a_angle);
    float b_angle_cos = cosf(b_angle), b_angle_sin = sinf(b_angle);
    for (int k = 0; k < 4; k++) {
        spin(center_a, a_angle_cos, a_angle_sin, ca[k]);
        spin(center_b, b_angle_cos, b_angle_sin, cb[k]);
    }
    ca[4] = ca[0];
    cb[4] = cb[0];

    P2 poly[16];
    P2 pc{0.f, 0.f};
    int cnt = 0;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++)
            if (edge_hit(ca[i + 1], ca[i], cb[j + 1], cb[j], poly[cnt])) {
                pc.x = pc.x + poly[cnt].x;
                pc.y = pc.y + poly[cnt].y;
                cnt++;
            }
    for (int k = 0; k < 4; k++) {
        if (point_in_box(box_a, cb[k])) {
            pc.x = pc.x + cb[k].x;
            pc.y = pc.y + cb[k].y;
            poly[cnt] = cb[k];
            cnt++;
        }
        if (point_in_box(box_b, ca[k])) {
            pc.x = pc.x + ca[k].x;
            pc.y = pc.y + ca[k].y;
            poly[cnt] = ca[k];
            cnt++;
        }
    }
    pc.x /= cnt;
    pc.y /= cnt;
    // bubble sort by polar angle about the centroid (same comparison sequence as the reference,
    // so ties and near-ties order identically)
    for (int j = 0; j < cnt - 1; j++)
        for (int i = 0; i < cnt - j - 1; i++)
            if (atan2f(poly[i].y - pc.y, poly[i].x - pc.x) > atan2f(poly[i + 1].y - pc.y, poly[i + 1].x - pc.x)) {
                P2 t = poly[i];
                poly[i] = poly[i + 1];
                poly[i + 1] = t;
            }
    float area = 0;
    for (int k = 0; k < cnt - 1; k++) {
        P2 u{poly[k].x - poly[0].x, poly[k].y - poly[0].y};
        P2 v{poly[k + 1].x - poly[0].x, poly[k + 1].y - poly[0].y};
        area += cross_v(u, v);
    }
    return fabsf(area) / 2.0f;
}

__device__ __forceinline__ float rotated_iou(const float* box_a, const float* box_b) {
    float sa = (box_a[2] - box_a[0]) * (box_a[3] - box_a[1]);
    float sb = (box_b[2] - box_b[0]) * (box_b[3] - box_b[1]);
    float s_overlap = rotated_overlap(box_a, box_b);
    return s_overlap / fmaxf(sa + sb - s_overlap, kEps);
}

// mask[(frame*n_cap + i) * colb_cap + cb] bit j <=> iou(i, cb*64+j) > thr ; tiles with cb >= rb only.
// The grid is fixed (CUDA-graph friendly); each CTA walks the frame's live upper-triangle work items, whose number
// depends on the device-side candidate count.  A work item is a QUARTER of a 64x64 tile - 64 rows x 16 columns, one
// pair per thread: the guided anchors of an object overlap each other heavily, so many pairs take the slow rotated
// polygon-clipping path, and with four pairs per thread (round 1) a frame's handful of tiles kept six SMs busy for
// ~40 us (profiles/r2_ncu_small_kernels.md).  Each item writes its own 16-bit quarter of the 64-bit mask words.
#define NMS_MASK_THREADS 1024   // 64 rows x 16 columns
__global__ void __launch_bounds__(NMS_MASK_THREADS)
nms_mask_kernel(const float* __restrict__ boxes5, const int* __restrict__ d_n, int n_fixed, int n_cap, int colb_cap,
                float thr, unsigned long long* __restrict__ mask) {
    const int f = blockIdx.y;
    const int n = d_n ? min(d_n[f], n_cap) : n_fixed;
    const int colb = (n + 63) / 64;
    const int nitems = 4 * (colb * (colb + 1) / 2);
    const float* bx = boxes5 + (size_t)f * n_cap * 5;
    __shared__ float s_col[16 * 5];
    __shared__ unsigned int s_bits[64];
    const int r = threadIdx.x & 63, g = threadIdx.x >> 6;   // row in tile, column within the quarter
    for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
        const int t = it >> 2, q = it & 3;
        int rb = 0, rem = t;
        while (rem >= colb - rb) { rem -= colb - rb; ++rb; }
        const int cb = rb + rem;
        const int row_size = min(n - rb * 64, 64), col_size = min(n - cb * 64, 64);
        if (threadIdx.x < 16 && q * 16 + (int)threadIdx.x < col_size) {
#pragma unroll
            for (int e = 0; e < 5; ++e) s_col[threadIdx.x * 5 + e] = bx[(size_t)(cb * 64 + q * 16 + threadIdx.x) * 5 + e];
        }
        if (threadIdx.x < 64) s_bits[threadIdx.x] = 0u;
        __syncthreads();
        const int j = q * 16 + g;                            // column of the tile
        if (r < row_size && j < col_size && !(rb == cb && j <= r)) {
            const int i = rb * 64 + r;
            float cur[5];
#pragma unroll
            for (int e = 0; e < 5; ++e) cur[e] = bx[(size_t)i * 5 + e];
            // Boxes whose circumscribed circles are apart cannot intersect: the reference's overlap is exactly 0
            // there and 0 > thr is false, so skipping them leaves the mask bit-identical (thr >= 0; the 1e-3 margin
            // keeps every touching pair on the exact path).  Most pairs go this way.
            const float* o = s_col + g * 5;
            bool far = false;
            if (thr >= 0.f) {
                const float cx = 0.5f * (cur[0] + cur[2]), cy = 0.5f * (cur[1] + cur[3]);
                const float rad = 0.5f * sqrtf((cur[2] - cur[0]) * (cur[2] - cur[0]) + (cur[3] - cur[1]) * (cur[3] - cur[1]));
                const float dx = 0.5f * (o[0] + o[2]) - cx, dy = 0.5f * (o[1] + o[3]) - cy;
                const float reach = rad + 0.5f * sqrtf((o[2] - o[0]) * (o[2] - o[0]) + (o[3] - o[1]) * (o[3] - o[1]));
                far = dx * dx + dy * dy > reach * reach * 1.002f + 1e-6f;
            }
            if (!far && rotated_iou(cur, o) > thr) atomicOr(&s_bits[r], 1u << g);
        }
        __syncthreads();
        if (threadIdx.x < row_size)      // my 16-bit quarter of the (row, cb) word (little endian: half-word q)
            ((unsigned short*)mask)[(((size_t)f * n_cap + rb * 64 + threadIdx.x) * colb_cap + cb) * 4 + q] =
                (unsigned short)s_bits[threadIdx.x];
        __syncthreads();
    }
}

// Greedy sweep, one CTA (256 threads) per frame.  keep_flag[i] = 1 if box i survives.
// Processes 64 boxes per step: thread 0 resolves the diagonal tile serially from shared
// memory, then all threads OR the kept rows into the removal words of the later columns.
__device__ void nms_sweep(const unsigned long long* __restrict__ mask, int n, int colb_cap,
                          unsigned long long* s_remv /*[colb]*/, unsigned long long* s_diag /*[64]*/,
                          unsigned long long* s_keepw /*[1]*/, unsigned long long* keep_words /*[colb] out (shared)*/) {
    const int colb = (n + 63) / 64;
    for (int c = threadIdx.x; c < colb; c += blockDim.x) { s_remv[c] = 0ULL; keep_words[c] = 0ULL; }
    __syncthreads();
    for (int blk = 0; blk < colb; ++blk) {
        const int rows = min(n - blk * 64, 64);
        if (threadIdx.x < 64)
            s_diag[threadIdx.x] = threadIdx.x < rows ? mask[(size_t)(blk * 64 + threadIdx.x) * colb_cap + blk] : 0ULL;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long removed = s_remv[blk], kept = 0ULL;
            for (int j = 0; j < rows; ++j)
                if (!((removed >> j) & 1ULL)) { kept |= 1ULL << j; removed |= s_diag[j]; }
            *s_keepw = kept;
            keep_words[blk] = kept;
        }
        __syncthreads();
        const unsigned long long kept = *s_keepw;
        for (int c = blk + 1 + threadIdx.x; c < colb; c += blockDim.x) {
            unsigned long long acc = s_remv[c];
            unsigned long long kk = kept;
            while (kk) {
                const int j = __ffsll((long long)kk) - 1;
                kk &= kk - 1;
                acc |= mask[(size_t)(blk * 64 + j) * colb_cap + c];
            }
            s_remv[c] = acc;
        }
        __syncthreads();
    }
}

#define RS_THREADS 1024

// Per frame: sigmoid(score) > thr, ordered compaction, stable sort by score (descending),
// BEV boxes.  Bitonic sort on (score, candidate position) in shared memory.
template <int CAP>
__global__ void __launch_bounds__(RS_THREADS)
rescore_sort_kernel(const float* __restrict__ boxes7, const float* __restrict__ scores, const int* __restrict__ d_k,
                    int k_cap, float score_thr, float* __restrict__ boxes5, float* __restrict__ s_sorted,
                    int* __restrict__ src_sorted, int* __restrict__ d_n, int* __restrict__ status) {
    __shared__ float s_key[CAP];
    __shared__ int s_idx[CAP];
    __shared__ int s_scan[33];
    const int f = blockIdx.x;
    const int k = min(d_k[f], k_cap);
    int base = 0;
    for (int i0 = 0; i0 < k; i0 += RS_THREADS) {
        const int i = i0 + threadIdx.x;
        float s = 0.f;
        bool pass = false;
        if (i < k) {
            const float x = scores[(size_t)f * k_cap + i];
            s = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-x)));
            pass = s > score_thr;
        }
        int total;
        const int pos = base + sassd_block_exscan(pass ? 1 : 0, s_scan, &total);
        if (pass && pos < CAP) { s_key[pos] = s; s_idx[pos] = i; }
        base += total;
    }
    int n = base;
    if (n > CAP) { if (threadIdx.x == 0) atomicOr(status, SASSD_FLAG_NMS_CAP); n = CAP; }
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (int i = n + threadIdx.x; i < np2; i += RS_THREADS) { s_key[i] = -1.f; s_idx[i] = 0x7fffffff; }
    __syncthreads();
    // order: higher score first; equal scores keep candidate order (s_idx ascending) => stable
    for (int size = 2; size <= np2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < np2 / 2; t += RS_THREADS) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const float ka = s_key[lo], kb = s_key[hi];
                const int ia = s_idx[lo], ib = s_idx[hi];
                const bool a_first = (ka > kb) || (ka == kb && ia < ib);  // a should precede b
                if (a_first != up) { s_key[lo] = kb; s_key[hi] = ka; s_idx[lo] = ib; s_idx[hi] = ia; }
            }
            __syncthreads();
        }
    for (int r = threadIdx.x; r < n; r += RS_THREADS) {
        const int src = s_idx[r];
        const float* b7 = boxes7 + ((size_t)f * k_cap + src) * 7;
        float* b5 = boxes5 + ((size_t)f * CAP + r) * 5;
        // boxes3d_to_bev_torch (iou3d_utils.py:55-59): half extents come from columns 3 and 4
        const float cu = b7[0], cv = b7[1], hl = __fdiv_rn(b7[3], 2.f), hw = __fdiv_rn(b7[4], 2.f);
        b5[0] = __fsub_rn(cu, hl); b5[1] = __fsub_rn(cv, hw);
        b5[2] = __fadd_rn(cu, hl); b5[3] = __fadd_rn(cv, hw);
        b5[4] = b7[6];
        s_sorted[(size_t)f * CAP + r] = s_key[r];
        src_sorted[(size_t)f * CAP + r] = src;
    }
    if (threadIdx.x == 0) d_n[f] = n;
}

template <int CAP>
__global__ void __launch_bounds__(256)
nms_gather_kernel(const unsigned long long* __restrict__ mask, const int* __restrict__ d_n,
                  const float* __restrict__ boxes7, const int* __restrict__ labels, int k_cap,
                  const float* __restrict__ s_sorted, const int* __restrict__ src_sorted, float* __restrict__ det,
                  int* __restrict__ d_ndet, int det_cap, int* __restrict__ status) {
    constexpr int COLB = CAP / 64;
    __shared__ unsigned long long s_remv[COLB], s_keep[COLB], s_diag[64], s_keepw;
    __shared__ int s_pref[COLB + 1];
    const int f = blockIdx.x;
    const int n = min(d_n[f], CAP);
    nms_sweep(mask + (size_t)f * CAP * COLB, n, COLB, s_remv, s_diag, &s_keepw, s_keep);
    const int colb = (n + 63) / 64;
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int c = 0; c < colb; ++c) { s_pref[c] = acc; acc += __popcll(s_keep[c]); }
        s_pref[colb] = acc;
        d_ndet[f] = acc < det_cap ? acc : det_cap;
        // the reference applies no per-image maximum (get_rescore_bboxes ignores max_per_img): dropping kept boxes
        // must not pass silently
        if (acc > det_cap) atomicOr(status, SASSD_FLAG_DET_CAP);
    }
    __syncthreads();
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        const unsigned long long w = s_keep[r >> 6];
        if (!((w >> (r & 63)) & 1ULL)) continue;
        const int pos = s_pref[r >> 6] + __popcll(w & ((1ULL << (r & 63)) - 1ULL));
        if (pos >= det_cap) continue;
        const int src = src_sorted[(size_t)f * CAP + r];
        const float* b7 = boxes7 + ((size_t)f * k_cap + src) * 7;
        float* o = det + ((size_t)f * det_cap + pos) * 9;
#pragma unroll
        for (int e = 0; e < 7; ++e) o[e] = b7[e];
        o[7] = s_sorted[(size_t)f * CAP + r];
        o[8] = (float)labels[(size_t)f * k_cap + src];
    }
}

__global__ void __launch_bounds__(256)
nms_keep_kernel(const unsigned long long* __restrict__ mask, int n, int colb, long long* __restrict__ keep,
                int* __restrict__ d_nkeep) {
    extern __shared__ unsigned long long s_dyn[];
    unsigned long long* s_remv = s_dyn;
    unsigned long long* s_keep = s_dyn + colb;
    __shared__ unsigned long long s_diag[64], s_keepw;
    nms_sweep(mask, n, colb, s_remv, s_diag, &s_keepw, s_keep);
    __shared__ int s_total;
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int c = 0; c < colb; ++c) {
            unsigned long long w = s_keep[c];
            while (w) {
                const int j = __ffsll((long long)w) - 1;
                w &= w - 1;
                keep[acc++] = (long long)c * 64 + j;
            }
        }
        s_total = acc;
        *d_nkeep = acc;
    }
}

__global__ void iou_matrix_kernel(const float* __restrict__ a, int na, const float* __restrict__ b, int nb,
                                  float* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= na || j >= nb) return;
    float ba[5], bb[5];
#pragma unroll
    for (int e = 0; e < 5; ++e) { ba[e] = a[(size_t)i * 5 + e]; bb[e] = b[(size_t)j * 5 + e]; }
    out[(size_t)i * nb + j] = rotated_iou(ba, bb);
}

constexpr int kNmsCap = 4096;
inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

extern "C" size_t sassd_rescore_nms_workspace_bytes(int batch, int k_cap, int nms_cap) {
    (void)k_cap;
    const size_t colb = (size_t)nms_cap / 64;
    return al256((size_t)batch * nms_cap * 5 * 4) + 2 * al256((size_t)batch * nms_cap * 4) +
           al256((size_t)batch * 4) + al256((size_t)batch * nms_cap * colb * 8);
}

extern "C" int sassd_rescore_nms(const float* boxes, const float* scores, const int32_t* labels, const int32_t* d_k,
                                 int batch, int k_cap, float score_thr, float iou_thr, int nms_cap, float* det,
                                 int32_t* d_ndet, int det_cap, int32_t* d_status, void* ws, size_t ws_bytes,
                                 sassd_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!boxes || !scores || !labels || !d_k || !det || !d_ndet || !d_status || !ws) return SASSD_ERR_ARG;
    if (nms_cap != kNmsCap) return SASSD_ERR_UNSUPPORTED;
    if (batch < 1 || k_cap < 1 || det_cap < 1) return SASSD_ERR_ARG;
    if (ws_bytes < sassd_rescore_nms_workspace_bytes(batch, k_cap, nms_cap)) return SASSD_ERR_WORKSPACE;
    constexpr int COLB = kNmsCap / 64;
    char* w = (char*)ws;
    float* boxes5 = (float*)w; w += al256((size_t)batch * kNmsCap * 5 * 4);
    float* s_sorted = (float*)w; w += al256((size_t)batch * kNmsCap * 4);
    int* src_sorted = (int*)w; w += al256((size_t)batch * kNmsCap * 4);
    int* d_n = (int*)w; w += al256((size_t)batch * 4);
    unsigned long long* mask = (unsigned long long*)w;
    rescore_sort_kernel<kNmsCap><<<batch, RS_THREADS, 0, stream>>>(boxes, scores, d_k, k_cap, score_thr, boxes5,
                                                                   s_sorted, src_sorted, d_n, d_status);
    dim3 grid(128, batch);
    nms_mask_kernel<<<grid, NMS_MASK_THREADS, 0, stream>>>(boxes5, d_n, 0, kNmsCap, COLB, iou_thr, mask);
    nms_gather_kernel<kNmsCap><<<batch, 256, 0, stream>>>(mask, d_n, boxes, labels, k_cap, s_sorted, src_sorted, det,
                                                          d_ndet, det_cap, d_status);
    return sassd_check_launch();
}

extern "C" size_t sassd_nms_workspace_bytes(int n) {
    const size_t colb = ((size_t)n + 63) / 64;
    return al256((size_t)(n > 0 ? n : 1) * colb * 8);
}

extern "C" int sassd_nms_mask(const float* boxes5, int n, float thr, uint64_t* mask, sassd_stream_t stream_) {
    if (!boxes5 || !mask || n < 0) return SASSD_ERR_ARG;
    if (n == 0) return SASSD_OK;
    const int colb = (n + 63) / 64;
    cudaMemsetAsync(mask, 0, (size_t)n * colb * 8, (cudaStream_t)stream_);
    const long long nitems = 4ll * colb * (colb + 1) / 2;    // quarter tiles
    dim3 grid((unsigned)(nitems < 148 * 16 ? nitems : 148 * 16), 1);
    nms_mask_kernel<<<grid, NMS_MASK_THREADS, 0, (cudaStream_t)stream_>>>(boxes5, nullptr, n, n, colb, thr,
                                                            (unsigned long long*)mask);
    return sassd_check_launch();
}

extern "C" int sassd_nms_sorted(const float* boxes5, int n, float thr, int64_t* keep, int32_t* d_nkeep, void* ws,
                                size_t ws_bytes, sassd_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!boxes5 || !keep || !d_nkeep || n < 0) return SASSD_ERR_ARG;
    // n == 0 needs no workspace (sassd_nms_workspace_bytes(0) == 0), so ws may be NULL there
    if (n == 0) { cudaMemsetAsync(d_nkeep, 0, 4, stream); return SASSD_OK; }
    if (!ws) return SASSD_ERR_ARG;
    if (ws_bytes < sassd_nms_workspace_bytes(n)) return SASSD_ERR_WORKSPACE;
    const int colb = (n + 63) / 64;
    if ((size_t)colb * 16 > 40000) return SASSD_ERR_UNSUPPORTED;  // > 160k boxes
    int rc = sassd_nms_mask(boxes5, n, thr, (uint64_t*)ws, stream_);
    if (rc != SASSD_OK) return rc;
    nms_keep_kernel<<<1, 256, (size_t)colb * 16, stream>>>((const unsigned long long*)ws, n, colb, (long long*)keep,
                                                           d_nkeep);
    return sassd_check_launch();
}

extern "C" int sassd_boxes_iou_bev(const float* boxes_a, int na, const float* boxes_b, int nb, float* iou,
                                   sassd_stream_t stream_) {
    if (!boxes_a || !boxes_b || !iou || na < 0 || nb < 0) return SASSD_ERR_ARG;
    if (na == 0 || nb == 0) return SASSD_OK;
    dim3 block(16, 16), grid((nb + 15) / 16, (na + 15) / 16);
    iou_matrix_kernel<<<grid, block, 0, (cudaStream_t)stream_>>>(boxes_a, na, boxes_b, nb, iou);
    return sassd_check_launch();
}
