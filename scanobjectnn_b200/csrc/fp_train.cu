// fp_train.cu -- training mode of the feature-propagation (FP) module and the joint loss of pointnet2_cls_bga.
//
// The reference's pointnet_fp_module (pointnet2/utils/pointnet_util.py:199-229) runs three_nn + three_interpolate on the CPU
// (tf_interpolate.cpp:60-153), concatenates [interpolated, skip] and feeds a 1x1 conv.  The interpolation is linear, so the first
// conv distributes over it:
//     y = [sum_i w_i P2[idx_i], skip] . W1 + b  =  sum_i w_i U[idx_i] + skip . W1[C_a:] + b,      U = P2 . W1[:C_a]
// U has one row per KNOWN point (4x fewer rows than unknown points at fa_layer2/3, one row per cloud at fa_layer1).  U and the
// skip product come from psa_train_dense_fwd; fp_conv1_prebn_kernel adds the interpolated U rows, writes idx / weight for the
// backward and the batch-norm sums.  The (b, n, C_a) interpolated tensor and the concatenation never exist in HBM.
//
// Backward: dU = ThreeInterpolateGrad(dy0) (tf_interpolate.cpp:131-153) with dy0 evaluated on load from a psa_grad_in, in the
// ordered scheme of scatter.cu (stable counting sort by destination, then a gather; products rounded before the add): with a plain
// gradient it is bit-identical to psa_three_interpolate_grad.
//
// Joint loss (pointnet2_cls_bga.py:78-93): (1-w) * mean CE(class) + w * mean CE(per-point mask), fixed-order sums.
#include <math.h>

#include "three_nn.cuh"
#include "train_gemm.cuh"

namespace psa {

// CTA = kNnThreads unknown points of one cloud.  Phase 1: thread-per-point 3-NN + weights (three_nn.cuh).  Phase 2: thread =
// (channel quad, row lane); pre[r] (+)= (U[i1] w1 + U[i2] w2) + U[i3] w3 (+ bias), per-channel sum / sum of squares of the stored
// values added over the row lanes in order into one partial per CTA.
template <bool ACC>
__global__ void __launch_bounds__(kNnThreads)
fp_conv1_prebn_kernel(int n, int m, int C1, const float* __restrict__ xyz1, const float* __restrict__ xyz2, const float* __restrict__ U,
                      const float* __restrict__ bias, float* __restrict__ pre, int* __restrict__ idx_o, float* __restrict__ weight_o,
                      float* __restrict__ partial) {
    __shared__ float4 tile[kNnTile];
    __shared__ int s_idx[kNnThreads][3];
    __shared__ float s_w[kNnThreads][3];
    const int cloud = blockIdx.y;
    const int j0 = blockIdx.x * kNnThreads;
    const int j = j0 + threadIdx.x;
    const bool active = j < n;
    float x1 = 0.f, y1 = 0.f, z1 = 0.f;
    if (active) {
        const float* p = xyz1 + ((size_t)cloud * n + j) * 3;
        x1 = __ldg(p); y1 = __ldg(p + 1); z1 = __ldg(p + 2);
    }
    Best3 s;
    best3_init(s);
    three_nn_scan(m, xyz2 + (size_t)cloud * m * 3, tile, x1, y1, z1, active, s);
    if (active) {
        float w0, w1, w2;
        three_weights(s, w0, w1, w2);
        s_idx[threadIdx.x][0] = s.i1; s_idx[threadIdx.x][1] = s.i2; s_idx[threadIdx.x][2] = s.i3;
        s_w[threadIdx.x][0] = w0; s_w[threadIdx.x][1] = w1; s_w[threadIdx.x][2] = w2;
        const size_t o = ((size_t)cloud * n + j) * 3;
        idx_o[o] = s.i1; idx_o[o + 1] = s.i2; idx_o[o + 2] = s.i3;
        weight_o[o] = w0; weight_o[o + 1] = w1; weight_o[o + 2] = w2;
    }
    __syncthreads();
    const int rows = min(kNnThreads, n - j0);
    const int C4 = C1 >> 2, RL = kNnThreads / C4;
    const int cq = threadIdx.x % C4, rl = threadIdx.x / C4;
    const float4* Ub = reinterpret_cast<const float4*>(U + (size_t)cloud * m * C1) + cq;
    float4* pb = reinterpret_cast<float4*>(pre + ((size_t)cloud * n + j0) * C1) + cq;
    float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!ACC && bias != nullptr) bs = __ldg(reinterpret_cast<const float4*>(bias) + cq);
    float4 sm = make_float4(0.f, 0.f, 0.f, 0.f), sq = sm;
    if (rl < RL) {
        for (int r = rl; r < rows; r += RL) {
            const float4 a = __ldg(Ub + (size_t)s_idx[r][0] * C4), b = __ldg(Ub + (size_t)s_idx[r][1] * C4), c = __ldg(Ub + (size_t)s_idx[r][2] * C4);
            const float wa = s_w[r][0], wb = s_w[r][1], wc = s_w[r][2];
            float4 v;
            v.x = __fadd_rn(__fadd_rn(__fmul_rn(a.x, wa), __fmul_rn(b.x, wb)), __fmul_rn(c.x, wc));
            v.y = __fadd_rn(__fadd_rn(__fmul_rn(a.y, wa), __fmul_rn(b.y, wb)), __fmul_rn(c.y, wc));
            v.z = __fadd_rn(__fadd_rn(__fmul_rn(a.z, wa), __fmul_rn(b.z, wb)), __fmul_rn(c.z, wc));
            v.w = __fadd_rn(__fadd_rn(__fmul_rn(a.w, wa), __fmul_rn(b.w, wb)), __fmul_rn(c.w, wc));
            const float4 base = ACC ? pb[(size_t)r * C4] : bs;
            v.x = __fadd_rn(base.x, v.x); v.y = __fadd_rn(base.y, v.y); v.z = __fadd_rn(base.z, v.z); v.w = __fadd_rn(base.w, v.w);
            pb[(size_t)r * C4] = v;
            sm.x += v.x; sm.y += v.y; sm.z += v.z; sm.w += v.w;
            sq.x = fmaf(v.x, v.x, sq.x); sq.y = fmaf(v.y, v.y, sq.y); sq.z = fmaf(v.z, v.z, sq.z); sq.w = fmaf(v.w, v.w, sq.w);
        }
    }
    if (partial == nullptr) return;
    // reuse the tile for the per-thread sums: (kNnThreads, 8) floats = 4 KB of the 32 KB tile
    __syncthreads();
    float* red = reinterpret_cast<float*>(tile);
    float* mine = red + threadIdx.x * 8;
    mine[0] = sm.x; mine[1] = sm.y; mine[2] = sm.z; mine[3] = sm.w; mine[4] = sq.x; mine[5] = sq.y; mine[6] = sq.z; mine[7] = sq.w;
    __syncthreads();
    float* dst = partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 2 * C1;
    for (int e = threadIdx.x; e < 2 * C1; e += kNnThreads) {
        const int which = e / C1, c = e - which * C1;
        float t = 0.f;
        for (int r = 0; r < RL; ++r) t += red[(r * C4 + (c >> 2)) * 8 + which * 4 + (c & 3)];      // row lanes in order
        dst[e] = t;
    }
}

// stats[e] = sum_p partial[p][e] in CTA order, in fp64
__global__ void fp_stats_reduce_kernel(int nparts, int twoC, const float* __restrict__ partial, float* __restrict__ stats) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= twoC) return;
    double s = 0.0;
    for (int p = 0; p < nparts; ++p) s += (double)__ldcg(partial + (size_t)p * twoC + e);
    stats[e] = (float)s;
}

// ThreeInterpolateGrad of the training path: one warp per KNOWN point (lane = 4 channels), entries e = 3*row + slot of the cloud
// in ascending order (scatter.cu's CSR), dU += round(dy0[row] * w[e]).  Same sum order and rounding as scatter_rows_kernel.
__global__ void __launch_bounds__(256)
fp_interp_grad_kernel(const GradIn g, int n, int m, int C1, long long total_points, const int* __restrict__ offsets,
                      const int* __restrict__ list, const float* __restrict__ weight, float* __restrict__ dU) {
    const int lane = threadIdx.x & 31;
    const long long pt = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);           // global known point b*m + k
    if (pt >= total_points) return;
    const long long cloud = pt / m;
    const int k = (int)(pt - cloud * m);
    const int mk = 3 * n;
    const int* off = offsets + (size_t)cloud * (m + 1);
    const int* lst = list + (size_t)cloud * mk;
    const float* wc = weight + (size_t)cloud * mk;
    const long long row0 = cloud * n;
    const int t0 = __ldg(off + k), t1 = __ldg(off + k + 1);
    for (int c0 = 0; c0 < C1; c0 += 128) {
        const int c = c0 + lane * 4;
        if (c >= C1) break;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int t = t0;
        for (; t + 3 < t1; t += 4) {                                              // four entries in flight, added in list order
            int e[4];
            float w[4];
            float4 d[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) e[u] = __ldg(lst + t + u);
#pragma unroll
            for (int u = 0; u < 4; ++u) { w[u] = __ldg(wc + e[u]); d[u] = g.get4(row0 + e[u] / 3, c); }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                acc.x = __fadd_rn(acc.x, __fmul_rn(d[u].x, w[u])); acc.y = __fadd_rn(acc.y, __fmul_rn(d[u].y, w[u]));
                acc.z = __fadd_rn(acc.z, __fmul_rn(d[u].z, w[u])); acc.w = __fadd_rn(acc.w, __fmul_rn(d[u].w, w[u]));
            }
        }
        for (; t < t1; ++t) {
            const int e0 = __ldg(lst + t);
            const float w0 = __ldg(wc + e0);
            const float4 d0 = g.get4(row0 + e0 / 3, c);
            acc.x = __fadd_rn(acc.x, __fmul_rn(d0.x, w0)); acc.y = __fadd_rn(acc.y, __fmul_rn(d0.y, w0));
            acc.z = __fadd_rn(acc.z, __fmul_rn(d0.z, w0)); acc.w = __fadd_rn(acc.w, __fmul_rn(d0.w, w0));
        }
        *reinterpret_cast<float4*>(dU + (size_t)pt * C1 + c) = acc;
    }
}

// ---- joint loss ----
constexpr int kXentThreads = 256;
constexpr int kSegRowsPerBlock = 8 * kXentThreads;

// fixed-order tree over the block's threads (kXentThreads doubles)
__device__ __forceinline__ double block_sum(double v, double* red) {
    red[threadIdx.x] = v;
    __syncthreads();
    for (int o = kXentThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    return red[0];
}

// one softmax cross-entropy row: loss, and d = (softmax - onehot) * scale written to drow.  A label outside [0, c) gives NaN (the
// reference's sparse_softmax_cross_entropy on the GPU).
__device__ __forceinline__ float xent_row(const float* __restrict__ l, int c, int lab, float scale, float* __restrict__ drow) {
    float mx = l[0];
    for (int i = 1; i < c; ++i) mx = fmaxf(mx, l[i]);
    float se = 0.f;
    for (int i = 0; i < c; ++i) se += expf(l[i] - mx);
    const bool ok = (unsigned)lab < (unsigned)c;
    for (int i = 0; i < c; ++i) drow[i] = ok ? (expf(l[i] - mx) / se - (i == lab ? 1.f : 0.f)) * scale : __int_as_float(0x7fc00000);
    return ok ? (logf(se) + mx) - l[lab] : __int_as_float(0x7fc00000);
}

// per-point 2-way cross-entropy: rows [blockIdx.x * kSegRowsPerBlock, +kSegRowsPerBlock), block sum of the row losses -> partial
__global__ void __launch_bounds__(kXentThreads)
seg_xent_kernel(long long rows, const float* __restrict__ seg, const int* __restrict__ mask, float scale, float* __restrict__ dseg,
                double* __restrict__ partial) {
    __shared__ double red[kXentThreads];
    const long long r0 = (long long)blockIdx.x * kSegRowsPerBlock;
    double s = 0.0;
    for (int k = 0; k < kSegRowsPerBlock / kXentThreads; ++k) {
        const long long r = r0 + k * kXentThreads + threadIdx.x;
        if (r < rows) s += (double)xent_row(seg + r * 2, 2, __ldg(mask + r), scale, dseg + r * 2);
    }
    const double t = block_sum(s, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

// class cross-entropy over the b rows + the seg partials in block order -> loss = [total, classify, seg]
__global__ void __launch_bounds__(kXentThreads)
cls_xent_final_kernel(int b, int c, long long seg_rows, const float* __restrict__ cls, const int* __restrict__ labels, float seg_weight,
                      float* __restrict__ dcls, int nparts, const double* __restrict__ partial, float* __restrict__ loss) {
    __shared__ double red[kXentThreads];
    const float cscale = (1.f - seg_weight) / (float)b;
    double s = 0.0;
    for (int r = threadIdx.x; r < b; r += kXentThreads) s += (double)xent_row(cls + (size_t)r * c, c, __ldg(labels + r), cscale, dcls + (size_t)r * c);
    const double tot = block_sum(s, red);
    if (threadIdx.x == 0) {
        double sg = 0.0;
        for (int p = 0; p < nparts; ++p) sg += partial[p];
        const double classify = tot / b, segl = sg / (double)seg_rows, w = seg_weight;
        loss[0] = (float)((1.0 - w) * classify + w * segl);
        loss[1] = (float)classify;
        loss[2] = (float)segl;
    }
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace psa

using namespace psa;

extern "C" size_t psa_fp_conv1_prebn_workspace_bytes(int b, int n, int C1) {
    if (b <= 0 || n <= 0 || C1 <= 0) return 256;
    return (size_t)b * ((n + kNnThreads - 1) / kNnThreads) * 2 * (size_t)C1 * sizeof(float) + 256;
}

extern "C" int psa_fp_conv1_prebn(int b, int n, int m, int C1, const float* xyz1, const float* xyz2, const float* U, const float* bias,
                                  int accumulate, float* pre, int* idx, float* weight, float* stats, void* workspace, size_t workspace_bytes,
                                  psa_stream_t stream) {
    PSA_REQUIRE(b >= 0 && n >= 0 && m >= 0, "fp_conv1_prebn: negative dimension");
    PSA_REQUIRE(C1 >= 4 && C1 % 4 == 0 && C1 <= 4 * kNnThreads, "fp_conv1_prebn: C1=%d must be a multiple of 4 in [4, %d]", C1, 4 * kNnThreads);
    if (b == 0 || n == 0) return PSA_OK;
    PSA_REQUIRE(m >= 1, "fp_conv1_prebn: needs at least one known point (m=%d)", m);
    PSA_REQUIRE(xyz1 && xyz2 && U && pre && idx && weight, "fp_conv1_prebn: null buffer");
    PSA_REQUIRE(aligned16(U) && aligned16(pre) && (bias == nullptr || aligned16(bias)), "fp_conv1_prebn: U, pre and bias must be 16-byte aligned");
    PSA_SUPPORTED(b <= 65535, "fp_conv1_prebn: b=%d exceeds gridDim.y", b);
    dim3 grid((n + kNnThreads - 1) / kNnThreads, b);
    float* partial = nullptr;
    if (stats != nullptr) {
        const size_t need = psa_fp_conv1_prebn_workspace_bytes(b, n, C1);
        PSA_REQUIRE(workspace != nullptr && workspace_bytes >= need, "fp_conv1_prebn: workspace of %zu bytes required", need);
        partial = reinterpret_cast<float*>(workspace);
    }
    cudaStream_t st = as_stream(stream);
    if (accumulate)
        fp_conv1_prebn_kernel<true><<<grid, kNnThreads, 0, st>>>(n, m, C1, xyz1, xyz2, U, nullptr, pre, idx, weight, partial);
    else
        fp_conv1_prebn_kernel<false><<<grid, kNnThreads, 0, st>>>(n, m, C1, xyz1, xyz2, U, bias, pre, idx, weight, partial);
    int rc = check_launch("fp_conv1_prebn_kernel");
    if (rc != PSA_OK || stats == nullptr) return rc;
    fp_stats_reduce_kernel<<<(2 * C1 + 127) / 128, 128, 0, st>>>((int)(grid.x * grid.y), 2 * C1, partial, stats);
    return check_launch("fp_stats_reduce_kernel");
}

extern "C" size_t psa_fp_conv1_bwd_workspace_bytes(int b, int n, int m) {
    if (b <= 0 || n <= 0 || m <= 0) return 256;
    return ((size_t)b * ((size_t)m + 1) + (size_t)b * 3 * (size_t)n) * sizeof(int) + 256;
}

extern "C" int psa_fp_conv1_bwd(int b, int n, int m, int C1, const int* idx, const float* weight, const psa_grad_in* g, float* dU,
                                void* workspace, size_t workspace_bytes, psa_stream_t stream) {
    PSA_REQUIRE(b >= 0 && n >= 0 && m >= 0, "fp_conv1_bwd: negative dimension");
    PSA_REQUIRE(C1 >= 4 && C1 % 4 == 0, "fp_conv1_bwd: C1=%d must be a positive multiple of 4", C1);
    if (b == 0 || m == 0) return PSA_OK;
    PSA_REQUIRE(dU != nullptr, "fp_conv1_bwd: null output");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        PSA_CUDA(cudaMemsetAsync(dU, 0, (size_t)b * m * C1 * sizeof(float), st));
        return PSA_OK;
    }
    PSA_REQUIRE(idx && weight && g, "fp_conv1_bwd: null buffer");
    PSA_REQUIRE(g->C == C1 && g->mode == 0 && g->dh != nullptr && g->ld_dh % 4 == 0 && (g->y == nullptr || g->ld % 4 == 0) && aligned16(dU),
                "fp_conv1_bwd: the gradient must be a dense (mode 0) psa_grad_in over C1 channels with row strides that are multiples of 4");
    // fp_interp_grad_kernel reads every operand of g as float4 (GradIn::get4)
    PSA_REQUIRE(((g->s == nullptr && g->ca == nullptr) || g->y != nullptr) && (g->s == nullptr || !g->relu || g->t != nullptr) &&
                    (g->ca == nullptr || (g->cb != nullptr && g->cc != nullptr)),
                "fp_conv1_bwd: psa_grad_in with batch-norm terms needs y (and t with relu, cb / cc with ca)");
    PSA_REQUIRE(aligned16(g->dh) && aligned16(g->mask) && aligned16(g->y) && aligned16(g->s) && aligned16(g->t) && aligned16(g->ca) &&
                    aligned16(g->cb) && aligned16(g->cc),
                "fp_conv1_bwd: every buffer of the psa_grad_in must be 16-byte aligned");
    PSA_SUPPORTED(3LL * n <= 0x7fffffffLL, "fp_conv1_bwd: n=%d too large", n);
    const size_t need = psa_fp_conv1_bwd_workspace_bytes(b, n, m);
    PSA_REQUIRE(workspace != nullptr && workspace_bytes >= need, "fp_conv1_bwd: workspace of %zu bytes required", need);
    int* offsets = reinterpret_cast<int*>(workspace);
    int* list = offsets + (size_t)b * ((size_t)m + 1);
    int rc = launch_group_csr(b, m, 3 * n, idx, offsets, list, st);
    if (rc != PSA_OK) return rc;
    const long long pts = (long long)b * m;
    fp_interp_grad_kernel<<<(unsigned)((pts + 7) / 8), 256, 0, st>>>(GradIn(*g), n, m, C1, pts, offsets, list, weight, dU);
    return check_launch("fp_interp_grad_kernel");
}

extern "C" size_t psa_cls_seg_xent_workspace_bytes(int b, int n) {
    if (b <= 0 || n <= 0) return 256;
    const long long rows = (long long)b * n;
    return (size_t)((rows + kSegRowsPerBlock - 1) / kSegRowsPerBlock) * sizeof(double) + 256;
}

extern "C" int psa_cls_seg_xent(int b, int c, int n, const float* cls_logits, const int* labels, const float* seg_logits, const int* mask,
                                float seg_weight, float* loss, float* dcls, float* dseg, void* workspace, size_t workspace_bytes,
                                psa_stream_t stream) {
    PSA_REQUIRE(b >= 1 && c >= 1 && n >= 1, "cls_seg_xent: bad dims b=%d c=%d n=%d", b, c, n);
    PSA_REQUIRE(cls_logits && labels && seg_logits && mask && loss && dcls && dseg, "cls_seg_xent: null buffer");
    PSA_REQUIRE(seg_weight >= 0.f && seg_weight <= 1.f, "cls_seg_xent: seg_weight=%g outside [0, 1]", (double)seg_weight);
    const size_t need = psa_cls_seg_xent_workspace_bytes(b, n);
    PSA_REQUIRE(workspace != nullptr && workspace_bytes >= need, "cls_seg_xent: workspace of %zu bytes required", need);
    cudaStream_t st = as_stream(stream);
    const long long rows = (long long)b * n;
    const long long blocks = (rows + kSegRowsPerBlock - 1) / kSegRowsPerBlock;
    PSA_SUPPORTED(blocks <= 0x7fffffffLL, "cls_seg_xent: %lld rows", rows);
    double* partial = reinterpret_cast<double*>(workspace);
    seg_xent_kernel<<<(unsigned)blocks, kXentThreads, 0, st>>>(rows, seg_logits, mask, seg_weight / (float)rows, dseg, partial);
    int rc = check_launch("seg_xent_kernel");
    if (rc != PSA_OK) return rc;
    cls_xent_final_kernel<<<1, kXentThreads, 0, st>>>(b, c, rows, cls_logits, labels, seg_weight, dcls, (int)blocks, partial, loss);
    return check_launch("cls_xent_final_kernel");
}
