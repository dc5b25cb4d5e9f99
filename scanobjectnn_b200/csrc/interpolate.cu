// interpolate.cu -- three_nn / three_interpolate (+grad) and the fused FP-module interpolation for sm_100a.
//
// The reference implements these only on the CPU (pointnet2/tf_ops/3d_interpolation/tf_interpolate.cpp:60-153,
// single thread, DEVICE_CPU registration :187,222,262), so every PointNet++-BGA step bounces device->host->device
// three times.  Arithmetic is kept bit-identical to that x86-64 (no-FMA) build: squared distance
// (dx*dx+dy*dy)+dz*dz, strict-'<' three-way cascade (earlier k wins ties), output (p1*w1+p2*w2)+p3*w3.
#include "three_nn.cuh"

namespace psa {

__global__ void __launch_bounds__(kNnThreads)
three_nn_kernel(int n, int m, const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                float* __restrict__ dist, int* __restrict__ idx) {
    __shared__ float4 tile[kNnTile];
    const int cloud = blockIdx.y;
    const int j = blockIdx.x * kNnThreads + threadIdx.x;
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
        size_t o = ((size_t)cloud * n + j) * 3;
        dist[o] = s.d1; dist[o + 1] = s.d2; dist[o + 2] = s.d3;
        idx[o] = s.i1; idx[o + 1] = s.i2; idx[o + 2] = s.i3;
    }
}

// out[b,j,l] = (p[i1,l]*w1 + p[i2,l]*w2) + p[i3,l]*w3   -- one thread per (j, 4-channel vector) or scalar
__global__ void three_interpolate_kernel(int m, int c, int n, long long total, const float* __restrict__ points,
                                         const int* __restrict__ idx, const float* __restrict__ weight,
                                         float* __restrict__ out) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        long long row = e / c;   // = b*n + j
        int l = (int)(e - row * c);
        long long bi = row / n;
        const int* id = idx + row * 3;
        const float* w = weight + row * 3;
        const float* pb = points + bi * m * (long long)c + l;
        float a = __fmul_rn(__ldg(pb + (long long)__ldg(id) * c), __ldg(w));
        float b2 = __fmul_rn(__ldg(pb + (long long)__ldg(id + 1) * c), __ldg(w + 1));
        float c3 = __fmul_rn(__ldg(pb + (long long)__ldg(id + 2) * c), __ldg(w + 2));
        out[e] = __fadd_rn(__fadd_rn(a, b2), c3);
    }
}

// pointnet_fp_module's interpolation half in one launch (pointnet_util.py:211-216).
// CTA = kNnThreads unknown points of one cloud: phase 1 thread-per-point 3-NN + weights into shared memory,
// phase 2 the CTA sweeps (point, channel) with channels fastest so the gathers/writes are coalesced.
__global__ void __launch_bounds__(kNnThreads)
three_nn_interpolate_kernel(int n, int m, int c, const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                            const float* __restrict__ points2, float* __restrict__ out, float* __restrict__ dist_o,
                            int* __restrict__ idx_o, float* __restrict__ weight_o) {
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
        size_t o = ((size_t)cloud * n + j) * 3;
        if (dist_o) { dist_o[o] = s.d1; dist_o[o + 1] = s.d2; dist_o[o + 2] = s.d3; }
        if (idx_o) { idx_o[o] = s.i1; idx_o[o + 1] = s.i2; idx_o[o + 2] = s.i3; }
        if (weight_o) { weight_o[o] = w0; weight_o[o + 1] = w1; weight_o[o + 2] = w2; }
    }
    __syncthreads();
    const int rows = min(kNnThreads, n - j0);
    const float* pb = points2 + (size_t)cloud * m * c;
    float* ob = out + ((size_t)cloud * n + j0) * c;
    for (int e = threadIdx.x; e < rows * c; e += kNnThreads) {
        int r = e / c, l = e - r * c;
        float a = __fmul_rn(__ldg(pb + (size_t)s_idx[r][0] * c + l), s_w[r][0]);
        float b2 = __fmul_rn(__ldg(pb + (size_t)s_idx[r][1] * c + l), s_w[r][1]);
        float c3 = __fmul_rn(__ldg(pb + (size_t)s_idx[r][2] * c + l), s_w[r][2]);
        ob[e] = __fadd_rn(__fadd_rn(a, b2), c3);
    }
}

static inline int grid_for(long long total, int block) {
    long long g = (total + block - 1) / block;
    long long cap = (long long)kNumSMs * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace psa

using namespace psa;

extern "C" int psa_three_nn(int b, int n, int m, const float* xyz1, const float* xyz2, float* dist, int* idx,
                            psa_stream_t stream) {
    PSA_REQUIRE(b >= 0 && n >= 0 && m >= 0, "ThreeNN: negative dimension");
    if (b == 0 || n == 0) return PSA_OK;
    PSA_REQUIRE(xyz1 && (xyz2 || m == 0) && dist && idx, "ThreeNN: null buffer");
    PSA_SUPPORTED(b <= 65535, "three_nn: b=%d exceeds gridDim.y", b);
    dim3 grid((n + kNnThreads - 1) / kNnThreads, b);
    three_nn_kernel<<<grid, kNnThreads, 0, as_stream(stream)>>>(n, m, xyz1, xyz2, dist, idx);
    return check_launch("three_nn_kernel");
}

extern "C" int psa_three_interpolate(int b, int m, int c, int n, const float* points, const int* idx,
                                     const float* weight, float* out, psa_stream_t stream) {
    PSA_REQUIRE(b >= 0 && n >= 0 && m >= 0 && c >= 0, "ThreeInterpolate: negative dimension");
    long long total = (long long)b * n * c;
    if (total == 0) return PSA_OK;
    PSA_REQUIRE(points && idx && weight && out, "ThreeInterpolate: null buffer");
    three_interpolate_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(m, c, n, total, points, idx, weight, out);
    return check_launch("three_interpolate_kernel");
}

extern "C" int psa_three_nn_interpolate(int b, int n, int m, int c, const float* xyz1, const float* xyz2,
                                        const float* points2, float* out, float* dist, int* idx, float* weight,
                                        psa_stream_t stream) {
    PSA_REQUIRE(b >= 0 && n >= 0 && m >= 0 && c >= 0, "three_nn_interpolate: negative dimension");
    if (b == 0 || n == 0) return PSA_OK;
    PSA_REQUIRE(m >= 1, "three_nn_interpolate: needs at least one known point (m=%d)", m);
    PSA_REQUIRE(xyz1 && xyz2 && (points2 || c == 0) && (out || c == 0), "three_nn_interpolate: null buffer");
    PSA_SUPPORTED(b <= 65535, "three_nn_interpolate: b=%d exceeds gridDim.y", b);
    dim3 grid((n + kNnThreads - 1) / kNnThreads, b);
    three_nn_interpolate_kernel<<<grid, kNnThreads, 0, as_stream(stream)>>>(n, m, c, xyz1, xyz2, points2, out, dist,
                                                                            idx, weight);
    return check_launch("three_nn_interpolate_kernel");
}
