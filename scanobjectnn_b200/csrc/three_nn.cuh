// three_nn.cuh -- the three-nearest-neighbour search and inverse-distance weights of pointnet_fp_module, shared by the
// inference interpolation (interpolate.cu) and the training-mode FP front (fp_train.cu) so that both produce bit-identical
// idx / weight.  Arithmetic is that of the reference's x86-64 (no-FMA) CPU op (tf_interpolate.cpp:60-103): squared distance
// (dx*dx+dy*dy)+dz*dz, strict-'<' three-way cascade (earlier k wins ties).
#pragma once
#include "common.cuh"

namespace psa {

constexpr int kNnThreads = 128;
constexpr int kNnTile = 2048;   // known points staged per shared-memory tile (float4 each: 32 KB)

struct Best3 {
    float d1, d2, d3;
    int i1, i2, i3;
};

__device__ __forceinline__ void best3_init(Best3& s) {
    // the reference starts its doubles at 1e40; every float compares like +inf against that
    s.d1 = s.d2 = s.d3 = __int_as_float(0x7f800000);
    s.i1 = s.i2 = s.i3 = 0;
}
__device__ __forceinline__ void best3_push(Best3& s, float d, int k) {
    if (d < s.d1) { s.d3 = s.d2; s.i3 = s.i2; s.d2 = s.d1; s.i2 = s.i1; s.d1 = d; s.i1 = k; }
    else if (d < s.d2) { s.d3 = s.d2; s.i3 = s.i2; s.d2 = d; s.i2 = k; }
    else if (d < s.d3) { s.d3 = d; s.i3 = k; }
}

// thread per unknown point; known points streamed through shared memory in index order
__device__ __forceinline__ void three_nn_scan(int m, const float* __restrict__ p2, float4* tile, float x1, float y1,
                                              float z1, bool active, Best3& s) {
    for (int base = 0; base < m; base += kNnTile) {
        const int cnt = min(kNnTile, m - base);
        __syncthreads();
        for (int i0 = threadIdx.x; i0 < cnt; i0 += 4 * kNnThreads) {      // 12 independent loads in flight per thread
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * kNnThreads;
                const float* q = p2 + (size_t)(base + (i < cnt ? i : 0)) * 3;
                v[u] = make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * kNnThreads;
                if (i < cnt) tile[i] = v[u];
            }
        }
        __syncthreads();
        if (active) {
#pragma unroll 4
            for (int k = 0; k < cnt; ++k) {
                const float4 q = tile[k];   // broadcast LDS.128
                // tf_interpolate.cpp:73: (x2-x1)^2 + (y2-y1)^2 + (z2-z1)^2, x2 = known point
                float d = dist2_ref_cpu(q.x - x1, q.y - y1, q.z - z1);
                best3_push(s, d, base + k);
            }
        }
    }
}

// pointnet_util.py:212-214: dist = max(dist,1e-10); norm = sum(1/dist); weight = (1/dist)/norm   (IEEE division, in order).
// Slots beyond m hold dist = +inf and get weight 0.
__device__ __forceinline__ void three_weights(const Best3& s, float& w0, float& w1, float& w2) {
    float r0 = __fdiv_rn(1.0f, fmaxf(s.d1, 1e-10f));
    float r1 = __fdiv_rn(1.0f, fmaxf(s.d2, 1e-10f));
    float r2 = __fdiv_rn(1.0f, fmaxf(s.d3, 1e-10f));
    float nrm = __fadd_rn(__fadd_rn(r0, r1), r2);
    w0 = __fdiv_rn(r0, nrm); w1 = __fdiv_rn(r1, nrm); w2 = __fdiv_rn(r2, nrm);
}

}  // namespace psa
