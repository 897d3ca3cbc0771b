// ccu_denoise.cuh - the guided denoiser (DESIGN §17): an edge-avoiding a-trous wavelet filter (Dammertz et al. 2010) on
// demodulated irradiance, with an SVGF-style luminance stop scaled by a spatial variance estimate.  Included only by its own
// unit (denoise.cu); chunkycu.cu calls denoise_launch.
//
// Arithmetic contract as for the render path: every fp32 operation is one IEEE round-to-nearest operation in the order written
// (-fmad=false -prec-div=true -prec-sqrt=true), dot is dot3 (§2 rule 2) and exp is dm_expf_weight, so that the CPU restatement
// (specular_oracle.c, denoise) evaluates the same bits.
#pragma once
#include "ccu_math.cuh"

namespace ccu {

#define CCU_DN_TX 32   // a-trous / variance block: 32 x 8 pixels, one warp per row
#define CCU_DN_TY 8
#define CCU_DN_R 3     // the variance window is 7 x 7

// Working records, one float4 per pixel each: E = (irradiance.rgb, variance) twice (ping-pong), A = (albedo.rgb, valid) and
// N = (normal.xyz, 0), both constant over the iterations.
__device__ __forceinline__ float dn_lum(float4 v) { return 0.2126f * v.x + 0.7152f * v.y + 0.0722f * v.z; }
__device__ __forceinline__ float dn_albedo_floor(float a) { return fmaxf(a, 0x1p-8f); }
// the B3-spline taps 1/16, 1/4, 3/8, 1/4, 1/16 at offset d in [-2, 2]
__device__ __forceinline__ float dn_k(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1 ? 0.25f : 0.0625f); }

// the pixel of this thread in a CCU_DN_TX x CCU_DN_TY tile; tiles are numbered row-major over a one-dimensional grid, so that
// any image height fits the grid
__device__ __forceinline__ void dn_tile_origin(int w, int &x0, int &y0) {
    const unsigned tiles_x = (unsigned)(w + CCU_DN_TX - 1) / CCU_DN_TX;
    x0 = (int)(blockIdx.x % tiles_x) * CCU_DN_TX;
    y0 = (int)(blockIdx.x / tiles_x) * CCU_DN_TY;
}

// §17 step 1: demodulation, the validity flag and the constant guide records
__global__ void __launch_bounds__(256) k_dn_setup(int64_t n, const double *__restrict__ color, const float *__restrict__ albedo,
                                                  const float *__restrict__ normal, float4 *__restrict__ E, float4 *__restrict__ A,
                                                  float4 *__restrict__ N) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float c[3], a[3], nv[3];
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        c[k] = (float)color[3 * i + k];
        a[k] = albedo[3 * i + k];
        nv[k] = normal[3 * i + k];
        ok = ok && isfinite(c[k]) && isfinite(a[k]) && isfinite(nv[k]);
    }
    E[i] = make_float4(c[0] / dn_albedo_floor(a[0]), c[1] / dn_albedo_floor(a[1]), c[2] / dn_albedo_floor(a[2]), 0.0f);
    A[i] = make_float4(a[0], a[1], a[2], ok ? 1.0f : 0.0f);
    N[i] = make_float4(nv[0], nv[1], nv[2], 0.0f);
}

// §17 step 2: the luminance variance over the valid pixels of the 7 x 7 window inside the image, from a shared-memory tile
// of luminances and validity flags.  Writes Eout = (Ein.rgb, variance).
__global__ void __launch_bounds__(CCU_DN_TX * CCU_DN_TY) k_dn_variance(int w, int h, const float4 *__restrict__ E,
                                                                      const float4 *__restrict__ A, float4 *__restrict__ Eout) {
    constexpr int TW = CCU_DN_TX + 2 * CCU_DN_R, TH = CCU_DN_TY + 2 * CCU_DN_R;
    __shared__ float lum[TH][TW];
    __shared__ bool ok[TH][TW];
    int x0, y0;
    dn_tile_origin(w, x0, y0);
    for (int j = threadIdx.y * CCU_DN_TX + threadIdx.x; j < TW * TH; j += CCU_DN_TX * CCU_DN_TY) {
        const int gx = x0 - CCU_DN_R + j % TW, gy = y0 - CCU_DN_R + j / TW;
        float l = 0.0f;
        bool v = false;
        if (gx >= 0 && gx < w && gy >= 0 && gy < h) {
            const int64_t g = (int64_t)gy * w + gx;
            v = A[g].w != 0.0f;
            if (v) l = dn_lum(E[g]);
        }
        lum[j / TW][j % TW] = l;
        ok[j / TW][j % TW] = v;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= w || y >= h) return;
    const int64_t g = (int64_t)y * w + x;
    const float4 e = E[g];
    float var = 0.0f;
    if (A[g].w != 0.0f) {
        float s1 = 0.0f, s2 = 0.0f, m = 0.0f;
#pragma unroll
        for (int dy = 0; dy <= 2 * CCU_DN_R; dy++)
#pragma unroll
            for (int dx = 0; dx <= 2 * CCU_DN_R; dx++) {
                if (!ok[threadIdx.y + dy][threadIdx.x + dx]) continue;
                const float l = lum[threadIdx.y + dy][threadIdx.x + dx];
                s1 = s1 + l;
                s2 = s2 + l * l;
                m = m + 1.0f;
            }
        const float mu = s1 / m;
        var = fmaxf(0.0f, s2 / m - mu * mu);
    }
    Eout[g] = make_float4(e.x, e.y, e.z, var);
}

// §17 step 3, one iteration with step `step`: the 5 x 5 taps p + step * (dx, dy) in row-major order, read through the read-only
// path (the footprint of a warp's taps is 32 x 5 records, L1-resident for the small steps).  LAST also remodulates and stores
// Chunky's doubles (§17 step 4) instead of the working record.
template <bool LAST>
__global__ void __launch_bounds__(CCU_DN_TX * CCU_DN_TY, 4) k_dn_atrous(int w, int h, int step, float sigma_l,
                                                                    const float4 *__restrict__ E, const float4 *__restrict__ A,
                                                                    const float4 *__restrict__ N, float4 *__restrict__ Eout,
                                                                    double *__restrict__ out) {
    int x0, y0;
    dn_tile_origin(w, x0, y0);
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= w || y >= h) return;
    const int64_t g = (int64_t)y * w + x;
    const float4 ep = __ldg(&E[g]), ap = __ldg(&A[g]);
    float4 r = ep;
    if (ap.w != 0.0f) {
        const float4 np4 = __ldg(&N[g]);
        const float3 np = f3(np4.x, np4.y, np4.z), a3 = f3(ap.x, ap.y, ap.z);
        const bool sky_p = np.x == 0.0f && np.y == 0.0f && np.z == 0.0f;
        const float lp = dn_lum(ep);
        const float dl_den = sigma_l * sqrtf(ep.w) + 1e-4f;
        float sw = 0.0f, sv = 0.0f, sx = 0.0f, sy = 0.0f, sz = 0.0f;
#pragma unroll
        for (int dy = -2; dy <= 2; dy++) {
            const int qy = y + dy * step;
            if (qy < 0 || qy >= h) continue;
#pragma unroll
            for (int dx = -2; dx <= 2; dx++) {
                const int qx = x + dx * step;
                if (qx < 0 || qx >= w) continue;
                const int64_t q = (int64_t)qy * w + qx;
                float4 eq;
                float wt;
                if (dx == 0 && dy == 0) {
                    eq = ep;
                    wt = 9.0f / 64.0f;
                } else {
                    const float4 aq = __ldg(&A[q]);
                    if (aq.w == 0.0f) continue;
                    const float4 nq = __ldg(&N[q]);
                    eq = __ldg(&E[q]);
                    const float dl = fabsf(lp - dn_lum(eq)) / dl_den;
                    const float3 dv = a3 - f3(aq.x, aq.y, aq.z);
                    const float da = dot3(dv, dv) / 0.01f;
                    float wn = 1.0f;
                    if (!(sky_p && nq.x == 0.0f && nq.y == 0.0f && nq.z == 0.0f)) {
                        wn = fmaxf(0.0f, dot3(np, f3(nq.x, nq.y, nq.z)));
#pragma unroll
                        for (int s = 0; s < 7; s++) wn = wn * wn;
                    }
                    wt = dn_k(dx) * dn_k(dy) * wn * dm_expf_weight(-(dl + da));
                }
                sx = sx + wt * eq.x;
                sy = sy + wt * eq.y;
                sz = sz + wt * eq.z;
                sv = sv + wt * wt * eq.w;
                sw = sw + wt;
            }
        }
        r = make_float4(sx / sw, sy / sw, sz / sw, sv / (sw * sw));
    }
    if (!LAST) {
        Eout[g] = r;
    } else {
        out[3 * g] = (double)(r.x * dn_albedo_floor(ap.x));
        out[3 * g + 1] = (double)(r.y * dn_albedo_floor(ap.y));
        out[3 * g + 2] = (double)(r.z * dn_albedo_floor(ap.z));
    }
}

// §17 step 4 alone (iterations = 0): the demodulate / remodulate round trip
__global__ void __launch_bounds__(256) k_dn_remodulate(int64_t n, const float4 *__restrict__ E, const float4 *__restrict__ A,
                                                       double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 e = E[i], a = A[i];
    out[3 * i] = (double)(e.x * dn_albedo_floor(a.x));
    out[3 * i + 1] = (double)(e.y * dn_albedo_floor(a.y));
    out[3 * i + 2] = (double)(e.z * dn_albedo_floor(a.z));
}

// The whole filter on the stream: io = double[3WH], the colour on entry and the result on return; albedo, normal = float[3WH];
// rec = 4 * W * H records (E0, E1, A, N).  W * H <= 2^34, so that every grid below fits.  Returns the number of kernels launched.
int denoise_launch(cudaStream_t st, int w, int h, int iterations, float sigma_l, double *io, const float *albedo, const float *normal,
                   float4 *rec) {
    const int64_t n = (int64_t)w * h;
    float4 *e0 = rec, *e1 = rec + n, *a = rec + 2 * n, *nrm = rec + 3 * n;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    k_dn_setup<<<blocks, 256, 0, st>>>(n, io, albedo, normal, e0, a, nrm);
    if (iterations == 0) {
        k_dn_remodulate<<<blocks, 256, 0, st>>>(n, e0, a, io);
        return 2;
    }
    const dim3 block(CCU_DN_TX, CCU_DN_TY);
    const unsigned tiles = (unsigned)(((int64_t)w + CCU_DN_TX - 1) / CCU_DN_TX * (((int64_t)h + CCU_DN_TY - 1) / CCU_DN_TY));
    k_dn_variance<<<tiles, block, 0, st>>>(w, h, e0, a, e1);
    const float4 *src = e1;
    float4 *dst = e0;
    for (int i = 0; i < iterations; i++) {
        if (i + 1 < iterations) {
            k_dn_atrous<false><<<tiles, block, 0, st>>>(w, h, 1 << i, sigma_l, src, a, nrm, dst, nullptr);
            float4 *t = const_cast<float4 *>(src);
            src = dst;
            dst = t;
        } else {
            k_dn_atrous<true><<<tiles, block, 0, st>>>(w, h, 1 << i, sigma_l, src, a, nrm, nullptr, io);
        }
    }
    return 2 + iterations;
}

}  // namespace ccu
