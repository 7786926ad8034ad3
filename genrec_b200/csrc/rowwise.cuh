// genrec_b200 - row-wise (per token) kernels: LayerNorm / gate / residual forward+backward, casts, column sums,
// embedding gather/scatter, the row passes of the fused cross-entropy, fused Adam.  HBM-bound; one warp per token row,
// 8-byte (bf16x4 / float2) vector accesses, D % 64 == 0, D <= 512.
#pragma once
#include "common.cuh"

namespace grb {

constexpr int ROW_THREADS = 256;  // 8 warps = 8 rows in flight per CTA

struct LnStats { float mean, rstd; };

// lane owns column pairs c = 2*lane + 64*p , p < NP
template <int NP>
GRB_DEVINL LnStats row_stats(const float (&v)[NP][2], int D, float eps) {
    float s = 0.f;
#pragma unroll
    for (int p = 0; p < NP; ++p) s += v[p][0] + v[p][1];
    float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int p = 0; p < NP; ++p) {
        float a = v[p][0] - mean, b = v[p][1] - mean;
        q += a * a + b * b;
    }
    float var = warp_sum(q) / (float)D;
    LnStats st;
    st.mean = mean;
    st.rstd = rsqrtf(var + eps);
    return st;
}

// ------------------------------------------------------------------------------------------------ HSTU: norm + gate + residual + norm
//   N = LN1(O) ; x1 = x + drop(N * U) ; xn = LN2(x1)          (genrec/models/hstu.py:271-278)
struct LnGateFwdArgs {
    const bf16* O; int ldo;
    const bf16* U; int ldu;
    const float* x;
    const float *g1, *b1, *g2, *b2;
    float* x1; bf16* xn;
    float* st1; float* st2;  // [T,2]
    int T, D;
    float eps;
    Dropout drop;
};
template <int NP>
__global__ void __launch_bounds__(ROW_THREADS) ln_gate_fwd_kernel(LnGateFwdArgs a) {
    pdl_wait();
    a.drop.resolve();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        float o[NP][2], u[NP][2], xv[NP][2];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float2 t = unpack_bf16(*reinterpret_cast<const uint32_t*>(a.O + (size_t)row * a.ldo + c));
            o[p][0] = t.x; o[p][1] = t.y;
            t = unpack_bf16(*reinterpret_cast<const uint32_t*>(a.U + (size_t)row * a.ldu + c));
            u[p][0] = t.x; u[p][1] = t.y;
            float2 f = *reinterpret_cast<const float2*>(a.x + (size_t)row * a.D + c);
            xv[p][0] = f.x; xv[p][1] = f.y;
        }
        LnStats s1 = row_stats<NP>(o, a.D, a.eps);
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float gv[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) gv[e] = ((o[p][e] - s1.mean) * s1.rstd * a.g1[c + e] + a.b1[c + e]) * u[p][e];
            a.drop.apply2(gv[0], gv[1], row, c);
            xv[p][0] += gv[0];
            xv[p][1] += gv[1];
            *reinterpret_cast<float2*>(a.x1 + (size_t)row * a.D + c) = make_float2(xv[p][0], xv[p][1]);
        }
        LnStats s2 = row_stats<NP>(xv, a.D, a.eps);
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float y0 = (xv[p][0] - s2.mean) * s2.rstd * a.g2[c] + a.b2[c];
            float y1 = (xv[p][1] - s2.mean) * s2.rstd * a.g2[c + 1] + a.b2[c + 1];
            *reinterpret_cast<uint32_t*>(a.xn + (size_t)row * a.D + c) = pack_bf16(y0, y1);
        }
        if (lane == 0) {
            a.st1[2 * row] = s1.mean; a.st1[2 * row + 1] = s1.rstd;
            a.st2[2 * row] = s2.mean; a.st2[2 * row + 1] = s2.rstd;
        }
    }
}

// backward of the above.  dy: grad of the layer output (flows through the FFN residual), dxn: grad of LN2 output.
struct LnGateBwdArgs {
    const float* dy; const float* dxn;
    const float* x1; const float* st1; const float* st2;
    const bf16* O; int ldo;
    const bf16* U; int ldu;
    const bf16* zu; int ldz;       // pre-activation of U (for silu')
    const float *g1, *b1, *g2;
    float* dx1;                    // [T,D] fp32
    bf16* dO; int lddo;            // [T,D]
    bf16* dzu; int lddz;           // [T, ...] grad wrt U pre-activation
    float *dg1, *db1, *dg2, *db2;  // accumulated (atomicAdd)
    int T, D;
    Dropout drop;
};
template <int NP>
__global__ void __launch_bounds__(ROW_THREADS) ln_gate_bwd_kernel(LnGateBwdArgs a) {
    pdl_wait();
    a.drop.resolve();
    __shared__ float red[4][ROW_THREADS / 32][64 * NP];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    float adg1[NP][2], adb1[NP][2], adg2[NP][2], adb2[NP][2];
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 2; ++e) adg1[p][e] = adb1[p][e] = adg2[p][e] = adb2[p][e] = 0.f;
    const float invD = 1.f / (float)a.D;

    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        const float m1 = a.st1[2 * row], r1 = a.st1[2 * row + 1], m2 = a.st2[2 * row], r2 = a.st2[2 * row + 1];
        // every operand of the row is requested up front (one memory round trip instead of two dependent phases)
        float2 xv[NP], dn[NP], dyv[NP];
        uint32_t ovp[NP], uvp[NP], zvp[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int c = 2 * lane + 64 * p;
            xv[p] = *reinterpret_cast<const float2*>(a.x1 + (size_t)row * a.D + c);
            dn[p] = *reinterpret_cast<const float2*>(a.dxn + (size_t)row * a.D + c);
            dyv[p] = *reinterpret_cast<const float2*>(a.dy + (size_t)row * a.D + c);
            ovp[p] = *reinterpret_cast<const uint32_t*>(a.O + (size_t)row * a.ldo + c);
            uvp[p] = *reinterpret_cast<const uint32_t*>(a.U + (size_t)row * a.ldu + c);
            zvp[p] = *reinterpret_cast<const uint32_t*>(a.zu + (size_t)row * a.ldz + c);
        }
        float xh2[NP][2], gg[NP][2], dx1[NP][2];
        float sa = 0.f, sb = 0.f;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            xh2[p][0] = (xv[p].x - m2) * r2; xh2[p][1] = (xv[p].y - m2) * r2;
            adg2[p][0] += dn[p].x * xh2[p][0]; adg2[p][1] += dn[p].y * xh2[p][1];
            adb2[p][0] += dn[p].x; adb2[p][1] += dn[p].y;
            gg[p][0] = dn[p].x * a.g2[c]; gg[p][1] = dn[p].y * a.g2[c + 1];
            sa += gg[p][0] + gg[p][1];
            sb += gg[p][0] * xh2[p][0] + gg[p][1] * xh2[p][1];
        }
        sa = warp_sum(sa) * invD; sb = warp_sum(sb) * invD;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            dx1[p][0] = dyv[p].x + r2 * (gg[p][0] - sa - xh2[p][0] * sb);
            dx1[p][1] = dyv[p].y + r2 * (gg[p][1] - sa - xh2[p][1] * sb);
            *reinterpret_cast<float2*>(a.dx1 + (size_t)row * a.D + c) = make_float2(dx1[p][0], dx1[p][1]);
        }
        // gate + LN1
        float xh1[NP][2], gn[NP][2];
        float ta = 0.f, tb = 0.f;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float2 ov = unpack_bf16(ovp[p]);
            float2 uv = unpack_bf16(uvp[p]);
            float2 zv = unpack_bf16(zvp[p]);
            float o2[2] = {ov.x, ov.y}, u2[2] = {uv.x, uv.y}, z2[2] = {zv.x, zv.y}, dzu[2];
            float dGv[2] = {dx1[p][0], dx1[p][1]};
            a.drop.apply2(dGv[0], dGv[1], row, c);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const float dG = dGv[e];
                xh1[p][e] = (o2[e] - m1) * r1;
                float n = xh1[p][e] * a.g1[c + e] + a.b1[c + e];
                dzu[e] = dG * n * dsiluf(z2[e]);
                float dN = dG * u2[e];
                adg1[p][e] += dN * xh1[p][e];
                adb1[p][e] += dN;
                gn[p][e] = dN * a.g1[c + e];
                ta += gn[p][e];
                tb += gn[p][e] * xh1[p][e];
            }
            *reinterpret_cast<uint32_t*>(a.dzu + (size_t)row * a.lddz + c) = pack_bf16(dzu[0], dzu[1]);
        }
        ta = warp_sum(ta) * invD; tb = warp_sum(tb) * invD;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float d0 = r1 * (gn[p][0] - ta - xh1[p][0] * tb), d1 = r1 * (gn[p][1] - ta - xh1[p][1] * tb);
            *reinterpret_cast<uint32_t*>(a.dO + (size_t)row * a.lddo + c) = pack_bf16(d0, d1);
        }
    }
    // CTA reduction of the four parameter-gradient vectors, then one atomicAdd per column per CTA
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            int c = 2 * lane + 64 * p + e;
            red[0][wib][c] = adg1[p][e]; red[1][wib][c] = adb1[p][e];
            red[2][wib][c] = adg2[p][e]; red[3][wib][c] = adb2[p][e];
        }
    __syncthreads();
    float* outs[4] = {a.dg1, a.db1, a.dg2, a.db2};
    for (int i = threadIdx.x; i < 4 * a.D; i += ROW_THREADS) {
        int which = i / a.D, c = i % a.D;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < ROW_THREADS / 32; ++w) s += red[which][w][c];
        atomicAdd(outs[which] + c, s);
    }
}

// ------------------------------------------------------------------------------------------------ plain LayerNorm fwd / bwd
// y = LN(x) (fp32 in) -> bf16 and/or fp32 out, stats saved.
struct LnFwdArgs {
    const float* x; const float *g, *b;
    bf16* y_bf16; float* y_f32;  // either nullable
    float* st;
    int T, D; float eps;
};
template <int NP>
__global__ void __launch_bounds__(ROW_THREADS) ln_fwd_kernel(LnFwdArgs a) {
    pdl_wait();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        float xv[NP][2];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            float2 f = *reinterpret_cast<const float2*>(a.x + (size_t)row * a.D + 2 * lane + 64 * p);
            xv[p][0] = f.x; xv[p][1] = f.y;
        }
        LnStats s = row_stats<NP>(xv, a.D, a.eps);
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float y0 = (xv[p][0] - s.mean) * s.rstd * a.g[c] + a.b[c];
            float y1 = (xv[p][1] - s.mean) * s.rstd * a.g[c + 1] + a.b[c + 1];
            if (a.y_bf16) *reinterpret_cast<uint32_t*>(a.y_bf16 + (size_t)row * a.D + c) = pack_bf16(y0, y1);
            if (a.y_f32) *reinterpret_cast<float2*>(a.y_f32 + (size_t)row * a.D + c) = make_float2(y0, y1);
        }
        if (lane == 0 && a.st) { a.st[2 * row] = s.mean; a.st[2 * row + 1] = s.rstd; }
    }
}
// dx = (res ? res : 0) + LNbwd(dy) ; dg += , db +=
struct LnBwdArgs {
    const float* dy; const float* x; const float* st; const float* g;
    const float* res;  // nullable, added to dx
    float* dx; float *dg, *db;
    int T, D;
};
template <int NP>
__global__ void __launch_bounds__(ROW_THREADS) ln_bwd_kernel(LnBwdArgs a) {
    pdl_wait();
    __shared__ float red[2][ROW_THREADS / 32][64 * NP];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    float adg[NP][2], adb[NP][2];
#pragma unroll
    for (int p = 0; p < NP; ++p) adg[p][0] = adg[p][1] = adb[p][0] = adb[p][1] = 0.f;
    const float invD = 1.f / (float)a.D;
    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        const float m = a.st[2 * row], r = a.st[2 * row + 1];
        float xh[NP][2], gg[NP][2];
        float sa = 0.f, sb = 0.f;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float2 xv = *reinterpret_cast<const float2*>(a.x + (size_t)row * a.D + c);
            float2 dv = *reinterpret_cast<const float2*>(a.dy + (size_t)row * a.D + c);
            xh[p][0] = (xv.x - m) * r; xh[p][1] = (xv.y - m) * r;
            adg[p][0] += dv.x * xh[p][0]; adg[p][1] += dv.y * xh[p][1];
            adb[p][0] += dv.x; adb[p][1] += dv.y;
            gg[p][0] = dv.x * a.g[c]; gg[p][1] = dv.y * a.g[c + 1];
            sa += gg[p][0] + gg[p][1];
            sb += gg[p][0] * xh[p][0] + gg[p][1] * xh[p][1];
        }
        sa = warp_sum(sa) * invD; sb = warp_sum(sb) * invD;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            int c = 2 * lane + 64 * p;
            float d0 = r * (gg[p][0] - sa - xh[p][0] * sb), d1 = r * (gg[p][1] - sa - xh[p][1] * sb);
            if (a.res) {
                float2 rv = *reinterpret_cast<const float2*>(a.res + (size_t)row * a.D + c);
                d0 += rv.x; d1 += rv.y;
            }
            *reinterpret_cast<float2*>(a.dx + (size_t)row * a.D + c) = make_float2(d0, d1);
        }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            int c = 2 * lane + 64 * p + e;
            red[0][wib][c] = adg[p][e]; red[1][wib][c] = adb[p][e];
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * a.D; i += ROW_THREADS) {
        int which = i / a.D, c = i % a.D;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < ROW_THREADS / 32; ++w) s += red[which][w][c];
        atomicAdd((which ? a.db : a.dg) + c, s);
    }
}

// ------------------------------------------------------------------------------------------------ casts / column sums
// out_bf16[i] = bf16(dropmask(in[i]) * row_scale[row])       (n = T*D elements, D = row length)
__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, size_t n, int D, Dropout drop,
                                     const float* __restrict__ row_scale) {
    pdl_wait();
    drop.resolve();
    // a thread converts 4 neighbouring columns per step; (row, column) advance without divisions inside the loop
    const size_t nq = n / 4, stride = (size_t)gridDim.x * blockDim.x;
    const uint32_t D4 = (uint32_t)D / 4;
    size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // < 2^32 (the grid is capped), as is stride
    uint32_t row = (uint32_t)q / D4, cq = (uint32_t)q % D4;
    const uint32_t srow = (uint32_t)stride / D4, scq = (uint32_t)stride % D4;
    for (; q < nq; q += stride) {
        const size_t i = q * 4;
        float4 v = *reinterpret_cast<const float4*>(in + i);
        const float rs = row_scale ? row_scale[row] : 1.f;
        uint2 o;
        drop.apply2(v.x, v.y, row, cq * 4);
        drop.apply2(v.z, v.w, row, cq * 4 + 2);
        o.x = pack_bf16(v.x * rs, v.y * rs);
        o.y = pack_bf16(v.z * rs, v.w * rs);
        *reinterpret_cast<uint2*>(out + i) = o;
        row += srow;
        cq += scq;
        if (cq >= D4) { cq -= D4; ++row; }
    }
}
// out_bf16[r, c] = bf16(dropmask(in[r, c]))  and  colsum[c] += sum_r out_bf16[r, c]   (the cast of dy and the bias gradient
// of the layer's last linear in one pass).  grid (ceil(D / 128), chunks) ; block 256 = 8 row lanes x 32 threads of 4 columns.
__global__ void __launch_bounds__(256) cast_colsum_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, int T, int D,
                                                                  Dropout drop, float* __restrict__ colsum) {
    pdl_wait();
    drop.resolve();
    __shared__ float red[8][128];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 128 + 4 * tx;
    const int rows_per = (T + gridDim.y - 1) / gridDim.y;
    const int r0 = blockIdx.y * rows_per, r1 = min(T, r0 + rows_per);
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    if (c < D) {
        auto one = [&](int r, float4 v) {
            drop.apply2(v.x, v.y, r, c);
            drop.apply2(v.z, v.w, r, c + 2);
            uint2 o;
            o.x = pack_bf16(v.x, v.y);
            o.y = pack_bf16(v.z, v.w);
            *reinterpret_cast<uint2*>(out + (size_t)r * D + c) = o;
            const float2 a = unpack_bf16(o.x), b = unpack_bf16(o.y);
            s[0] += a.x; s[1] += a.y; s[2] += b.x; s[3] += b.y;
        };
        int r = r0 + ty;
        for (; r + 24 < r1; r += 32) {
            float4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = *reinterpret_cast<const float4*>(in + (size_t)(r + 8 * u) * D + c);
#pragma unroll
            for (int u = 0; u < 4; ++u) one(r + 8 * u, q[u]);
        }
        for (; r < r1; r += 8) one(r, *reinterpret_cast<const float4*>(in + (size_t)r * D + c));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) red[ty][4 * tx + k] = s[k];
    __syncthreads();
    if (threadIdx.x < 128) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
        const int cc = blockIdx.x * 128 + threadIdx.x;
        if (cc < D) atomicAdd(colsum + cc, t);
    }
}
// out[c] += sum_r in[r, c]   in: bf16 [T, ld] (ld % 8 == 0), columns [0, N) ; grid (ceil(N/256), chunks) ;
// block 256 = 32 column groups of 8 (one 16-byte load each) x 8 row lanes, 4 rows in flight per thread
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ in, int T, int N, int ld, float* __restrict__ out) {
    pdl_wait();
    __shared__ float red[8][256];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 256 + 8 * tx;
    const int rows_per = (T + gridDim.y - 1) / gridDim.y;
    const int r0 = blockIdx.y * rows_per, r1 = min(T, r0 + rows_per);
    float s[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = 0.f;
    if (c < N) {
        int r = r0 + ty;
        for (; r + 24 < r1; r += 32) {
            uint4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = *reinterpret_cast<const uint4*>(in + (size_t)(r + 8 * u) * ld + c);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float2 f = unpack_bf16(w[k]);
                    s[2 * k] += f.x; s[2 * k + 1] += f.y;
                }
            }
        }
        for (; r < r1; r += 8) {
            const uint4 q = *reinterpret_cast<const uint4*>(in + (size_t)r * ld + c);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float2 f = unpack_bf16(w[k]);
                s[2 * k] += f.x; s[2 * k + 1] += f.y;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[ty][8 * tx + k] = s[k];
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    const int cc = blockIdx.x * 256 + threadIdx.x;
    if (cc < N) atomicAdd(out + cc, t);
}

// ------------------------------------------------------------------------------------------------ embedding
// x[t,:] = drop(E[ids[t],:] * scale (+ pos[t % L,:]))  -> fp32 ; pad[t] = ids[t]==0   (hstu.py:124-128 ; sasrec.py:100-111)
struct EmbedArgs {
    const long long* ids; const float* E; const float* pos;  // pos nullable [>=L, D]
    float* x; uint8_t* pad;
    int T, L, D; float scale; int mask_pad_rows;  // sasrec: x *= (id != 0)
    Dropout drop;
};
__global__ void __launch_bounds__(ROW_THREADS) embed_fwd_kernel(EmbedArgs a) {
    pdl_wait();
    a.drop.resolve();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        long long id = a.ids[row];
        if (lane == 0 && a.pad) a.pad[row] = id == 0;
        const float* src = a.E + (size_t)id * a.D;
        const float* ps = a.pos ? a.pos + (size_t)(row % a.L) * a.D : nullptr;
        const float keep = (a.mask_pad_rows && id == 0) ? 0.f : 1.f;
        for (int c = lane * 4; c < a.D; c += 128) {
            float4 v = *reinterpret_cast<const float4*>(src + c);
            float e[4] = {v.x * a.scale, v.y * a.scale, v.z * a.scale, v.w * a.scale};
            if (ps) {
                float4 p = *reinterpret_cast<const float4*>(ps + c);
                e[0] += p.x; e[1] += p.y; e[2] += p.z; e[3] += p.w;
            }
            size_t o = (size_t)row * a.D + c;
#pragma unroll
            for (int k = 0; k < 4; k += 2) {
                a.drop.apply2(e[k], e[k + 1], row, c + k);
                e[k] *= keep;
                e[k + 1] *= keep;
            }
            *reinterpret_cast<float4*>(a.x + o) = make_float4(e[0], e[1], e[2], e[3]);
        }
    }
}
// dE[ids[t],:] += scale * dropmask(dx[t,:]) for ids[t] != 0 (padding_idx) ; dpos[t % L,:] += dropmask(dx[t,:])
struct EmbedBwdArgs {
    const long long* ids; const float* dx; float* dE; float* dpos;
    int T, L, D; float scale; int mask_pad_rows;
    Dropout drop;
};
__global__ void __launch_bounds__(ROW_THREADS) embed_bwd_kernel(EmbedBwdArgs a) {
    pdl_wait();
    a.drop.resolve();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = gridDim.x * (ROW_THREADS / 32);
    for (int row = blockIdx.x * (ROW_THREADS / 32) + wib; row < a.T; row += nw) {
        long long id = a.ids[row];
        if (id == 0 && (a.mask_pad_rows || !a.dpos)) continue;
        // four columns per lane and one 16-byte vector reduction per destination (D % 4 == 0, rows 16-byte aligned)
        for (int c = 4 * lane; c < a.D; c += 128) {
            float4 v = *reinterpret_cast<const float4*>(a.dx + (size_t)row * a.D + c);
            a.drop.apply2(v.x, v.y, row, c);
            a.drop.apply2(v.z, v.w, row, c + 2);
            if (id != 0) red_add_v4(a.dE + (size_t)id * a.D + c, v.x * a.scale, v.y * a.scale, v.z * a.scale, v.w * a.scale);
            if (a.dpos && !(a.mask_pad_rows && id == 0)) red_add_v4(a.dpos + (size_t)(row % a.L) * a.D + c, v.x, v.y, v.z, v.w);
        }
    }
}

// ------------------------------------------------------------------------------------------------ fused CE: target count
// count = #(targets != 0)  -> inv_count (0 if none); loss <- 0, or NaN when no target is valid (F.cross_entropy's 0 / 0 mean,
// hstu.py:141-146; the gradients of such a batch are zero here, NaN in the reference)
__global__ void ce_count_kernel(const long long* __restrict__ tg, int T, float* __restrict__ inv_count, float* __restrict__ loss) {
    pdl_wait();
    __shared__ int red[32];
    int c = 0;
    // 16-byte loads, deeply unrolled: all loads of a thread are in flight together (this single-CTA kernel is one DRAM
    // round trip long instead of one per target)
    const longlong2* tg2 = reinterpret_cast<const longlong2*>(tg);
    const int T2 = ((reinterpret_cast<uintptr_t>(tg) & 15) == 0) ? T / 2 : 0;
#pragma unroll 16
    for (int i = threadIdx.x; i < T2; i += blockDim.x) {
        const longlong2 v = tg2[i];
        c += (v.x != 0) + (v.y != 0);
    }
    for (int i = 2 * T2 + threadIdx.x; i < T; i += blockDim.x) c += tg[i] != 0;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
        *inv_count = s > 0 ? 1.f / (float)s : 0.f;
        *loss = s > 0 ? 0.f : __int_as_float(0x7fc00000);
    }
}

// ------------------------------------------------------------------------------------------------ fused Adam (torch.optim.Adam semantics)
// state[0] = step (as float), state[1] = 1 - beta1^step, state[2] = 1 - beta2^step ; ticked on device so a CUDA graph replays correctly.
// The powers are taken in double: under --use_fast_math powf is exp2(step * log2(beta)) on the approximate MUFU units, and the
// cancellation in 1 - beta2^step (beta2 = 0.999) magnified their error to 6e-5 of the bias correction on a B200 - every update of the
// first steps was off by the same factor.  Double arithmetic is not affected by fast math.
__global__ void adam_tick_kernel(float* state, float beta1, float beta2) {
    pdl_wait();
    float step = state[0] + 1.f;
    state[0] = step;
    state[1] = (float)(1.0 - pow((double)beta1, (double)step));
    state[2] = (float)(1.0 - pow((double)beta2, (double)step));
}
struct AdamArgs {
    float* p; float* g; float* m; float* v; bf16* p_bf16;  // p_bf16 nullable
    size_t n;
    const float* state;
    float lr, beta1, beta2, eps, weight_decay, grad_scale;
    int zero_grad;
};
__global__ void adam_step_kernel(AdamArgs a) {
    pdl_wait();
    const float bc1 = a.state[1], bc2 = a.state[2];
    const float step_size = a.lr / bc1;
    const float inv_sqrt_bc2 = rsqrtf(bc2);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < a.n; i += stride) {
        float p = a.p[i], g = a.g[i] * a.grad_scale;
        if (a.weight_decay != 0.f) g += a.weight_decay * p;
        float m = a.beta1 * a.m[i] + (1.f - a.beta1) * g;
        float v = a.beta2 * a.v[i] + (1.f - a.beta2) * g * g;
        a.m[i] = m;
        a.v[i] = v;
        float denom = sqrtf(v) * inv_sqrt_bc2 + a.eps;
        p -= step_size * (m / denom);
        a.p[i] = p;
        if (a.p_bf16) a.p_bf16[i] = __float2bfloat16(p);
        if (a.zero_grad) a.g[i] = 0.f;
    }
}
__global__ void cast_flat_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, size_t n) {
    pdl_wait();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = __float2bfloat16(in[i]);
}


// ------------------------------------------------------------------------------------------------ split-bf16 operands
// fp32-accurate GEMM on the bf16 tensor path: x = hi + mid + lo with three bf16 terms (24 mantissa bits together); the product
// of two such numbers keeps the six terms of weight >= 2^-16 (hi*hi, hi*mid, mid*hi, hi*lo, lo*hi, mid*mid).  Laying the terms
// out along K,   A' = [hi | hi | mid | hi | lo | mid]   B' = [hi | mid | hi | lo | hi | mid]   (K' = 6 K),
// turns the sum of the six partial GEMMs into ONE ordinary GEMM with fp32 accumulation in TMEM.
// out [rows, 6 K] bf16 ; operand 0 = A layout, 1 = B layout.
__global__ void __launch_bounds__(256) split3_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, size_t rows, int K, int operand) {
    pdl_wait();
    const size_t n = rows * (size_t)K;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / K;
        const int k = (int)(e % K);
        const float x = in[e];
        const bf16 hi = __float2bfloat16_rn(x);
        const float r1 = x - __bfloat162float(hi);
        const bf16 mid = __float2bfloat16_rn(r1);
        const bf16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
        bf16* o = out + r * (size_t)(6 * K) + k;
        if (operand == 0) { o[0] = hi; o[K] = hi; o[2 * K] = mid; o[3 * K] = hi; o[4 * K] = lo; o[5 * K] = mid; }
        else              { o[0] = hi; o[K] = mid; o[2 * K] = hi; o[3 * K] = lo; o[4 * K] = hi; o[5 * K] = mid; }
    }
}


// ------------------------------------------------------------------------------------------------ leave-one-out metrics
// Replaces the per-sample Python loop of genrec/trainers/hstu_trainer.py:55-81 (`logits[:, 0] = -inf`, top-k, `.item()` per
// sample): the rank of the held-out target among classes 1..C-1 is counted directly - rank = 1 + #{j >= 1 : logit_j > logit_t or
// (logit_j == logit_t and j < t)} (torch.topk's order on ties: lower index first) - and Recall@k / NDCG@k for k in {1, 5, 10}
// are ACCUMULATED on the device:  out[0..2] += hit@{1,5,10}, out[3..5] += ndcg@{1,5,10}.  One CTA per sample; targets of 0
// (padding) contribute nothing.  ranks (nullable) receives the per-sample rank (0 for skipped samples).
__global__ void __launch_bounds__(256) eval_rank_kernel(const float* __restrict__ logits, int C, const long long* __restrict__ targets,
                                                       float* __restrict__ out, int* __restrict__ ranks) {
    pdl_wait();
    __shared__ int red[8];
    const int b = blockIdx.x;
    const long long t = targets[b];
    if (t <= 0 || t >= C) {
        if (threadIdx.x == 0 && ranks) ranks[b] = 0;
        return;
    }
    const float* row = logits + (size_t)b * C;
    const float lt = row[t];
    int c = 0;
    for (int j = 1 + threadIdx.x; j < C; j += 256) {
        const float v = row[j];
        c += (v > lt) || (v == lt && j < (int)t);
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int rank = 1;
        for (int w = 0; w < 8; ++w) rank += red[w];
        if (ranks) ranks[b] = rank;
        const float nd = 1.f / log2f((float)rank + 1.f);
        if (rank <= 1) { atomicAdd(out + 0, 1.f); atomicAdd(out + 3, nd); }
        if (rank <= 5) { atomicAdd(out + 1, 1.f); atomicAdd(out + 4, nd); }
        if (rank <= 10) { atomicAdd(out + 2, 1.f); atomicAdd(out + 5, nd); }
    }
}


// ------------------------------------------------------------------------------------------------ jagged -> left-padded batch
// Device-side hstu_collate_fn (genrec/data/amazon_hstu.py:137-173): user b's history is items[offsets[b] .. offsets[b+1]) (time
// order) with the held-out target targets[b].  With n = min(len_b, L) kept (the LAST n events) and pad = L - n:
//   input_ids[b, p]  = p < pad ? 0 : hist[p - pad]          timestamps[b, p] = p < pad ? 0 : ts[p - pad]
//   targets[b, p]    = p + 1 < pad ? 0 : (p + 1 - pad < n ? hist[p + 1 - pad] : target_b)      (the sequence shifted by one)
// One thread per output position; stamps / out_ts may be null (SASRec: genrec/data/amazon_sasrec.py:125-161).
__global__ void __launch_bounds__(256) collate_jagged_kernel(const long long* __restrict__ items, const long long* __restrict__ stamps,
                                                            const long long* __restrict__ offsets, const long long* __restrict__ targets, int B,
                                                            int L, long long* __restrict__ out_ids, long long* __restrict__ out_tg,
                                                            long long* __restrict__ out_ts) {
    pdl_wait();
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)B * L) return;
    const int b = (int)(e / L), p = (int)(e % L);
    const long long lo = offsets[b], hi = offsets[b + 1];
    const long long len = hi - lo;
    const int n = (int)(len < L ? len : L);
    const int pad = L - n;
    const long long* h = items + (hi - n);            // the last n events
    out_ids[e] = p < pad ? 0 : h[p - pad];
    out_tg[e] = p + 1 < pad ? 0 : (p + 1 - pad < n ? h[p + 1 - pad] : targets[b]);
    if (out_ts != nullptr) out_ts[e] = (p < pad || stamps == nullptr) ? 0 : stamps[(hi - n) + (p - pad)];
}


// ------------------------------------------------------------------------------------------------ fused CE: normalisation pass
// The fused CE kernel (tc_ce.cuh) leaves G' = exp(s - max) / count unnormalised and reports, per row, the sum of G' over each
// class half, the row max and the target logit.  With rs = 1 / sum_c exp(s_c - max) (so that G = G' rs is the softmax / count):
//   loss    += (max + log sum exp - logit[target]) / count
//   dxf      = dxf' rs - E[target] / count                 (dxf' = G' E from the CE kernel or the GEMM)
//   xs       = bf16(x rs)                                   -> a dE GEMM over the stored G' computes G'^T xs = G^T x, or
//   col_shift = log2e * logsumexp - log2(1 / count)         -> the class-stationary pass (tc_ce.cuh CE_ACCUM_T) recomputes G from it
//   dE[target] -= x / count                                 (the one-hot term of dE, a 16-byte-vector scatter)
// One warp per token row; rows with target 0 (ignore_index) get rs = 0 and contribute nothing.
struct CeFinishArgs {
    const float* row_sums;       // [2][T]
    const float2* row_stats;     // [T] {exponent shift (the row max, or the one-sweep kernel's estimate), target logit}
    const float* tl_parts;       // nullable [2][T]: the target logit as two per-half partials (one-sweep kernel) instead of row_stats.y
    const long long* targets;    // [T]
    const float* inv_count;
    const bf16* xf;              // [T, D]
    const bf16* table;           // [C, D] bf16 mirror of the tied embedding table
    float* dxf;                  // [T, D] in: G' E, out: d loss / d xf   (nullable: loss only)
    bf16* xs;                    // [T, D] out (nullable)
    float* col_shift;            // [ceil(T / 128) * 128] out (nullable); +inf for ignored rows and the padding
    float* dtable;               // [C, D] += (nullable)
    float* loss;                 // += (zeroed by ce_count_kernel)
    int T, D;
};
__global__ void __launch_bounds__(ROW_THREADS) ce_finish_kernel(CeFinishArgs a) {
    pdl_wait();
    __shared__ float s_loss[ROW_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wpb = ROW_THREADS / 32;
    const float ic = *a.inv_count;
    float lsum = 0.f;
    for (int row = blockIdx.x * wpb + warp; row < a.T; row += gridDim.x * wpb) {
        const int t = (int)a.targets[row];
        const float icr = t != 0 ? ic : 0.f;
        const float gs = a.row_sums[row] + a.row_sums[(size_t)a.T + row];        // = sum_c exp(s_c - max) * icr
        const float rs = (icr > 0.f && gs > 0.f) ? icr / gs : 0.f;                // 1 / sum_c exp(s_c - max)
        if (lane == 0) {
            const float2 st = a.row_stats[row];
            const float tlog = a.tl_parts ? a.tl_parts[row] + a.tl_parts[(size_t)a.T + row] : st.y;
            const bool live = icr > 0.f && gs > 0.f;
            if (live) lsum += (st.x + __logf(gs / icr) - tlog) * icr;
            if (a.col_shift) a.col_shift[row] = live ? st.x * 1.4426950408889634f + __log2f(gs / icr) - __log2f(icr) : INFINITY;
        }
        const bf16* x = a.xf + (size_t)row * a.D;
        const bf16* e = a.table + (size_t)t * a.D;
        for (int c = lane * 4; c < a.D; c += 128) {
            const uint2 xu = *reinterpret_cast<const uint2*>(x + c);
            const float2 x0 = unpack_bf16(xu.x), x1 = unpack_bf16(xu.y);
            if (a.xs) {
                uint2 o;
                o.x = pack_bf16(x0.x * rs, x0.y * rs); o.y = pack_bf16(x1.x * rs, x1.y * rs);
                *reinterpret_cast<uint2*>(a.xs + (size_t)row * a.D + c) = o;
            }
            if (a.dxf) {
                float4 d = *reinterpret_cast<float4*>(a.dxf + (size_t)row * a.D + c);
                const uint2 eu = *reinterpret_cast<const uint2*>(e + c);
                const float2 e0 = unpack_bf16(eu.x), e1 = unpack_bf16(eu.y);
                d.x = d.x * rs - icr * e0.x; d.y = d.y * rs - icr * e0.y; d.z = d.z * rs - icr * e1.x; d.w = d.w * rs - icr * e1.y;
                *reinterpret_cast<float4*>(a.dxf + (size_t)row * a.D + c) = d;
            }
            if (a.dtable && icr > 0.f) red_add_v4(a.dtable + (size_t)t * a.D + c, -icr * x0.x, -icr * x0.y, -icr * x1.x, -icr * x1.y);
        }
    }
    if (a.col_shift && blockIdx.x == 0)
        for (int i = a.T + threadIdx.x; i < ((a.T + 127) / 128) * 128; i += ROW_THREADS) a.col_shift[i] = INFINITY;
    if (lane == 0) s_loss[warp] = lsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int w = 0; w < wpb; ++w) tot += s_loss[w];
        if (tot != 0.f) atomicAdd(a.loss, tot);
    }
}

}  // namespace grb
