// Backward passes of the HBM-bound kernels (instance norm, ConvLSTM gates, CDNA, compositing, dense,
// small LSTM, pooling) + losses + fused TF-Adam.  Same layout conventions as elementwise.cu.
// Parameter gradients are accumulated with atomics into zero-initialised flat gradient buffers
// (BPTT sums over timesteps, savp_model.py unrolls share variables).
#include <cstdint>

#include "common.h"
#include "ptx.cuh"

namespace vp {

__device__ __forceinline__ float sigm(float v) { return 1.f / (1.f + __expf(-v)); }
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int kN>
__device__ __forceinline__ void bsum(float* vals, float* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < kN; ++i) vals[i] = wsum(vals[i]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < kN; ++i) scratch[i * 32 + warp] = vals[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < kN; ++i) {
    float v = (lane < nw) ? scratch[i * 32 + lane] : 0.f;
    vals[i] = wsum(v);
  }
}
__device__ __forceinline__ float act_grad(float yp, int act, float alpha) {  // d act(yp) / d yp
  switch (act) {
    case VP_ACT_RELU: return yp > 0.f ? 1.f : 0.f;
    case VP_ACT_LRELU: return yp > 0.f ? 1.f : alpha;
    default: return 1.f;
  }
}

struct SrcList {  // up to 4 gradient sources that are summed (each a channel slice with its own stride)
  const float* ptr[4];
  int stride[4];
  int count;
};

// ------------------------------------------------------------------------------------------------
// instance norm (+act) backward.  x: pre-norm input (dense, stride xs); dy: sum of `srcs`.
// dx = r*(dxh - mean(dxh) - xh*mean(dxh*xh)),  dxh = dyp*gamma,  dyp = dy*act'(gamma*xh+beta)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) inorm_act_bwd_kernel(const float* __restrict__ x, int xs, SrcList srcs,
                                                            float* __restrict__ dx, int dxs, int P, int C,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ stats, int act, float alpha,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta, int staged) {
  extern __shared__ float4 sbuf[];   // staged: [P] x values, then [P] summed upstream gradients
  __shared__ float scratch[8 * 32];
  const int n = blockIdx.y, c0 = blockIdx.x * 4;
  const float* xp = x + static_cast<long long>(n) * P * xs + c0;
  float m[4], r[4], g[4], b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = stats[(static_cast<long long>(n) * C + c0 + i) * 2];
    r[i] = stats[(static_cast<long long>(n) * C + c0 + i) * 2 + 1];
    g[i] = gamma[c0 + i];
    b[i] = beta[c0 + i];
  }
  auto load_dy = [&](int p) {
    float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < srcs.count; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(srcs.ptr[s] + (static_cast<long long>(n) * P + p) * srcs.stride[s] + c0);
      d.x += v.x; d.y += v.y; d.z += v.z; d.w += v.w;
    }
    return d;
  };
  float s[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0.f;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const float4 xv = *reinterpret_cast<const float4*>(xp + static_cast<long long>(p) * xs);
    const float4 dy = load_dy(p);
    if (staged) { sbuf[p] = xv; sbuf[P + p] = dy; }
    const float xh[4] = {(xv.x - m[0]) * r[0], (xv.y - m[1]) * r[1], (xv.z - m[2]) * r[2], (xv.w - m[3]) * r[3]};
    const float dv[4] = {dy.x, dy.y, dy.z, dy.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float dyp = dv[i] * act_grad(g[i] * xh[i] + b[i], act, alpha);
      s[i] += dyp;
      s[4 + i] += dyp * xh[i];
    }
  }
  bsum<8>(s, scratch);
  if (threadIdx.x < 4) {
    atomicAdd(dbeta + c0 + threadIdx.x, s[threadIdx.x]);
    atomicAdd(dgamma + c0 + threadIdx.x, s[4 + threadIdx.x]);
  }
  const float inv = 1.f / P;
  float* dp = dx + static_cast<long long>(n) * P * dxs + c0;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const float4 xv = staged ? sbuf[p] : *reinterpret_cast<const float4*>(xp + static_cast<long long>(p) * xs);
    const float4 dy = staged ? sbuf[P + p] : load_dy(p);
    const float xh[4] = {(xv.x - m[0]) * r[0], (xv.y - m[1]) * r[1], (xv.z - m[2]) * r[2], (xv.w - m[3]) * r[3]};
    const float dv[4] = {dy.x, dy.y, dy.z, dy.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float dyp = dv[i] * act_grad(g[i] * xh[i] + b[i], act, alpha);
      // dxh = dyp*g ; mean(dxh) = g*s[i]/P ; mean(dxh*xh) = g*s[4+i]/P
      o[i] = r[i] * g[i] * (dyp - s[i] * inv - xh[i] * s[4 + i] * inv);
    }
    *reinterpret_cast<float4*>(dp + static_cast<long long>(p) * dxs) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// ConvLSTM gates backward (see lstm_gates_fwd_kernel).  One CTA per (sample, 4 state channels).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) lstm_gates_bwd_kernel(
    const float* __restrict__ pre, int P, int F, const float* __restrict__ c_prev, const float* __restrict__ g1,
    const float* __restrict__ b1, const float* __restrict__ g2, const float* __restrict__ b2,
    const float* __restrict__ stats1, const float* __restrict__ stats2, float forget_bias, SrcList dh_srcs,
    const float* __restrict__ dc_next, float* __restrict__ dpre, float* __restrict__ dc_prev, float* __restrict__ dg1,
    float* __restrict__ db1, float* __restrict__ dg2, float* __restrict__ db2) {
  extern __shared__ float sm[];  // [16][P] gate grads, [4][P] dcn, [4][P] chat, [16][P] staged pre-activations
  __shared__ float scratch[32 * 32];
  float4* sdg = reinterpret_cast<float4*>(sm);  // [4 gates][P]
  float4* sdc = sdg + 4 * P;
  float4* sch = sdc + P;
  float4* spre = sch + P;                       // [4 gates][P]: the conv output is read from HBM/L2 exactly once
  const int n = blockIdx.y, c0 = blockIdx.x * 4;
  const float inv = 1.f / P;
  float ga[16], be[16], m1[16], r1[16];
#pragma unroll
  for (int g = 0; g < 4; ++g)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int ch = g * F + c0 + k;
      m1[4 * g + k] = stats1[(static_cast<long long>(n) * 4 * F + ch) * 2];
      r1[4 * g + k] = stats1[(static_cast<long long>(n) * 4 * F + ch) * 2 + 1];
      ga[4 * g + k] = g1[ch];
      be[4 * g + k] = b1[ch];
    }
  float m2[4], r2[4], cg[4], cb[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    m2[k] = stats2[(static_cast<long long>(n) * F + c0 + k) * 2];
    r2[k] = stats2[(static_cast<long long>(n) * F + c0 + k) * 2 + 1];
    cg[k] = g2[c0 + k];
    cb[k] = b2[c0 + k];
  }
  const float* pp = pre + static_cast<long long>(n) * P * 4 * F;
  const float* cp = c_prev + static_cast<long long>(n) * P * F + c0;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
      spre[g * P + p] = *reinterpret_cast<const float4*>(pp + static_cast<long long>(p) * 4 * F + g * F + c0);
  }
  __syncthreads();
  auto gate = [&](int p, int g, float* out) {  // normalised + affine gate values of 4 channels
    const float4 v = spre[g * P + p];
    out[0] = (v.x - m1[4 * g]) * r1[4 * g] * ga[4 * g] + be[4 * g];
    out[1] = (v.y - m1[4 * g + 1]) * r1[4 * g + 1] * ga[4 * g + 1] + be[4 * g + 1];
    out[2] = (v.z - m1[4 * g + 2]) * r1[4 * g + 2] * ga[4 * g + 2] + be[4 * g + 2];
    out[3] = (v.w - m1[4 * g + 3]) * r1[4 * g + 3] * ga[4 * g + 3] + be[4 * g + 3];
  };
  // ---- pass A: dcn, chat; sums for the state norm
  float sA[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sA[i] = 0.f;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    float gi[4], gj[4], gf[4], go[4];
    gate(p, 0, gi); gate(p, 1, gj); gate(p, 2, gf); gate(p, 3, go);
    const float4 c4 = *reinterpret_cast<const float4*>(cp + static_cast<long long>(p) * F);
    const float cpv[4] = {c4.x, c4.y, c4.z, c4.w};
    float dh[4] = {0.f, 0.f, 0.f, 0.f};
    for (int s = 0; s < dh_srcs.count; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(dh_srcs.ptr[s] + (static_cast<long long>(n) * P + p) * dh_srcs.stride[s] + c0);
      dh[0] += v.x; dh[1] += v.y; dh[2] += v.z; dh[3] += v.w;
    }
    float4 dcn4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (dc_next) dcn4 = *reinterpret_cast<const float4*>(dc_next + (static_cast<long long>(n) * P + p) * F + c0);
    const float dcx[4] = {dcn4.x, dcn4.y, dcn4.z, dcn4.w};
    float dcn[4], chat[4], dgo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float cpre = cpv[k] * sigm(gf[k] + forget_bias) + sigm(gi[k]) * tanhf(gj[k]);
      chat[k] = (cpre - m2[k]) * r2[k];
      const float cn = chat[k] * cg[k] + cb[k];
      const float th = tanhf(cn), so = sigm(go[k]);
      dgo[k] = dh[k] * th * so * (1.f - so);
      dcn[k] = dh[k] * so * (1.f - th * th) + dcx[k];
      sA[k] += dcn[k];
      sA[4 + k] += dcn[k] * chat[k];
    }
    sdc[p] = make_float4(dcn[0], dcn[1], dcn[2], dcn[3]);
    sch[p] = make_float4(chat[0], chat[1], chat[2], chat[3]);
    sdg[3 * P + p] = make_float4(dgo[0], dgo[1], dgo[2], dgo[3]);
  }
  bsum<8>(sA, scratch);
  if (threadIdx.x < 4) {
    atomicAdd(db2 + c0 + threadIdx.x, sA[threadIdx.x]);
    atomicAdd(dg2 + c0 + threadIdx.x, sA[4 + threadIdx.x]);
  }
  // ---- pass B: dc' -> gate grads (w.r.t. normalised+affine gates); sums for the gate norm
  float sB[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) sB[i] = 0.f;
  float* dcp = dc_prev + static_cast<long long>(n) * P * F + c0;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    float gi[4], gj[4], gf[4];
    gate(p, 0, gi); gate(p, 1, gj); gate(p, 2, gf);
    const float4 c4 = *reinterpret_cast<const float4*>(cp + static_cast<long long>(p) * F);
    const float cpv[4] = {c4.x, c4.y, c4.z, c4.w};
    const float4 dcn4 = sdc[p], ch4 = sch[p], dgo4 = sdg[3 * P + p];
    const float dcn[4] = {dcn4.x, dcn4.y, dcn4.z, dcn4.w}, chat[4] = {ch4.x, ch4.y, ch4.z, ch4.w};
    const float dgo[4] = {dgo4.x, dgo4.y, dgo4.z, dgo4.w};
    float di[4], dj[4], df[4], dcpv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float dcpre = r2[k] * cg[k] * (dcn[k] - sA[k] * inv - chat[k] * sA[4 + k] * inv);
      const float si = sigm(gi[k]), tj = tanhf(gj[k]), sf = sigm(gf[k] + forget_bias);
      di[k] = dcpre * tj * si * (1.f - si);
      dj[k] = dcpre * si * (1.f - tj * tj);
      df[k] = dcpre * cpv[k] * sf * (1.f - sf);
      dcpv[k] = dcpre * sf;
    }
    *reinterpret_cast<float4*>(dcp + static_cast<long long>(p) * F) = make_float4(dcpv[0], dcpv[1], dcpv[2], dcpv[3]);
    sdg[p] = make_float4(di[0], di[1], di[2], di[3]);
    sdg[P + p] = make_float4(dj[0], dj[1], dj[2], dj[3]);
    sdg[2 * P + p] = make_float4(df[0], df[1], df[2], df[3]);
    const float* dall[4] = {di, dj, df, dgo};
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 v = spre[g * P + p];
      const float xv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float xh = (xv[k] - m1[4 * g + k]) * r1[4 * g + k];
        sB[4 * g + k] += dall[g][k];
        sB[16 + 4 * g + k] += dall[g][k] * xh;
      }
    }
  }
  bsum<32>(sB, scratch);
  if (threadIdx.x < 16) {
    const int g = threadIdx.x >> 2, k = threadIdx.x & 3;
    atomicAdd(db1 + g * F + c0 + k, sB[threadIdx.x]);
    atomicAdd(dg1 + g * F + c0 + k, sB[16 + threadIdx.x]);
  }
  // ---- pass C: gate-norm backward -> dpre
  float* dpp = dpre + static_cast<long long>(n) * P * 4 * F;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 v = spre[g * P + p];
      const float4 d4 = sdg[g * P + p];
      const float xv[4] = {v.x, v.y, v.z, v.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w};
      float o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float xh = (xv[k] - m1[4 * g + k]) * r1[4 * g + k];
        o[k] = r1[4 * g + k] * ga[4 * g + k] * (dv[k] - sB[4 * g + k] * inv - xh * sB[16 + 4 * g + k] * inv);
      }
      *reinterpret_cast<float4*>(dpp + static_cast<long long>(p) * 4 * F + g * F + c0) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// compositing backward: dlogit_l = m_l*(g_l - sum_k m_k g_k), g_l = <dgen, layer_l>; dlayer_l = m_l*dgen
// ------------------------------------------------------------------------------------------------
__global__ void composite_bwd_kernel(const float4* __restrict__ dgen, const float* __restrict__ masks, int ms,
                                     const float* __restrict__ layers, int ls, float* __restrict__ dlogits, int dls,
                                     float* __restrict__ dlayers, int dlays, long long total, int L) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const float4 dg = dgen[idx];
  float m[8], g[8];
  float dot = 0.f;
  for (int l = 0; l < L; ++l) {
    m[l] = masks[idx * ms + l];
    const float4 v = *reinterpret_cast<const float4*>(layers + idx * ls + 4 * l);
    g[l] = dg.x * v.x + dg.y * v.y + dg.z * v.z + dg.w * v.w;
    dot += m[l] * g[l];
    *reinterpret_cast<float4*>(dlayers + idx * dlays + 4 * l) = make_float4(m[l] * dg.x, m[l] * dg.y, m[l] * dg.z, m[l] * dg.w);
  }
  for (int l = 0; l < L; ++l) dlogits[idx * dls + l] = m[l] * (g[l] - dot);
  for (int l = L; l < dls && l < 8; ++l) dlogits[idx * dls + l] = 0.f;
}

__device__ __forceinline__ int reflect_i(int i, int n) {
  if (i < 0) i = -i - 1;
  if (i >= n) i = 2 * n - 1 - i;
  return i;
}
// CDNA apply backward.  dT_k = dA[.., 4k] + dB[.., 4k] (two gradient sources: compositor + masks conv).
//  dimage += scatter_k,tap K[tap][k]*dT_k  (+ dprev slot NK)      dkern[n][tap][k] += <dT_k, img[reflect(.+tap)]>
__global__ void __launch_bounds__(256) cdna_apply_bwd_kernel(const float4* __restrict__ image, const float* __restrict__ kern,
                                                             const float* __restrict__ dA, int das,
                                                             const float* __restrict__ dB, int dbs,
                                                             float* __restrict__ dimage, float* __restrict__ dkern, int N,
                                                             int H, int W, int KH, int KW, int NK) {
  extern __shared__ float sk[];  // [KK*NK] kernels, then [KK*NK] dkern partials
  const int n = blockIdx.y;
  const int KK = KH * KW;
  float* sdk = sk + KK * NK;
  for (int i = threadIdx.x; i < KK * NK; i += blockDim.x) {
    sk[i] = kern[static_cast<long long>(n) * KK * NK + i];
    sdk[i] = 0.f;
  }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = p < H * W;
  const int y = valid ? p / W : 0, x = valid ? p % W : 0;
  const float4* img = image + static_cast<long long>(n) * H * W;
  float* dimg = dimage + static_cast<long long>(n) * H * W * 4;
  float4 dT[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    dT[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid && k < NK) {
      const long long o = (static_cast<long long>(n) * H * W + p);
      const float4 a = *reinterpret_cast<const float4*>(dA + o * das + 4 * k);
      const float4 b = *reinterpret_cast<const float4*>(dB + o * dbs + 4 * k);
      dT[k] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
  }
  if (valid) {  // prev-image background layer (slot NK) passes its gradient straight to the image
    const long long o = (static_cast<long long>(n) * H * W + p);
    const float4 a = *reinterpret_cast<const float4*>(dA + o * das + 4 * NK);
    const float4 b = *reinterpret_cast<const float4*>(dB + o * dbs + 4 * NK);
    atomicAdd(dimg + p * 4 + 0, a.x + b.x); atomicAdd(dimg + p * 4 + 1, a.y + b.y);
    atomicAdd(dimg + p * 4 + 2, a.z + b.z);
  }
  const int ph = (KH - 1) / 2, pw = (KW - 1) / 2;
  const int lane = threadIdx.x & 31;
  for (int i = 0; i < KH; ++i) {
    const int yy = reflect_i(y + i - ph, H);
    for (int j = 0; j < KW; ++j) {
      const int xx = reflect_i(x + j - pw, W);
      const int q = yy * W + xx;
      const float4 v = valid ? img[q] : make_float4(0.f, 0.f, 0.f, 0.f);
      const float* kk = sk + (i * KW + j) * NK;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < NK) {
          acc.x += kk[k] * dT[k].x; acc.y += kk[k] * dT[k].y; acc.z += kk[k] * dT[k].z;
          float d = dT[k].x * v.x + dT[k].y * v.y + dT[k].z * v.z + dT[k].w * v.w;
          d = wsum(d);
          if (lane == 0) atomicAdd(&sdk[(i * KW + j) * NK + k], d);
        }
      }
      if (valid) {
        atomicAdd(dimg + q * 4 + 0, acc.x); atomicAdd(dimg + q * 4 + 1, acc.y); atomicAdd(dimg + q * 4 + 2, acc.z);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < KK * NK; i += blockDim.x) atomicAdd(dkern + static_cast<long long>(n) * KK * NK + i, sdk[i]);
}

// cdna kernel normalisation backward (see cdna_kernel_norm_kernel): raw/out/dout/draw [B][KK][NK]
__global__ void cdna_kernel_norm_bwd_kernel(const float* __restrict__ raw, const float* __restrict__ out,
                                            const float* __restrict__ dout, float* __restrict__ draw, int B, int KH, int KW,
                                            int NK) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * NK) return;
  const int b = idx / NK, k = idx % NK;
  const int KK = KH * KW;
  const long long base = static_cast<long long>(b) * KK * NK + k;
  const int ci = KH / 2, cj = KW / 2;
  float s = 0.f, dot = 0.f;
  for (int t = 0; t < KK; ++t) {
    float idv = 0.f;
    const int i = t / KW, j = t % KW;
    const bool in_i = (KH % 2) ? (i == ci) : (i == ci - 1 || i == ci);
    const bool in_j = (KW % 2) ? (j == cj) : (j == cj - 1 || j == cj);
    if (in_i && in_j) idv = 1.f / (((KH % 2) ? 1 : 2) * ((KW % 2) ? 1 : 2));
    s += fmaxf(raw[base + static_cast<long long>(t) * NK] + idv - 1e-12f, 0.f) + 1e-12f;
    dot += dout[base + static_cast<long long>(t) * NK] * out[base + static_cast<long long>(t) * NK];
  }
  for (int t = 0; t < KK; ++t) {
    float idv = 0.f;
    const int i = t / KW, j = t % KW;
    const bool in_i = (KH % 2) ? (i == ci) : (i == ci - 1 || i == ci);
    const bool in_j = (KW % 2) ? (j == cj) : (j == cj - 1 || j == cj);
    if (in_i && in_j) idv = 1.f / (((KH % 2) ? 1 : 2) * ((KW % 2) ? 1 : 2));
    const float pre = raw[base + static_cast<long long>(t) * NK] + idv - 1e-12f;
    const float dv = (dout[base + static_cast<long long>(t) * NK] - dot) / s;
    draw[base + static_cast<long long>(t) * NK] = pre > 0.f ? dv : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------
// dense backward: dx[b][k] (+)= sum_j dy[b][j] W[k][j]/scale ; dW[k][j] += sum_b x[b][k] dy[b][j]/scale ;
// db[j] += sum_b dy[b][j]
// ------------------------------------------------------------------------------------------------
__global__ void dense_bwd_dx_kernel(const float* __restrict__ dy, int dys, const float* __restrict__ W,
                                    const float* __restrict__ inv_scale, float* __restrict__ dx, int dxs, int B, int K, int J,
                                    int accumulate) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(B) * K) return;
  const int k = static_cast<int>(idx % K), b = static_cast<int>(idx / K);
  float s = 0.f;
  for (int j = 0; j < J; ++j) s += dy[static_cast<long long>(b) * dys + j] * W[static_cast<long long>(k) * J + j];
  if (inv_scale) s /= __ldg(inv_scale);
  float* o = dx + static_cast<long long>(b) * dxs + k;
  *o = accumulate ? *o + s : s;
}
__global__ void dense_bwd_dw_kernel(const float* __restrict__ x, int xs, const float* __restrict__ dy, int dys,
                                    const float* __restrict__ inv_scale, float* __restrict__ dW, float* __restrict__ db,
                                    int B, int K, int J) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(K) * J) return;
  const int j = static_cast<int>(idx % J), k = static_cast<int>(idx / J);
  float s = 0.f, sb = 0.f;
  for (int b = 0; b < B; ++b) {
    const float d = dy[static_cast<long long>(b) * dys + j];
    s += x[static_cast<long long>(b) * xs + k] * d;
    sb += d;
  }
  if (inv_scale) s /= __ldg(inv_scale);
  dW[idx] += s;
  if (db && k == 0) db[j] += sb;
}


// Tiled versions for the wide CDNA-kernel dense layer (K = 8192 flattened lstm_h2 features -> J = 100, B = 2*batch rows),
// Both keep a 4 x 4 register tile per thread fed by two 16-byte shared loads per reduction step.
// dx: one CTA per 64 k; W tile (transposed, k contiguous) and dy (transposed, b contiguous) staged in shared memory.
// dW: one CTA per 32 k over ALL rows (the time-batched call passes B = (T-1)*NB rows), rows staged 32 at a time.
constexpr int kDenseJMax = 128;
constexpr int kDxK = 64, kDxPitch = kDxK + 4;
__global__ void __launch_bounds__(256) dense_bwd_dx_tiled_kernel(const float* __restrict__ dy, int dys, const float* __restrict__ W,
                                                                 const float* __restrict__ inv_scale, float* __restrict__ dx, int dxs,
                                                                 int B, int K, int J, int accumulate) {
  extern __shared__ __align__(16) float dsm[];
  const int BP = (B + 3) & ~3;
  float* Wt = dsm;                      // [J][kDxPitch]   Wt[j][kk] = W[k0 + kk][j]
  float* dyT = dsm + J * kDxPitch;      // [J][BP]         dyT[j][b] = dy[b][j]
  const int k0 = blockIdx.x * kDxK;
  for (int i = threadIdx.x; i < kDxK * J; i += blockDim.x) {
    const int kk = i / J, j = i - kk * J;
    Wt[j * kDxPitch + kk] = (k0 + kk < K) ? W[static_cast<long long>(k0 + kk) * J + j] : 0.f;
  }
  for (int i = threadIdx.x; i < BP * J; i += blockDim.x) {
    const int b = i / J, j = i - b * J;
    dyT[j * BP + b] = b < B ? dy[static_cast<long long>(b) * dys + j] : 0.f;
  }
  __syncthreads();
  const float sc = inv_scale ? 1.f / __ldg(inv_scale) : 1.f;
  const int BT = BP >> 2;
  for (int t = threadIdx.x; t < BT * (kDxK / 4); t += blockDim.x) {
    const int kt = t % (kDxK / 4), bt = t / (kDxK / 4);
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
#pragma unroll 4
    for (int j = 0; j < J; ++j) {
      const float4 dv = *reinterpret_cast<const float4*>(dyT + j * BP + 4 * bt);
      const float4 wv = *reinterpret_cast<const float4*>(Wt + j * kDxPitch + 4 * kt);
      const float dr[4] = {dv.x, dv.y, dv.z, dv.w}, wc[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] += dr[r] * wc[c];
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int b = 4 * bt + r;
      if (b >= B) continue;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int k = k0 + 4 * kt + c;
        if (k >= K) continue;
        float* o = dx + static_cast<long long>(b) * dxs + k;
        const float v = acc[r][c] * sc;
        *o = accumulate ? *o + v : v;
      }
    }
  }
}

__global__ void __launch_bounds__(256) dense_bwd_dw_tiled_kernel(const float* __restrict__ x, int xs, const float* __restrict__ dy,
                                                                 int dys, const float* __restrict__ inv_scale,
                                                                 float* __restrict__ dW, float* __restrict__ db, int B, int K, int J) {
  __shared__ __align__(16) float xsm[32][32];               // [row][k]
  __shared__ __align__(16) float dsm2[32][kDenseJMax];      // [row][j]
  const int k0 = blockIdx.x * 32;
  const int J4 = (J + 3) >> 2;
  const int kt = threadIdx.x & 7, jt = threadIdx.x >> 3;     // tile: k = 4 kt .. +3, j = 4 jt .. +3 (jt < J4 <= 32)
  const bool active = jt < J4;
  for (int i = threadIdx.x; i < 32 * kDenseJMax; i += blockDim.x) dsm2[i / kDenseJMax][i % kDenseJMax] = 0.f;   // columns >= J stay zero
  __syncthreads();
  float acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
  float bsum = 0.f;                                          // CTA 0: thread t < J sums dy[:, t]
  for (int b0 = 0; b0 < B; b0 += 32) {
    const int nb = min(32, B - b0);
    for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) {
      const int bb = i >> 5, k2 = i & 31;
      xsm[bb][k2] = (bb < nb && k0 + k2 < K) ? x[static_cast<long long>(b0 + bb) * xs + k0 + k2] : 0.f;
    }
    for (int i = threadIdx.x; i < 32 * J; i += blockDim.x) {
      const int bb = i / J, j = i - bb * J;
      dsm2[bb][j] = bb < nb ? dy[static_cast<long long>(b0 + bb) * dys + j] : 0.f;
    }
    __syncthreads();
    if (active) {
#pragma unroll 8
      for (int bb = 0; bb < 32; ++bb) {                      // rows >= nb are zero
        const float4 xv = *reinterpret_cast<const float4*>(&xsm[bb][4 * kt]);
        const float4 dv = *reinterpret_cast<const float4*>(&dsm2[bb][4 * jt]);
        const float xr[4] = {xv.x, xv.y, xv.z, xv.w}, dc[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[r][c] += xr[r] * dc[c];
      }
    }
    if (db && blockIdx.x == 0 && threadIdx.x < J)
      for (int bb = 0; bb < nb; ++bb) bsum += dsm2[bb][threadIdx.x];
    __syncthreads();
  }
  const float sc = inv_scale ? 1.f / __ldg(inv_scale) : 1.f;
  if (active) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int k = k0 + 4 * kt + r;
      if (k >= K) continue;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (4 * jt + c < J) dW[static_cast<long long>(k) * J + 4 * jt + c] += acc[r][c] * sc;
    }
  }
  if (db && blockIdx.x == 0 && threadIdx.x < J) db[threadIdx.x] += bsum;
}

// dense LSTM cell backward (tf LSTMCell, gates i,j,f,o, forget bias)
__global__ void lstm_cell_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev,
                                     const float* __restrict__ c_new, const float* __restrict__ dh,
                                     const float* __restrict__ dc_next, float* __restrict__ dgates,
                                     float* __restrict__ dc_prev, int B, int U, float forget_bias) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * U) return;
  const int b = idx / U, u = idx % U;
  const float* g = gates + static_cast<long long>(b) * 4 * U;
  float* dg = dgates + static_cast<long long>(b) * 4 * U;
  const float si = sigm(g[u]), tj = tanhf(g[U + u]), sf = sigm(g[2 * U + u] + forget_bias), so = sigm(g[3 * U + u]);
  const float th = tanhf(c_new[idx]);
  const float dhv = dh[idx];
  const float dc = dhv * so * (1.f - th * th) + (dc_next ? dc_next[idx] : 0.f);
  dg[u] = dc * tj * si * (1.f - si);
  dg[U + u] = dc * si * (1.f - tj * tj);
  dg[2 * U + u] = dc * c_prev[idx] * sf * (1.f - sf);
  dg[3 * U + u] = dhv * th * so * (1.f - so);
  dc_prev[idx] = dc * sf;
}

// ------------------------------------------------------------------------------------------------
// reductions / elementwise
// ------------------------------------------------------------------------------------------------
// out[n][c] (+)= scale * sum_p x[n][p][c]   (bias gradients with n = 1; tile_concat / avg-pool adjoints)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ x, int xs, float* __restrict__ out, int os, int P,
                                                     int C, float scale, int rows_per_block) {
  const int n = blockIdx.z;
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int p0 = blockIdx.y * rows_per_block, p1 = min(P, p0 + rows_per_block);
  const int sub = threadIdx.x >> 5;
  float s = 0.f;
  if (c < C)
    for (int p = p0 + sub; p < p1; p += 8) s += x[(static_cast<long long>(n) * P + p) * xs + c];
  __shared__ float red[8][32];
  red[sub][threadIdx.x & 31] = s;
  __syncthreads();
  if (sub == 0 && c < C) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x & 31];
    atomicAdd(out + static_cast<long long>(n) * os + c, t * scale);
  }
}
// dst[r][c] = (accumulate ? dst : 0) + scale[r / rows_per_scale or none] * src[r][c]
__global__ void axpy_channels_kernel(const float* __restrict__ src, int ss, float* __restrict__ dst, int ds, long long total,
                                     int C, float scale, const int32_t* __restrict__ row_mask, long long rows_per_mask,
                                     int accumulate) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const long long r = idx / C;
  float v = scale * src[r * ss + c];
  if (row_mask && row_mask[r / rows_per_mask] != 0) v = 0.f;   // mask == 1 -> ground truth was used -> no gradient
  float* o = dst + r * ds + c;
  *o = accumulate ? *o + v : v;
}
// dy_pre = dy * act'(y)  from the activation OUTPUT y (sigmoid: y(1-y); lrelu/relu: sign of y)
__global__ void act_bwd_from_output_kernel(const float* __restrict__ y, int ys, const float* __restrict__ dyA, int das,
                                           const float* __restrict__ dyB, int dbs, float* __restrict__ dx, int dxs,
                                           long long total, int C, int act, float alpha) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const long long r = idx / C;
  const float yv = y[r * ys + c];
  float d = dyA[r * das + c] + (dyB ? dyB[r * dbs + c] : 0.f);
  if (act == VP_ACT_SIGMOID) d *= yv * (1.f - yv);
  else if (act == VP_ACT_RELU) d = yv > 0.f ? d : 0.f;
  else if (act == VP_ACT_LRELU) d = yv > 0.f ? d : alpha * d;
  else if (act == VP_ACT_TANH) d *= (1.f - yv * yv);
  dx[r * dxs + c] = d;
}
// avg-pool backward: dx[n][p][c] = dy[n][c] / P
__global__ void avgpool_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int dxs, long long total, int P, int C) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const long long np = idx / C;
  dx[np * dxs + c] = dy[(np / P) * C + c] / P;
}
// z = mu + sqrt(exp(lss))*eps backward + KL gradient:  kl = -0.5*mean_{rows} sum_z (1 + lss - mu^2 - exp(lss))
// dmu = dz + klw*mu/rows ; dlss = dz*eps*0.5*sqrt(exp(lss)) + klw*0.5*(exp(lss)-1)/rows ; zero where lss was clipped
__global__ void sample_z_bwd_kernel(const float* __restrict__ mu, const float* __restrict__ lss, const float* __restrict__ eps,
                                    const float* __restrict__ dz, float* __restrict__ dmu, float* __restrict__ dlss, int total,
                                    const float* __restrict__ kl_scale_dev) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const float kl_scale = kl_scale_dev ? __ldg(kl_scale_dev) : 0.f;
  const float l = lss[idx], e = expf(l);
  const float d = dz ? dz[idx] : 0.f;
  dmu[idx] = d + kl_scale * mu[idx];
  float dl = d * eps[idx] * 0.5f * sqrtf(e) + kl_scale * 0.5f * (e - 1.f);
  if (l <= -10.f || l >= 10.f) dl = 0.f;  // tf.clip_by_value passes no gradient outside the range
  dlss[idx] = dl;
}

// ------------------------------------------------------------------------------------------------
// losses: out[0] += value; gradient written (scaled by `gscale`) when dpred != null
// ------------------------------------------------------------------------------------------------
// mode 0: mean |t-p| (losses.l1_loss)   mode 1: mean (t-p)^2 (losses.l2_loss); over C valid channels of [rows][cs]
__global__ void __launch_bounds__(256) pixel_loss_kernel(const float* __restrict__ pred, int ps, const float* __restrict__ target,
                                                         int ts, float* __restrict__ dpred, int dps, long long rows, int C,
                                                         int mode, float inv_count, float gscale, float* __restrict__ out) {
  __shared__ float scratch[32];
  float s[1] = {0.f};
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < rows * C;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const long long r = idx / C;
    const float d = pred[r * ps + c] - target[r * ts + c];
    float g;
    if ((mode & 1) == 0) {
      s[0] += fabsf(d);
      g = gscale * inv_count * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
    } else {
      s[0] += d * d;
      g = gscale * inv_count * 2.f * d;
    }
    if (dpred) dpred[r * dps + c] = (mode & 2) ? dpred[r * dps + c] + g : g;   // bit 1: accumulate (l1 and l2 together)
  }
  bsum<1>(s, scratch);
  if (threadIdx.x == 0) atomicAdd(out, s[0] * inv_count);
}
// losses.gan_loss for labels in {0, 1}: kind 0 = LSGAN mean (l - y)^2; kind 1 = GAN = mean sigmoid-cross-entropy(l, y);
// kind 2 = SNGAN = mean softplus(l) (y = 0) / softplus(-l) (y = 1) -- numerically the same function as kind 1 for y in {0,1}.
// dlogits = gscale * d value / d logits.
__global__ void gan_loss_kernel(const float* __restrict__ logits, float label, int n, float gscale, int kind,
                                float* __restrict__ dlogits, float* __restrict__ out) {
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float x = logits[i];
    if (kind == 0) {
      const float d = x - label;
      s += d * d;
      if (dlogits) dlogits[i] = gscale * 2.f * d / n;
    } else {
      // max(x, 0) - x*y + log(1 + exp(-|x|))   (tf.nn.sigmoid_cross_entropy_with_logits)
      s += fmaxf(x, 0.f) - x * label + log1pf(expf(-fabsf(x)));
      // sigmoid(x) - y without the cancellation of 1 - sigmoid(x) for y = 1 (confident logits keep their tiny gradient)
      if (dlogits) dlogits[i] = gscale * (label != 0.f ? -1.f / (1.f + expf(x)) : 1.f / (1.f + expf(-x))) / n;
    }
  }
  __shared__ float scratch[32];
  float v[1] = {s};
  bsum<1>(v, scratch);
  if (threadIdx.x == 0) atomicAdd(out, v[0] / n);
}
// KL(q || N(0,1)) value (losses.kl_loss): -0.5 * mean_rows sum_z(1 + lss - mu^2 - exp(lss))
__global__ void kl_loss_kernel(const float* __restrict__ mu, const float* __restrict__ lss, int total, float inv_rows,
                               float* __restrict__ out) {
  float s = 0.f;
  for (int i = threadIdx.x; i < total; i += blockDim.x) s += 1.f + lss[i] - mu[i] * mu[i] - expf(lss[i]);
  __shared__ float scratch[32];
  float v[1] = {s};
  bsum<1>(v, scratch);
  if (threadIdx.x == 0) atomicAdd(out, -0.5f * v[0] * inv_rows);
}
// cosine distance (losses.cosine_distance): mean_rows sum_c (a/(|a|+eps) - b/(|b|+eps))^2 / 2 ; gradient w.r.t. a only.
// one warp per row of C channels.
__global__ void __launch_bounds__(256) cosine_distance_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                              float* __restrict__ da, long long rows, int C, float inv_rows,
                                                              float gscale, float* __restrict__ out) {
  const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  if (row < rows) {
    const float* ap = a + row * C;
    const float* bp = b + row * C;
    float na = 0.f, nb = 0.f;
    for (int c = lane; c < C; c += 32) { na += ap[c] * ap[c]; nb += bp[c] * bp[c]; }
    na = sqrtf(wsum(na)); nb = sqrtf(wsum(nb));
    const float ia = 1.f / (na + 1e-10f), ib = 1.f / (nb + 1e-10f);
    float s = 0.f, dotad = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float d = ap[c] * ia - bp[c] * ib;
      s += d * d;
      dotad += ap[c] * d;
    }
    s = wsum(s); dotad = wsum(dotad);
    acc = 0.5f * s * inv_rows;
    if (da) {
      // d/da_c [0.5*sum_k (a_k*ia - bh_k)^2] = d_c*ia - (sum_k a_k d_k) * ia^2 * a_c/na
      const float coef = (na > 0.f) ? dotad * ia * ia / na : 0.f;
      for (int c = lane; c < C; c += 32) {
        const float d = ap[c] * ia - bp[c] * ib;
        da[row * C + c] += gscale * inv_rows * (d * ia - coef * ap[c]);
      }
    }
  }
  __shared__ float red[8];
  if (lane == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(out, t);
  }
}

// The same with LPR lanes per row holding one float4 each (C = 4 * LPR <= 128): a and b are read once, every access is 16 bytes.
template <int LPR>
__global__ void __launch_bounds__(256) cosine_distance_vec_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                                  float* __restrict__ da, long long rows, float inv_rows, float gscale,
                                                                  float* __restrict__ out) {
  constexpr int C = 4 * LPR;
  const int sub = threadIdx.x % LPR;
  const long long row = (static_cast<long long>(blockIdx.x) * 256 + threadIdx.x) / LPR;
  const bool live = row < rows;
  float4 av = make_float4(0.f, 0.f, 0.f, 0.f), bv = av;
  if (live) {
    av = *reinterpret_cast<const float4*>(a + row * C + 4 * sub);
    bv = *reinterpret_cast<const float4*>(b + row * C + 4 * sub);
  }
  float na = av.x * av.x + av.y * av.y + av.z * av.z + av.w * av.w;
  float nb = bv.x * bv.x + bv.y * bv.y + bv.z * bv.z + bv.w * bv.w;
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) {
    na += __shfl_xor_sync(0xffffffffu, na, o);
    nb += __shfl_xor_sync(0xffffffffu, nb, o);
  }
  na = sqrtf(na); nb = sqrtf(nb);
  const float ia = 1.f / (na + 1e-10f), ib = 1.f / (nb + 1e-10f);
  const float d[4] = {av.x * ia - bv.x * ib, av.y * ia - bv.y * ib, av.z * ia - bv.z * ib, av.w * ia - bv.w * ib};
  float s = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3];
  float dotad = av.x * d[0] + av.y * d[1] + av.z * d[2] + av.w * d[3];
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    dotad += __shfl_xor_sync(0xffffffffu, dotad, o);
  }
  if (live && da) {
    const float coef = (na > 0.f) ? dotad * ia * ia / na : 0.f;
    const float k = gscale * inv_rows;
    float4* dp = reinterpret_cast<float4*>(da + row * C + 4 * sub);
    float4 o = *dp;
    o.x += k * (d[0] * ia - coef * av.x); o.y += k * (d[1] * ia - coef * av.y);
    o.z += k * (d[2] * ia - coef * av.z); o.w += k * (d[3] * ia - coef * av.w);
    *dp = o;
  }
  float acc = (live && sub == 0) ? 0.5f * s * inv_rows : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(out, t);
  }
}

// ------------------------------------------------------------------------------------------------
// fused TF-Adam over a flat parameter buffer (tf.train.AdamOptimizer, epsilon-hat form):
//   lr_t = lr*sqrt(1-b2^t)/(1-b1^t) ; m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; p -= lr_t m/(sqrt(v)+eps)
// gscale folds the 1/world_size of the data-parallel gradient mean (tf_utils.py:473-474).
// ------------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, const float* __restrict__ lr_t_dev, float b1, float b2, float eps, float gscale) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const float lr_t = __ldg(lr_t_dev);
  const float gv = g[idx] * gscale;
  const float mv = b1 * m[idx] + (1.f - b1) * gv;
  const float vv = b2 * v[idx] + (1.f - b2) * gv * gv;
  m[idx] = mv;
  v[idx] = vv;
  p[idx] -= lr_t * mv / (sqrtf(vv) + eps);
}

}  // namespace vp

using namespace vp;

static SrcList make_srcs(const float* const* ptrs, const int* strides, int count) {
  SrcList s;
  s.count = count;
  for (int i = 0; i < 4; ++i) { s.ptr[i] = i < count ? ptrs[i] : nullptr; s.stride[i] = i < count ? strides[i] : 0; }
  return s;
}

extern "C" int vp_inorm_act_bwd(const float* x, int x_cstride, const float* const* dy, const int* dy_cstride, int num_dy,
                                float* dx, int dx_cstride, int n, int positions, int c, const float* gamma, const float* beta,
                                const float* stats, int act, float alpha, float* dgamma, float* dbeta, vp_stream_t stream) {
  if (!x || !dy || !dx || !stats || !gamma || !beta || !dgamma || !dbeta) return set_error("vp_inorm_act_bwd: null pointer");
  if (c % 4 || num_dy < 1 || num_dy > 4) return set_error("vp_inorm_act_bwd: bad channel count / source count");
  {
    const int rc = slab_inorm_act_bwd(x, x_cstride, dy, dy_cstride, num_dy, dx, dx_cstride, n, positions, c, gamma, beta, stats, act, alpha,
                                      dgamma, dbeta, stream);
    if (rc <= 0) return rc;
  }
  dim3 grid(c / 4, n);
  const int staged = positions <= 4096 ? 1 : 0;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(inorm_act_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 4096 * 16);
    attr_set = true;
  }
  inorm_act_bwd_kernel<<<grid, positions >= 2048 ? 512 : 256, staged ? static_cast<size_t>(positions) * 32 : 0, as_stream(stream)>>>(
      x, x_cstride, make_srcs(dy, dy_cstride, num_dy), dx, dx_cstride, positions, c, gamma, beta, stats, act, alpha, dgamma, dbeta,
      staged);
  return check_launch("inorm_act_bwd_kernel");
}

extern "C" int vp_lstm_gates_bwd(const float* pre, int n, int positions, int filters, const float* c_prev, const float* gamma1,
                                 const float* beta1, const float* gamma2, const float* beta2, const float* stats1,
                                 const float* stats2, float forget_bias, const float* const* dh, const int* dh_cstride,
                                 int num_dh, const float* dc_next, float* dpre, float* dc_prev, float* dgamma1, float* dbeta1,
                                 float* dgamma2, float* dbeta2, vp_stream_t stream) {
  if (positions > 1024) return set_error("vp_lstm_gates_bwd: plane too large");
  if (filters % 4 || num_dh < 1 || num_dh > 4) return set_error("vp_lstm_gates_bwd: bad filters / source count");
  {
    const int rc = slab_gates_bwd(pre, n, positions, filters, c_prev, gamma1, beta1, gamma2, beta2, stats1, stats2, forget_bias, dh, dh_cstride,
                                  num_dh, dc_next, dpre, dc_prev, dgamma1, dbeta1, dgamma2, dbeta2, stream);
    if (rc <= 0) return rc;
  }
  const size_t smem = static_cast<size_t>(positions) * 40 * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(lstm_gates_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 1024 * 40 * 4);
    attr_set = true;
  }
  dim3 grid(filters / 4, n);
  lstm_gates_bwd_kernel<<<grid, positions >= 512 ? 512 : 256, smem, as_stream(stream)>>>(pre, positions, filters, c_prev, gamma1, beta1, gamma2, beta2,
                                                               stats1, stats2, forget_bias, make_srcs(dh, dh_cstride, num_dh),
                                                               dc_next, dpre, dc_prev, dgamma1, dbeta1, dgamma2, dbeta2);
  return check_launch("lstm_gates_bwd_kernel");
}

extern "C" int vp_composite_bwd(const float* dgen, const float* masks, int masks_cstride, const float* layers, int layers_cstride,
                                float* dlogits, int dlogits_cstride, float* dlayers, int dlayers_cstride, long long positions,
                                int num_layers, vp_stream_t stream) {
  composite_bwd_kernel<<<grid_for(positions, 256), 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const float4*>(dgen), masks, masks_cstride, layers, layers_cstride, dlogits, dlogits_cstride, dlayers,
      dlayers_cstride, positions, num_layers);
  return check_launch("composite_bwd_kernel");
}

extern "C" int vp_cdna_apply_bwd(const float* image, const float* kernels, const float* d_a, int d_a_cstride, const float* d_b,
                                 int d_b_cstride, float* dimage, float* dkernels, int n, int h, int w, int kh, int kw, int nk,
                                 vp_stream_t stream) {
  if (nk > 4) return set_error("vp_cdna_apply_bwd: at most 4 transformations");
  dim3 grid((h * w + 255) / 256, n);
  cdna_apply_bwd_kernel<<<grid, 256, 2 * kh * kw * nk * sizeof(float), as_stream(stream)>>>(
      reinterpret_cast<const float4*>(image), kernels, d_a, d_a_cstride, d_b, d_b_cstride, dimage, dkernels, n, h, w, kh, kw, nk);
  return check_launch("cdna_apply_bwd_kernel");
}

extern "C" int vp_cdna_kernel_norm_bwd(const float* raw, const float* out, const float* dout, float* draw, int b, int kh, int kw,
                                       int nk, vp_stream_t stream) {
  cdna_kernel_norm_bwd_kernel<<<grid_for(static_cast<long long>(b) * nk, 64), 64, 0, as_stream(stream)>>>(raw, out, dout, draw, b,
                                                                                                       kh, kw, nk);
  return check_launch("cdna_kernel_norm_bwd_kernel");
}

extern "C" int vp_dense_bwd(const float* x, int x_stride, const float* w, const float* inv_scale, const float* dy, int dy_stride,
                            float* dx, int dx_stride, int dx_accumulate, float* dw, float* dbias, int b, int k, int j,
                            vp_stream_t stream) {
  const bool wide = k >= 1024 && j <= kDenseJMax;
  if (dx) {
    const size_t smem = (static_cast<size_t>(j) * kDxPitch + static_cast<size_t>((b + 3) & ~3) * j) * sizeof(float);
    if (wide && smem <= 48 * 1024) {
      dense_bwd_dx_tiled_kernel<<<(k + kDxK - 1) / kDxK, 256, smem, as_stream(stream)>>>(dy, dy_stride, w, inv_scale, dx, dx_stride, b, k,
                                                                                         j, dx_accumulate);
      if (check_launch("dense_bwd_dx_tiled_kernel")) return -1;
    } else {
      dense_bwd_dx_kernel<<<grid_for(static_cast<long long>(b) * k, 256), 256, 0, as_stream(stream)>>>(dy, dy_stride, w, inv_scale, dx,
                                                                                                     dx_stride, b, k, j, dx_accumulate);
      if (check_launch("dense_bwd_dx_kernel")) return -1;
    }
  }
  if (dw) {
    if (wide) {
      dense_bwd_dw_tiled_kernel<<<(k + 31) / 32, 256, 0, as_stream(stream)>>>(x, x_stride, dy, dy_stride, inv_scale, dw, dbias, b, k, j);
      if (check_launch("dense_bwd_dw_tiled_kernel")) return -1;
    } else {
      dense_bwd_dw_kernel<<<grid_for(static_cast<long long>(k) * j, 256), 256, 0, as_stream(stream)>>>(x, x_stride, dy, dy_stride,
                                                                                                     inv_scale, dw, dbias, b, k, j);
      if (check_launch("dense_bwd_dw_kernel")) return -1;
    }
  }
  return 0;
}

extern "C" int vp_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c_new, const float* dh, const float* dc_next,
                                float* dgates, float* dc_prev, int b, int units, float forget_bias, vp_stream_t stream) {
  lstm_cell_bwd_kernel<<<grid_for(static_cast<long long>(b) * units, 128), 128, 0, as_stream(stream)>>>(
      gates, c_prev, c_new, dh, dc_next, dgates, dc_prev, b, units, forget_bias);
  return check_launch("lstm_cell_bwd_kernel");
}

extern "C" int vp_colsum(const float* x, int x_cstride, float* out, int out_stride, int n, long long positions, int c,
                         float scale, vp_stream_t stream) {
  const int rpb = 256;
  dim3 grid((c + 31) / 32, static_cast<unsigned>((positions + rpb - 1) / rpb), n);
  if (grid.y > 65535) return set_error("vp_colsum: too many rows");
  colsum_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, x_cstride, out, out_stride, static_cast<int>(positions), c, scale, rpb);
  return check_launch("colsum_kernel");
}

extern "C" int vp_axpy_channels(const float* src, int src_cstride, float* dst, int dst_cstride, long long rows, int c, float scale,
                                const int32_t* row_mask, long long rows_per_mask, int accumulate, vp_stream_t stream) {
  const long long total = rows * c;
  if (total == 0) return 0;
  axpy_channels_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(src, src_cstride, dst, dst_cstride, total, c, scale,
                                                                           row_mask, rows_per_mask, accumulate);
  return check_launch("axpy_channels_kernel");
}

extern "C" int vp_act_bwd(const float* y, int y_cstride, const float* dy_a, int dy_a_cstride, const float* dy_b, int dy_b_cstride,
                          float* dx, int dx_cstride, long long rows, int c, int act, float alpha, vp_stream_t stream) {
  const long long total = rows * c;
  act_bwd_from_output_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(y, y_cstride, dy_a, dy_a_cstride, dy_b,
                                                                                 dy_b_cstride, dx, dx_cstride, total, c, act, alpha);
  return check_launch("act_bwd_from_output_kernel");
}

extern "C" int vp_avgpool_bwd(const float* dy, float* dx, int dx_cstride, int n, int positions, int c, vp_stream_t stream) {
  const long long total = static_cast<long long>(n) * positions * c;
  avgpool_bwd_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(dy, dx, dx_cstride, total, positions, c);
  return check_launch("avgpool_bwd_kernel");
}

extern "C" int vp_sample_z_bwd(const float* mu, const float* lss, const float* eps, const float* dz, float* dmu, float* dlss,
                               int total, const float* kl_scale, vp_stream_t stream) {
  sample_z_bwd_kernel<<<grid_for(total, 128), 128, 0, as_stream(stream)>>>(mu, lss, eps, dz, dmu, dlss, total, kl_scale);
  return check_launch("sample_z_bwd_kernel");
}

extern "C" int vp_pixel_loss(const float* pred, int pred_cstride, const float* target, int target_cstride, float* dpred,
                             int dpred_cstride, long long rows, int c, int mode, long long mean_count, float grad_scale,
                             float* out, vp_stream_t stream) {
  const float inv = 1.f / static_cast<float>(mean_count);
  const int blocks = static_cast<int>(std::min<long long>(1184, (rows * c + 255) / 256));
  pixel_loss_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pred, pred_cstride, target, target_cstride, dpred, dpred_cstride, rows, c,
                                                           mode, inv, grad_scale, out);
  return check_launch("pixel_loss_kernel");
}

extern "C" int vp_gan_loss(const float* logits, float label, int n, float grad_scale, int kind, float* dlogits, float* out,
                           vp_stream_t stream) {
  if (kind < 0 || kind > 2) return set_error("vp_gan_loss: kind must be 0 (LSGAN), 1 (GAN) or 2 (SNGAN)");
  if (label != 0.f && label != 1.f && kind != 0) return set_error("vp_gan_loss: GAN / SNGAN need a label in {0, 1}");
  gan_loss_kernel<<<1, 256, 0, as_stream(stream)>>>(logits, label, n, grad_scale, kind, dlogits, out);
  return check_launch("gan_loss_kernel");
}

extern "C" int vp_kl_loss(const float* mu, const float* lss, int rows, int nz, float* out, vp_stream_t stream) {
  kl_loss_kernel<<<1, 256, 0, as_stream(stream)>>>(mu, lss, rows * nz, 1.f / rows, out);
  return check_launch("kl_loss_kernel");
}

extern "C" int vp_cosine_distance(const float* a, const float* b, float* da, long long rows, int c, float grad_scale, float* out,
                                  vp_stream_t stream) {
  const bool aligned = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(da)) & 15) == 0;
  if (aligned && (c == 32 || c == 64 || c == 128)) {
    const int lpr = c / 4;
    const unsigned blocks = static_cast<unsigned>((rows * lpr + 255) / 256);
    if (lpr == 8) cosine_distance_vec_kernel<8><<<blocks, 256, 0, as_stream(stream)>>>(a, b, da, rows, 1.f / rows, grad_scale, out);
    else if (lpr == 16) cosine_distance_vec_kernel<16><<<blocks, 256, 0, as_stream(stream)>>>(a, b, da, rows, 1.f / rows, grad_scale, out);
    else cosine_distance_vec_kernel<32><<<blocks, 256, 0, as_stream(stream)>>>(a, b, da, rows, 1.f / rows, grad_scale, out);
    return check_launch("cosine_distance_vec_kernel");
  }
  cosine_distance_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, as_stream(stream)>>>(a, b, da, rows, c, 1.f / rows,
                                                                                              grad_scale, out);
  return check_launch("cosine_distance_kernel");
}

extern "C" int vp_adam(float* p, const float* g, float* m, float* v, long long n, const float* lr_t, float beta1, float beta2,
                       float eps, float grad_scale, vp_stream_t stream) {
  adam_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(p, g, m, v, n, lr_t, beta1, beta2, eps, grad_scale);
  return check_launch("adam_kernel");
}
