// DPN_MODE_FP32: the whole hot path on CUDA cores in fp32 (residual physics in fp64).
//
// This is the mode that carries the 1e-4 parity claim against the reference's autograd path; it is
// also the on-device cross-check for the tcgen05 mode.  It executes the same algorithm as the tensor
// core path (DESIGN.md section 3: one value row, one reverse sweep, one combined tangent row per
// point; weight gradients as K = points contractions) as a sequence of batched SGEMMs with fused
// epilogues plus a handful of per-point kernels; activations live in the caller's workspace.
#include "dpn_fp32.cuh"

namespace dpn {
namespace f32 {

// ------------------------------------------------------------------------------------------------
// Batched SGEMM, 128x128x16 tiles, 256 threads, 8x8 outputs per thread.
//   C[m,n] = sum_k A(m,k) * B(k,n)
//   A_KC: A is [M,K] row-major (k contiguous), else A is [K,M] row-major (m contiguous)
//   B_KC: B is [N,K] row-major (k contiguous), else B is [K,N] row-major (n contiguous)
// blockIdx.z = batch * ksplit + split.  Requires K-contiguous operands to have K % 16 == 0 and all
// leading dimensions % 4 == 0 (true for 192 / 256); the k extent of MN-contiguous operands is free.
// ------------------------------------------------------------------------------------------------
constexpr int BM = 128, BN = 128, BK = 16, PADW = BM + 4;

template <bool KC>
__device__ __forceinline__ void tile_fetch(const float* __restrict__ P, int ld, int mn0, int mn_max, int k0,
                                           int k_max, int tid, float4 (&r)[2]) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    int idx = tid + 256 * j;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KC) {
      int row = idx >> 2, kq = idx & 3;
      if (mn0 + row < mn_max && k0 + kq * 4 < k_max)
        v = __ldg(reinterpret_cast<const float4*>(P + (size_t)(mn0 + row) * ld + k0 + kq * 4));
    } else {
      int k = idx >> 5, mq = idx & 31;
      if (k0 + k < k_max && mn0 + mq * 4 < mn_max)
        v = __ldg(reinterpret_cast<const float4*>(P + (size_t)(k0 + k) * ld + mn0 + mq * 4));
    }
    r[j] = v;
  }
}

template <bool KC>
__device__ __forceinline__ void tile_stash(float (*S)[PADW], int tid, const float4 (&r)[2]) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    int idx = tid + 256 * j;
    if (KC) {
      int row = idx >> 2, kq = idx & 3;
      S[kq * 4 + 0][row] = r[j].x;
      S[kq * 4 + 1][row] = r[j].y;
      S[kq * 4 + 2][row] = r[j].z;
      S[kq * 4 + 3][row] = r[j].w;
    } else {
      int k = idx >> 5, mq = idx & 31;
      *reinterpret_cast<float4*>(&S[k][mq * 4]) = r[j];
    }
  }
}

template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(256, 2) sgemm_kernel(const Gemm g) {
  __shared__ __align__(16) float As[BK][PADW];
  __shared__ __align__(16) float Bs[BK][PADW];
  const int tid = threadIdx.x;
  const int batch = blockIdx.z / g.ksplit, split = blockIdx.z % g.ksplit;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int kchunk = ((g.K + g.ksplit - 1) / g.ksplit + BK - 1) / BK * BK;
  const int kbeg = split * kchunk, kend = min(g.K, kbeg + kchunk);
  const float* A = g.A + (size_t)batch * g.sA;
  const float* B = g.B + (size_t)batch * g.sB;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float4 ra[2], rb[2];
  if (kbeg < kend) {
    tile_fetch<A_KC>(A, g.lda, m0, g.M, kbeg, kend, tid, ra);
    tile_fetch<B_KC>(B, g.ldb, n0, g.N, kbeg, kend, tid, rb);
  }
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    tile_stash<A_KC>(As, tid, ra);
    tile_stash<B_KC>(Bs, tid, rb);
    __syncthreads();
    if (k0 + BK < kend) {
      tile_fetch<A_KC>(A, g.lda, m0, g.M, k0 + BK, kend, tid, ra);
      tile_fetch<B_KC>(B, g.ldb, n0, g.N, k0 + BK, kend, tid, rb);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[8], b[8];
      *reinterpret_cast<float4*>(&a[0]) = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      *reinterpret_cast<float4*>(&a[4]) = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
      *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      *reinterpret_cast<float4*>(&b[4]) = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  // ---- fused epilogue ----
  const float* bias = g.bias ? g.bias + (size_t)batch * g.sBias : nullptr;
  const float* mask = g.mask ? g.mask + (size_t)batch * g.sMask : nullptr;
  const float* addsrc = g.addsrc ? g.addsrc + (size_t)batch * g.sAdd : nullptr;
  const float* rowscale = g.rowscale ? g.rowscale + batch * g.sRow : nullptr;
  float* out = g.out ? g.out + (size_t)batch * g.sOut : nullptr;
  float* out2 = g.out2 ? g.out2 + (size_t)batch * g.sOut2 : nullptr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (m >= g.M) continue;
    const float rs = rowscale ? rowscale[(size_t)m * g.ldRow] : 0.f;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int n = n0 + jh * 64 + tx * 4;
      if (n >= g.N) continue;
      float v[4] = {acc[i][jh * 4 + 0], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]};
      const size_t off = (size_t)m * g.N + n;
      if (g.atomic) {
#pragma unroll
        for (int e = 0; e < 4; ++e) atomicAdd(out + off + e, v[e]);
        continue;
      }
      if (bias) {
        const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + n));
        v[0] += bv.x; v[1] += bv.y; v[2] += bv.z; v[3] += bv.w;
      }
      if (g.accumulate) {
        const float4 ov = *reinterpret_cast<const float4*>(out + off);
        v[0] += ov.x; v[1] += ov.y; v[2] += ov.z; v[3] += ov.w;
      }
      if (g.relu) {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = fmaxf(v[e], 0.f);
      }
      if (mask) {
        const float4 mv = __ldg(reinterpret_cast<const float4*>(mask + off));
        v[0] = mv.x > 0.f ? v[0] : 0.f; v[1] = mv.y > 0.f ? v[1] : 0.f;
        v[2] = mv.z > 0.f ? v[2] : 0.f; v[3] = mv.w > 0.f ? v[3] : 0.f;
      }
      if (out) *reinterpret_cast<float4*>(out + off) = make_float4(v[0], v[1], v[2], v[3]);
      if (out2) {
        const float4 sv = __ldg(reinterpret_cast<const float4*>(addsrc + off));
        *reinterpret_cast<float4*>(out2 + off) =
            make_float4(v[0] + rs * sv.x, v[1] + rs * sv.y, v[2] + rs * sv.z, v[3] + rs * sv.w);
      }
    }
  }
}

int launch_gemm(const Gemm& g, int layout, int batches, cudaStream_t st) {
  dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, batches * g.ksplit);
  if (g.M <= 0) return 0;
  switch (layout) {
    case NT: sgemm_kernel<true, true><<<grid, 256, 0, st>>>(g); break;
    case NN: sgemm_kernel<true, false><<<grid, 256, 0, st>>>(g); break;
    case TN: sgemm_kernel<false, false><<<grid, 256, 0, st>>>(g); break;
    default: set_error("bad gemm layout"); return DPN_E_INVALID;
  }
  DPN_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Per-point kernels
// ------------------------------------------------------------------------------------------------
// PE [P,192] (interface_physics.py:322-332 + position_encoding.py:35-50) and PE6 [P,192] (variable_net.py:73).
__global__ void encode_kernel(const DevConsts K, int P, const float* __restrict__ x, const float* __restrict__ y,
                              const float* __restrict__ t, const float* __restrict__ cd, float* __restrict__ pe,
                              float* __restrict__ pe6) {
  const int p = blockIdx.x * blockDim.y + threadIdx.y;
  if (p >= P) return;
  const int l = threadIdx.x;  // 0..31
  if (pe) {
    const float z[3] = {(x[p] / K.dxf) / K.wm1, (y[p] / K.dyf) / K.hm1, t[p] / K.t_span};
    const float band = K.band[l];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float s, co;
      sincosf(z[c] * band, &s, &co);
      pe[(size_t)p * C + l * 6 + c] = s;
      pe[(size_t)p * C + l * 6 + 3 + c] = co;
    }
  }
  if (pe6 && l < NF6) {
    const float band = K.band6[l];
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      float s, co;
      sincosf(cd[(size_t)p * 6 + c] * band, &s, &co);
      pe6[(size_t)p * C + l * 12 + c] = s;
      pe6[(size_t)p * C + l * 12 + 6 + c] = co;
    }
  }
}

// o[p,k] = 2 wo.c + u.g + (wo.bb + bo) + ref ;  UM[p,:] = u * (g > 0).   One warp per (point, net).
__global__ void out_kernel(int P, int Kn, const float* __restrict__ CC, const float* __restrict__ GG,
                           const float* __restrict__ wo2, const float* __restrict__ uvec,
                           const float* __restrict__ cst, const float* __restrict__ ref, int ref_ld,
                           float* __restrict__ o, float* __restrict__ UM) {
  const int p = blockIdx.x * blockDim.y + threadIdx.y, k = blockIdx.y, l = threadIdx.x;
  if (p >= P) return;
  const size_t base = ((size_t)k * P + p) * H;
  float s = 0.f;
#pragma unroll
  for (int j = l; j < H; j += 32) {
    const float g = GG[base + j], u = uvec[k * H + j];
    s = fmaf(wo2[k * H + j], CC[base + j], s);
    s = fmaf(u, g, s);
    if (UM) UM[base + j] = g > 0.f ? u : 0.f;
  }
#pragma unroll
  for (int w = 16; w; w >>= 1) s += __shfl_xor_sync(0xffffffffu, s, w);
  if (l == 0) o[(size_t)p * Kn + k] = s + cst[k] + ref[(size_t)p * ref_ld + k];
}

// od[p,k,c] = sum_j JIN[p,j] dPE[p,j] over j%3==c, dPE from PE: d sin = band*cos, d cos = -band*sin.
__global__ void jac_kernel(const DevConsts K, int P, int Kn, const float* __restrict__ JIN,
                           const float* __restrict__ pe, float* __restrict__ od) {
  const int p = blockIdx.x * blockDim.y + threadIdx.y, k = blockIdx.y, l = threadIdx.x;
  if (p >= P) return;
  const float* jin = JIN + ((size_t)k * P + p) * C;
  const float* pr = pe + (size_t)p * C;
  const float band = K.band[l];
  float s[3];
#pragma unroll
  for (int c = 0; c < 3; ++c)
    s[c] = band * (jin[l * 6 + c] * pr[l * 6 + 3 + c] - jin[l * 6 + 3 + c] * pr[l * 6 + c]);
#pragma unroll
  for (int w = 16; w; w >>= 1) {
#pragma unroll
    for (int c = 0; c < 3; ++c) s[c] += __shfl_xor_sync(0xffffffffu, s[c], w);
  }
  if (l == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) od[((size_t)p * Kn + k) * 3 + c] = s[c];
  }
}

// Residuals, loss sums and seeds (see residual_point).  One thread per point; block-reduced fp64 atomics.
// blockIdx.y = sample: per-point work arrays advance by `srow` rows per sample, caller arrays (f, vals, jac) by `sq` points.
__global__ void residual_kernel(const DevConsts K, int P, const float* __restrict__ o, const float* __restrict__ od,
                                const float* __restrict__ f, double inv_n, double seed_scale,
                                double* __restrict__ loss6, float* __restrict__ dov, float* __restrict__ dod,
                                float* __restrict__ vals, float* __restrict__ jac, size_t srow, size_t sq) {
  __shared__ double red[6][8];
  const size_t bs = blockIdx.y;
  o += bs * srow * 6; od += bs * srow * 18; dov += bs * srow * 6; dod += bs * srow * 18;
  f += bs * sq; loss6 += bs * 6;
  if (vals) vals += bs * sq * 6;
  if (jac) jac += bs * sq * 18;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  double r2w[6] = {0, 0, 0, 0, 0, 0};
  if (p < P) {
    float ol[6], odl[18];
#pragma unroll
    for (int i = 0; i < 6; ++i) ol[i] = o[(size_t)p * 6 + i];
#pragma unroll
    for (int i = 0; i < 18; ++i) odl[i] = od[(size_t)p * 18 + i];
    double dv[6], dd[18], vl[6], jc[18];
    residual_point(K, ol, odl, (double)f[p], inv_n, seed_scale, r2w, dv, dd, vl, jc);
#pragma unroll
    for (int i = 0; i < 6; ++i) dov[(size_t)p * 6 + i] = (float)dv[i];
#pragma unroll
    for (int i = 0; i < 18; ++i) dod[(size_t)p * 18 + i] = (float)dd[i];
    if (vals) {
#pragma unroll
      for (int i = 0; i < 6; ++i) vals[(size_t)p * 6 + i] = (float)vl[i];
    }
    if (jac) {
#pragma unroll
      for (int i = 0; i < 18; ++i) jac[(size_t)p * 18 + i] = (float)jc[i];
    }
  }
#pragma unroll
  for (int e = 0; e < 6; ++e) {
    double v = r2w[e];
#pragma unroll
    for (int w = 16; w; w >>= 1) v += __shfl_xor_sync(0xffffffffu, v, w);
    if ((threadIdx.x & 31) == 0) red[e][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[threadIdx.x][w];
    atomicAdd(loss6 + threadIdx.x, v);
  }
}

// Supervised data loss on the points of a PDE call (SURVEY 8(f) N1; interface_physics.py:464-474, losses/weights_loss.py:12-20):
// loss += factor * inv_n/6 * sum smooth_l1(o - target; beta) and the seed of the value row gets d(loss)/d(o) added, so the one
// backward pass that follows serves both losses.  One thread per point; o is the normalised net output (before inverse_norm).
__global__ void margin_seed_kernel(int P, const float* __restrict__ o, const float* __restrict__ target, double beta, double coef,
                                   double seed_scale, double* __restrict__ loss, float* __restrict__ dov, float* __restrict__ o_out,
                                   size_t srow, size_t sq) {
  __shared__ double red[8];
  const size_t bs = blockIdx.y;
  o += bs * srow * 6; dov += bs * srow * 6; target += bs * sq * 6; loss += bs;
  if (o_out) o_out += bs * sq * 6;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  double acc = 0.0;
  if (p < P) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float ov = o[(size_t)p * 6 + k];
      const double d = (double)ov - (double)target[(size_t)p * 6 + k], ad = fabs(d);
      const bool quad = ad < beta;
      acc += quad ? 0.5 * d * d / beta : ad - 0.5 * beta;
      const double g = quad ? d / beta : (d > 0.0 ? 1.0 : -1.0);
      dov[(size_t)p * 6 + k] += (float)(seed_scale * coef * g);
      if (o_out) o_out[(size_t)p * 6 + k] = ov;
    }
  }
#pragma unroll
  for (int w = 16; w; w >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, w);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[w];
    atomicAdd(loss, coef * v);
  }
}

// Backward inputs: XT[k][p,j] = dod[p,k,j%3] dPE[p,j];  ZP = dov PE + XT;  ZD = dov PE6.
__global__ void bwd_in_kernel(const DevConsts K, int P, int Kn, const float* __restrict__ pe,
                              const float* __restrict__ pe6, const float* __restrict__ dov,
                              const float* __restrict__ dod, float* __restrict__ XT, float* __restrict__ ZP,
                              float* __restrict__ ZD) {
  const int p = blockIdx.x * blockDim.y + threadIdx.y, k = blockIdx.y, l = threadIdx.x;
  if (p >= P) return;
  const float dv = dov[(size_t)p * Kn + k];
  const float* pr = pe + (size_t)p * C;
  const size_t base = ((size_t)k * P + p) * C;
  if (dod) {
    const float band = K.band[l];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float dd = dod[((size_t)p * Kn + k) * 3 + c];
      const float s = pr[l * 6 + c], co = pr[l * 6 + 3 + c];
      const float xs = dd * band * co, xc = -dd * band * s;
      XT[base + l * 6 + c] = xs;
      XT[base + l * 6 + 3 + c] = xc;
      ZP[base + l * 6 + c] = fmaf(dv, s, xs);
      ZP[base + l * 6 + 3 + c] = fmaf(dv, co, xc);
    }
  } else {
#pragma unroll
    for (int j = l; j < C; j += 32) ZP[base + j] = dv * pr[j];
  }
  const float* p6 = pe6 + (size_t)p * C;
#pragma unroll
  for (int j = l; j < C; j += 32) ZD[base + j] = dv * p6[j];
}

// Z[k][p,:] = rowscale[p,k] * X[k][p,:]   (values-only backward: no tangent row)
__global__ void scale_rows_kernel(int P, int Kn, int W, const float* __restrict__ X, const float* __restrict__ rs,
                                  float* __restrict__ Z) {
  const int p = blockIdx.x * blockDim.y + threadIdx.y, k = blockIdx.y, l = threadIdx.x;
  if (p >= P) return;
  const float s = rs[(size_t)p * Kn + k];
  const size_t base = ((size_t)k * P + p) * W;
  for (int j = l; j < W; j += 32) Z[base + j] = s * X[base + j];
}

// out[k][j] += sum_p w[p,k] * X[k][p,j]   (w == nullptr -> plain column sum);  also sums w itself when X == nullptr.
__global__ void colsum_kernel(int P, int Kn, int rows_per_block, const float* __restrict__ X,
                              const float* __restrict__ w, float* __restrict__ out, float* __restrict__ out_b,
                              float* __restrict__ out_c) {
  const int k = blockIdx.y, j = threadIdx.x;  // 256 threads
  const int p0 = blockIdx.x * rows_per_block, p1 = min(P, p0 + rows_per_block);
  float s = 0.f;
  for (int p = p0; p < p1; ++p) {
    const float ww = w ? w[(size_t)p * Kn + k] : 1.f;
    s = fmaf(ww, X[((size_t)k * P + p) * H + j], s);
  }
  atomicAdd(out + k * H + j, s);
  if (out_b) atomicAdd(out_b + k * H + j, s);
  if (out_c) atomicAdd(out_c + k * H + j, s);
}

__global__ void sum_seed_kernel(int P, int Kn, const float* __restrict__ dov, float* __restrict__ sdo) {
  const int k = blockIdx.y;
  float s = 0.f;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) s += dov[(size_t)p * Kn + k];
#pragma unroll
  for (int w = 16; w; w >>= 1) s += __shfl_xor_sync(0xffffffffu, s, w);
  if ((threadIdx.x & 31) == 0) atomicAdd(sdo + k, s);
}

// Per-call constants of the folded output layer: u = Wb^T wo, wo2 = 2 wo, cst = wo.bb + bo; bsum[b,k] = b2+bd+e.
__global__ void prep_kernel(int B, int Kn, const float* __restrict__ Wb, const float* __restrict__ bb,
                            const float* __restrict__ wo, const float* __restrict__ bo, const float* __restrict__ b2,
                            const float* __restrict__ bd, const float* __restrict__ e, float* __restrict__ uvec,
                            float* __restrict__ wo2, float* __restrict__ cst, float* __restrict__ bsum) {
  const int k = blockIdx.x, j = threadIdx.x;  // 256 threads
  __shared__ float red[8];
  const float* W = Wb + (size_t)k * H * H;
  float s = 0.f;
  for (int i = 0; i < H; ++i) s = fmaf(W[(size_t)i * H + j], wo[k * H + i], s);
  uvec[k * H + j] = s;
  wo2[k * H + j] = 2.f * wo[k * H + j];
  float d = wo[k * H + j] * bb[k * H + j];
#pragma unroll
  for (int w = 16; w; w >>= 1) d += __shfl_xor_sync(0xffffffffu, d, w);
  if ((j & 31) == 0) red[j >> 5] = d;
  __syncthreads();
  if (j == 0) {
    float tot = 0.f;
    for (int w = 0; w < 8; ++w) tot += red[w];
    cst[k] = tot + bo[k];
  }
  for (int b = 0; b < B; ++b)
    bsum[((size_t)b * Kn + k) * H + j] = b2[((size_t)b * Kn + k) * H + j] + bd[k * H + j] + e[((size_t)b * Kn + k) * H + j];
}

// Gradients of the folded layer from the column sums: dWb = wo (x) vg ; dwo = 2 vc + Wb vg + bb sdo ;
// dbb = wo sdo ; dbo = sdo.
__global__ void __launch_bounds__(256) finalize_kernel(const float* __restrict__ Wb, const float* __restrict__ bb, const float* __restrict__ wo,
                                const float* __restrict__ vc, const float* __restrict__ vg,
                                const float* __restrict__ sdo, float* __restrict__ gWb, float* __restrict__ gbb,
                                float* __restrict__ gwo, float* __restrict__ gbo) {
  // grid (Kn, 8): block y handles 32 rows of Wb, one warp per row at a time, lanes along the row (coalesced)
  const int k = blockIdx.x, lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  __shared__ float vgs[H];
  vgs[threadIdx.x] = vg[k * H + threadIdx.x];
  __syncthreads();
  const float sd = sdo[k];
  for (int i = blockIdx.y * 32 + wrp; i < blockIdx.y * 32 + 32; i += 8) {
    const float* W = Wb + ((size_t)k * H + i) * H;
    float* G = gWb + ((size_t)k * H + i) * H;
    const float w = wo[k * H + i];
    float s = 0.f;
#pragma unroll
    for (int j = lane; j < H; j += 32) {
      s = fmaf(W[j], vgs[j], s);
      G[j] = w * vgs[j];
    }
#pragma unroll
    for (int m = 16; m; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    if (lane == 0) {
      gwo[k * H + i] = 2.f * vc[k * H + i] + s + bb[k * H + i] * sd;
      gbb[k * H + i] = w * sd;
    }
  }
  if (blockIdx.y == 0 && threadIdx.x == 0) gbo[k] = sd;
}

// Caller seeds -> workspace seeds, one thread per point, blockIdx.y = sample (srow / sq as residual_kernel):
//   dov[p,k] = d_o[q,k] scale;  dod[p,k,c] = d_jac[q,k,c] sc_c scale - the chain rule from the caller's physical units into the
//   normalised z = (x / (dx (W-1)), y / (dy (H-1)), t / t_span) that od and the residual's dod are taken against.
__global__ void seed_in_kernel(const DevConsts K, int P, int Kn, const float* __restrict__ d_o, const float* __restrict__ d_jac,
                               float scale, double scale_d, float* __restrict__ dov, float* __restrict__ dod, size_t srow, size_t sq) {
  const size_t bs = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const size_t row = bs * srow + p, q = bs * sq + p;
  const double sc[3] = {K.sx, K.sy, K.st};
  for (int k = 0; k < Kn; ++k) {
    dov[row * Kn + k] = d_o ? d_o[q * Kn + k] * scale : 0.f;
    if (dod) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
        dod[(row * Kn + k) * 3 + c] = d_jac ? (float)((double)d_jac[(q * Kn + k) * 3 + c] * sc[c] * scale_d) : 0.f;
    }
  }
}

// The fields of dpn_decoder_jac_fwd: o_out[q,k] = o[p,k], jac[q,k,c] = od[p,k,c] sc_c (physical units, before inverse_norm).
__global__ void fields_kernel(const DevConsts K, int P, int Kn, const float* __restrict__ o, const float* __restrict__ od,
                              float* __restrict__ o_out, float* __restrict__ jac, size_t srow, size_t sq) {
  const size_t bs = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const size_t row = bs * srow + p, q = bs * sq + p;
  const double sc[3] = {K.sx, K.sy, K.st};
  for (int k = 0; k < Kn; ++k) {
    o_out[q * Kn + k] = o[row * Kn + k];
#pragma unroll
    for (int c = 0; c < 3; ++c) jac[(q * Kn + k) * 3 + c] = (float)((double)od[(row * Kn + k) * 3 + c] * sc[c]);
  }
}

// ------------------------------------------------------------------------------------------------
// Workspace carving
// ------------------------------------------------------------------------------------------------
static inline size_t al(size_t n) { return (n + 255) & ~(size_t)255; }

// What a values-only pass touches comes first; what only the reverse sweep, the residual or the backward touches follows.
// values_only: the prefix plus the staging of the lattice job's per-point inputs (one sample's chunk), in place of the rest.
Workspace carve(char* base, int P, int Kn, int B, bool values_only = false) {
  Workspace w;
  memset(&w, 0, sizeof(w));
  size_t off = 0;
  auto take = [&](size_t floats) { float* p = reinterpret_cast<float*>(base + off); off += al(floats * 4); return p; };
  w.pe = take((size_t)P * C);
  w.pe6 = take((size_t)P * C);
  w.o = take((size_t)P * Kn);
  float** vs[] = {&w.H1, &w.CC, &w.GG};
  for (auto h : vs) *h = take((size_t)Kn * P * H);
  w.uvec = take((size_t)Kn * H);
  w.wo2 = take((size_t)Kn * H);
  w.cst = take(Kn);
  w.bsum = take((size_t)B * Kn * H);
  if (values_only) {
    w.lx = take(P);
    w.ly = take(P);
    w.lt = take(P);
    w.lcd = take((size_t)P * 6);
    w.bytes = off;
    return w;
  }
  w.od = take((size_t)P * Kn * 3);
  w.dov = take((size_t)P * Kn);
  w.dod = take((size_t)P * Kn * 3);
  float** hs[] = {&w.UM, &w.YT, &w.QM, &w.HT, &w.CT, &w.ZH, &w.ZC, &w.GZ};
  for (auto h : hs) *h = take((size_t)Kn * P * H);
  float** cs[] = {&w.JIN, &w.ZP, &w.ZD};
  for (auto c : cs) *c = take((size_t)Kn * P * C);
  w.vc = take((size_t)Kn * H);
  w.vg = take((size_t)Kn * H);
  w.sdo = take(Kn);
  w.bytes = off;
  return w;
}

size_t workspace_bytes(int P, int Kn, int B) { return carve(nullptr, P, Kn, B).bytes; }
size_t lattice_workspace_bytes(int P, int Kn, int B) { return carve(nullptr, P, Kn, B, true).bytes; }

// ------------------------------------------------------------------------------------------------
// Driver
// ------------------------------------------------------------------------------------------------
static Gemm mk(int M, int N, int Kd, const float* A, int lda, size_t sA, const float* Bm, int ldb, size_t sB,
               float* out, size_t sOut) {
  Gemm g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N; g.K = Kd; g.A = A; g.lda = lda; g.sA = sA; g.B = Bm; g.ldb = ldb; g.sB = sB;
  g.out = out; g.sOut = sOut; g.ksplit = 1;
  return g;
}

int run(const Job& J, cudaStream_t st) {
  const int B = J.shape.B, N = J.shape.N, Kn = J.shape.K;
  const int chunk = J.chunk;
  const DevConsts& DC = J.dc;
  const bool lattice = J.kind == JOB_LATTICE;
  Workspace w = carve(reinterpret_cast<char*>(J.workspace), chunk, Kn, B, lattice);
  const DpnWeights& Wt = *J.w;
  const bool pde = J.kind == JOB_PDE;
  const bool jac_fwd = J.kind == JOB_JAC_FWD;
  const bool want_bwd = J.grads != nullptr;
  const bool need_sweep = pde || jac_fwd || J.kind == JOB_DEC_BWD || J.kind == JOB_JAC_BWD;   // reverse sweep (J-side vectors)
  const bool want_od = pde || jac_fwd;                       // G6 and the Jacobian itself: the backward never reads od
  const bool tangent = pde || J.d_jac != nullptr;           // seeds on the Jacobian: the tangent row (dod, G7 - G9) in the backward
  const double inv_n = 1.0 / (double)(J.shape.n_norm > 0 ? J.shape.n_norm : N);
  const double seed_scale = J.shape.seed_scale != 0.f ? (double)J.shape.seed_scale : 1.0;

  prep_kernel<<<Kn, 256, 0, st>>>(B, Kn, Wt.Wb, Wt.bb, Wt.wo, Wt.bo, Wt.b2, Wt.bd, Wt.e, w.uvec, w.wo2, w.cst, w.bsum);
  DPN_LAUNCH_OK();
  if (pde) DPN_CUDA_OK(cudaMemsetAsync(J.out->loss_terms, 0, sizeof(double) * 6 * B, st));
  if (pde && J.margin) DPN_CUDA_OK(cudaMemsetAsync(J.margin->loss, 0, sizeof(double) * B, st));
  if (want_bwd) {
    const DpnGrads& G = *J.grads;
    const size_t BK_ = (size_t)B * Kn;
    DPN_CUDA_OK(cudaMemsetAsync(G.W1, 0, BK_ * H * C * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.b1, 0, BK_ * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.W2, 0, BK_ * H * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.b2, 0, BK_ * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.e, 0, BK_ * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.Wd, 0, (size_t)Kn * H * C * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.bd, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.Wa, 0, (size_t)Kn * H * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.ba, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(w.vc, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(w.vg, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(w.sdo, 0, (size_t)Kn * 4, st));
  }
  const dim3 pb(32, 8);
  for (int b = 0; b < B; ++b) {
    const size_t gW1 = (size_t)b * Kn * H * C, gW2 = (size_t)b * Kn * H * H, gb = (size_t)b * Kn * H;
    for (int p0 = 0; p0 < N; p0 += chunk) {
      const int P = min(chunk, N - p0);
      const size_t q0 = (size_t)b * N + p0;
      const size_t sH = (size_t)P * H, sC = (size_t)P * C;
      const unsigned gp = (P + 7) / 8;
      const float* pe = w.pe;
      int rc;
      if (lattice) {                                                 // staged inputs of this (sample, chunk)
        if ((rc = launch_lattice(J.lat, b, 1, p0, P, w.lx, w.ly, w.lt, w.lcd, st))) return rc;
        encode_kernel<<<gp, pb, 0, st>>>(DC, P, w.lx, w.ly, w.lt, w.lcd, w.pe, w.pe6);
      } else if (J.pts->coord_pe) {
        pe = J.pts->coord_pe + q0 * C;
        encode_kernel<<<gp, pb, 0, st>>>(DC, P, nullptr, nullptr, nullptr, J.pts->coord_data + q0 * 6, nullptr, w.pe6);
      } else {
        encode_kernel<<<gp, pb, 0, st>>>(DC, P, J.pts->x + q0, J.pts->y + q0, J.pts->t + q0,
                                         J.pts->coord_data + q0 * 6, w.pe, w.pe6);
      }
      DPN_LAUNCH_OK();
      // G1: H1 = relu(PE W1^T + b1)
      Gemm g = mk(P, H, C, pe, C, 0, Wt.W1 + gW1, C, (size_t)H * C, w.H1, sH);
      g.bias = Wt.b1 + gb; g.sBias = H; g.relu = 1;
      if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
      // G2: CC = H1 W2^T + PE6 Wd^T + (b2 + bd + e)
      g = mk(P, H, H, w.H1, H, sH, Wt.W2 + gW2, H, (size_t)H * H, w.CC, sH);
      g.bias = w.bsum + gb; g.sBias = H;
      if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
      g = mk(P, H, C, w.pe6, C, 0, Wt.Wd, C, (size_t)H * C, w.CC, sH);
      g.accumulate = 1;
      if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
      // G3: GG = relu(CC Wa^T + ba)
      g = mk(P, H, H, w.CC, H, sH, Wt.Wa, H, (size_t)H * H, w.GG, sH);
      g.bias = Wt.ba; g.sBias = H; g.relu = 1;
      if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
      // outputs
      float* o_dst = (J.kind == JOB_DEC_FWD) ? J.o + q0 * Kn : w.o;
      const float* ref = lattice ? w.lcd : (J.pts->ref ? J.pts->ref + q0 * Kn : J.pts->coord_data + q0 * 6);
      const int ref_ld = !lattice && J.pts->ref ? Kn : 6;
      out_kernel<<<dim3(gp, Kn), pb, 0, st>>>(P, Kn, w.CC, w.GG, w.wo2, w.uvec, w.cst, ref, ref_ld, o_dst,
                                              need_sweep ? w.UM : nullptr);
      DPN_LAUNCH_OK();
      if (lattice && (rc = launch_lattice_emit(J.lat, 1, P, w.o, (size_t)P, J.o + q0 * 6, (size_t)N * 6, st))) return rc;
      if (!need_sweep) continue;
      // G4: YT = UM Wa + 2wo ; G5: QM = (YT W2) * [H1>0] ; G6: JIN = QM W1
      g = mk(P, H, H, w.UM, H, sH, Wt.Wa, H, (size_t)H * H, w.YT, sH);
      g.bias = w.wo2; g.sBias = H;
      if ((rc = launch_gemm(g, NN, Kn, st))) return rc;
      g = mk(P, H, H, w.YT, H, sH, Wt.W2 + gW2, H, (size_t)H * H, w.QM, sH);
      g.mask = w.H1; g.sMask = sH;
      if ((rc = launch_gemm(g, NN, Kn, st))) return rc;
      if (want_od) {
        g = mk(P, C, H, w.QM, H, sH, Wt.W1 + gW1, C, (size_t)H * C, w.JIN, sC);
        if ((rc = launch_gemm(g, NN, Kn, st))) return rc;
        jac_kernel<<<dim3(gp, Kn), pb, 0, st>>>(DC, P, Kn, w.JIN, pe, w.od);
        DPN_LAUNCH_OK();
      }
      if (jac_fwd) {
        if ((rc = launch_fields(DC, 1, P, Kn, 0, 0, w.o, w.od, J.o + q0 * Kn, J.jac + q0 * Kn * 3, st))) return rc;
        continue;
      }
      if (pde) {
        residual_kernel<<<(P + 255) / 256, 256, 0, st>>>(DC, P, w.o, w.od, J.pts->f + q0, inv_n, seed_scale,
                                                         J.out->loss_terms + (size_t)b * 6, w.dov, w.dod,
                                                         J.out->vals ? J.out->vals + q0 * 6 : nullptr,
                                                         J.out->jac ? J.out->jac + q0 * 18 : nullptr, 0, 0);
        DPN_LAUNCH_OK();
        if (J.margin && (rc = launch_margin(1, P, 0, 0, w.o, J.margin->target + q0 * 6, *J.margin, inv_n, seed_scale, J.margin->loss + b,
                                            w.dov, J.margin->o ? J.margin->o + q0 * 6 : nullptr, st)))
          return rc;
      } else {
        if ((rc = launch_seed_in(DC, 1, P, Kn, 0, 0, J.d_o ? J.d_o + q0 * Kn : nullptr, J.d_jac ? J.d_jac + q0 * Kn * 3 : nullptr,
                                 seed_scale, w.dov, tangent ? w.dod : nullptr, st)))
          return rc;
      }
      if (!want_bwd) continue;
      const DpnGrads& G = *J.grads;
      // backward inputs and the combined tangent row
      bwd_in_kernel<<<dim3(gp, Kn), pb, 0, st>>>(DC, P, Kn, pe, w.pe6, w.dov, tangent ? w.dod : nullptr, w.JIN, w.ZP, w.ZD);
      DPN_LAUNCH_OK();
      if (tangent) {
        // G7: HT = (XT W1^T) * [H1>0], ZH = HT + dov H1
        g = mk(P, H, C, w.JIN, C, sC, Wt.W1 + gW1, C, (size_t)H * C, w.HT, sH);
        g.mask = w.H1; g.sMask = sH; g.out2 = w.ZH; g.sOut2 = sH; g.addsrc = w.H1; g.sAdd = sH;
        g.rowscale = w.dov; g.sRow = 1; g.ldRow = Kn;
        if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
        // G8: CT = HT W2^T, ZC = CT + dov CC
        g = mk(P, H, H, w.HT, H, sH, Wt.W2 + gW2, H, (size_t)H * H, w.CT, sH);
        g.out2 = w.ZC; g.sOut2 = sH; g.addsrc = w.CC; g.sAdd = sH; g.rowscale = w.dov; g.sRow = 1; g.ldRow = Kn;
        if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
        // G9: GZ = (CT Wa^T) * [GG>0] + dov GG
        g = mk(P, H, H, w.CT, H, sH, Wt.Wa, H, (size_t)H * H, nullptr, 0);
        g.mask = w.GG; g.sMask = sH; g.out2 = w.GZ; g.sOut2 = sH; g.addsrc = w.GG; g.sAdd = sH;
        g.rowscale = w.dov; g.sRow = 1; g.ldRow = Kn;
        if ((rc = launch_gemm(g, NT, Kn, st))) return rc;
      } else {
        scale_rows_kernel<<<dim3(gp, Kn), pb, 0, st>>>(P, Kn, H, w.H1, w.dov, w.ZH); DPN_LAUNCH_OK();
        scale_rows_kernel<<<dim3(gp, Kn), pb, 0, st>>>(P, Kn, H, w.CC, w.dov, w.ZC); DPN_LAUNCH_OK();
        scale_rows_kernel<<<dim3(gp, Kn), pb, 0, st>>>(P, Kn, H, w.GG, w.dov, w.GZ); DPN_LAUNCH_OK();
      }
      // weight gradients: K = points contractions (split-K, atomics)
      const int ks = max(1, min(64, P / 512));
      g = mk(H, C, P, w.QM, H, sH, w.ZP, C, sC, G.W1 + gW1, (size_t)H * C); g.ksplit = ks; g.atomic = 1;
      if ((rc = launch_gemm(g, TN, Kn, st))) return rc;
      g = mk(H, H, P, w.YT, H, sH, w.ZH, H, sH, G.W2 + gW2, (size_t)H * H); g.ksplit = ks; g.atomic = 1;
      if ((rc = launch_gemm(g, TN, Kn, st))) return rc;
      g = mk(H, H, P, w.UM, H, sH, w.ZC, H, sH, G.Wa, (size_t)H * H); g.ksplit = ks; g.atomic = 1;
      if ((rc = launch_gemm(g, TN, Kn, st))) return rc;
      g = mk(H, C, P, w.YT, H, sH, w.ZD, C, sC, G.Wd, (size_t)H * C); g.ksplit = ks; g.atomic = 1;
      if ((rc = launch_gemm(g, TN, Kn, st))) return rc;
      // bias gradients and the column sums of the folded layer
      const int rpb = 256;
      const dim3 cg((P + rpb - 1) / rpb, Kn);
      colsum_kernel<<<cg, 256, 0, st>>>(P, Kn, rpb, w.QM, w.dov, G.b1 + gb, nullptr, nullptr); DPN_LAUNCH_OK();
      colsum_kernel<<<cg, 256, 0, st>>>(P, Kn, rpb, w.YT, w.dov, G.b2 + gb, G.e + gb, G.bd); DPN_LAUNCH_OK();
      colsum_kernel<<<cg, 256, 0, st>>>(P, Kn, rpb, w.UM, w.dov, G.ba, nullptr, nullptr); DPN_LAUNCH_OK();
      colsum_kernel<<<cg, 256, 0, st>>>(P, Kn, rpb, w.ZC, nullptr, w.vc, nullptr, nullptr); DPN_LAUNCH_OK();
      colsum_kernel<<<cg, 256, 0, st>>>(P, Kn, rpb, w.GZ, nullptr, w.vg, nullptr, nullptr); DPN_LAUNCH_OK();
      sum_seed_kernel<<<dim3(min(64, (P + 255) / 256), Kn), 256, 0, st>>>(P, Kn, w.dov, w.sdo); DPN_LAUNCH_OK();
    }
  }
  if (want_bwd) {
    const DpnGrads& G = *J.grads;
    finalize_kernel<<<dim3(Kn, 8), 256, 0, st>>>(Wt.Wb, Wt.bb, Wt.wo, w.vc, w.vg, w.sdo, G.Wb, G.bb, G.wo, G.bo);
    DPN_LAUNCH_OK();
  }
  return 0;
}

// ---- launch wrappers shared with the tensor-core mode (dpn_tc.cu) ----------------------------------
int launch_prep(int B, int Kn, const DpnWeights& Wt, float* uvec, float* wo2, float* cst, float* bsum, cudaStream_t st) {
  prep_kernel<<<Kn, 256, 0, st>>>(B, Kn, Wt.Wb, Wt.bb, Wt.wo, Wt.bo, Wt.b2, Wt.bd, Wt.e, uvec, wo2, cst, bsum);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_residual(const DevConsts& DC, int B, int P, size_t srow, size_t sq, const float* o, const float* od, const float* f,
                    double inv_n, double seed_scale, double* loss6, float* dov, float* dod, float* vals, float* jac, cudaStream_t st) {
  residual_kernel<<<dim3((P + 255) / 256, B), 256, 0, st>>>(DC, P, o, od, f, inv_n, seed_scale, loss6, dov, dod, vals, jac, srow, sq);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_margin(int B, int P, size_t srow, size_t sq, const float* o, const float* target, const DpnMargin& M, double inv_n,
                  double seed_scale, double* loss, float* dov, float* o_out, cudaStream_t st) {
  margin_seed_kernel<<<dim3((P + 255) / 256, B), 256, 0, st>>>(P, o, target, M.beta, M.factor * inv_n / 6.0, seed_scale, loss, dov, o_out,
                                                               srow, sq);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_seed_in(const DevConsts& DC, int B, int P, int Kn, size_t srow, size_t sq, const float* d_o, const float* d_jac,
                   double seed_scale, float* dov, float* dod, cudaStream_t st) {
  seed_in_kernel<<<dim3((P + 255) / 256, B), 256, 0, st>>>(DC, P, Kn, d_o, d_jac, (float)seed_scale, seed_scale, dov, dod, srow, sq);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_fields(const DevConsts& DC, int B, int P, int Kn, size_t srow, size_t sq, const float* o, const float* od, float* o_out,
                  float* jac, cudaStream_t st) {
  fields_kernel<<<dim3((P + 255) / 256, B), 256, 0, st>>>(DC, P, Kn, o, od, o_out, jac, srow, sq);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_finalize(int Kn, const DpnWeights& Wt, const float* vc, const float* vg, const float* sdo, const DpnGrads& G,
                    cudaStream_t st) {
  finalize_kernel<<<dim3(Kn, 8), 256, 0, st>>>(Wt.Wb, Wt.bb, Wt.wo, vc, vg, sdo, G.Wb, G.bb, G.wo, G.bo);
  DPN_LAUNCH_OK();
  return 0;
}

}  // namespace f32
}  // namespace dpn
