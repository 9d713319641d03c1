// Row N2 of SURVEY 8(f): the query-point producer on the GPU.
// Replaces the CPU `xarray.DataArray.interp(x=..., y=..., t=...)` of dataset/physics_dataset.py:477-486 (interior points),
// :406-415 (margin points) and :567-576 (dense grid): point-wise trilinear interpolation of the normalised coarse
// (1 degree, 6-hourly) field stack at continuous (lon, lat, hour) queries, plus the Coriolis parameter of :521-526.
// Values only - the reference does not differentiate through this interpolation (SURVEY D1) and neither do we.
#include "dpn_fp32.cuh"

namespace dpn {

// Coordinates -> cell index and weights in fp64 (the fractional part of a cell coordinate ~64 needs more than fp32 to stay within
// 2e-6 of the fp64 reference); the 8 x 6 multiply-adds in fp32; the [N,6] output leaves through a shared-memory transpose so that
// every warp store covers 128 contiguous bytes.  The texels (6 floats = 24 bytes) are fetched with three 8-byte read-only loads
// from the L2-resident coarse stack.
// trilinear sample of one query point: acc[6] (NaN outside the stack)
__device__ __forceinline__ void sample_point(const DpnSampler& S, const float* __restrict__ base, float xv, float yv, float tv, float (&acc)[6]) {
  const double rx = 1.0 / (S.dx * S.cells_per_coarse), ry = 1.0 / (S.dy * S.cells_per_coarse), rt = 1.0 / S.t_step;
  const double gx = (double)xv * rx, gy = (double)yv * ry, gt = (double)tv * rt;
  // interval search of a regular grid; the last node belongs to the last interval (as scipy's interpn does)
  const int ix = min(max((int)floor(gx), 0), S.Wc - 2), iy = min(max((int)floor(gy), 0), S.Hc - 2);
  const int it = min(max((int)floor(gt), 0), S.Tt - 2);
  const float wx = (float)(gx - ix), wy = (float)(gy - iy), wt = (float)(gt - it);
  // Outside the coarse stack (or NaN coordinates) the reference's DataArray.interp yields NaN - scipy interpn(bounds_error=False,
  // fill_value=nan); clamping the cell while leaving the weights free would extrapolate silently, e.g. after a unit mix-up.
  constexpr double EPS = 1e-9;
  const bool inside = gx >= -EPS && gx <= (double)(S.Wc - 1) + EPS && gy >= -EPS && gy <= (double)(S.Hc - 1) + EPS &&
                      gt >= -EPS && gt <= (double)(S.Tt - 1) + EPS;
#pragma unroll
  for (int c = 0; c < 6; ++c) acc[c] = 0.f;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int dt_ = c >> 2, dy_ = (c >> 1) & 1, dx_ = c & 1;
    const float wgt = (dt_ ? wt : 1.f - wt) * (dy_ ? wy : 1.f - wy) * (dx_ ? wx : 1.f - wx);
    const float2* p = reinterpret_cast<const float2*>(base + (((size_t)(it + dt_) * S.Hc + (iy + dy_)) * S.Wc + (ix + dx_)) * 6);
    const float2 a = __ldg(p), bq = __ldg(p + 1), cq = __ldg(p + 2);     // one 24-byte texel: 6 variables
    acc[0] = fmaf(wgt, a.x, acc[0]); acc[1] = fmaf(wgt, a.y, acc[1]); acc[2] = fmaf(wgt, bq.x, acc[2]);
    acc[3] = fmaf(wgt, bq.y, acc[3]); acc[4] = fmaf(wgt, cq.x, acc[4]); acc[5] = fmaf(wgt, cq.y, acc[5]);
  }
  if (!inside) {
#pragma unroll
    for (int c = 0; c < 6; ++c) acc[c] = __int_as_float(0x7fc00000);
  }
}

__device__ __forceinline__ float coriolis(const DpnSampler& S, float yv) {
  const double lat = S.begin_lat + (double)yv / S.dy * S.deg_per_cell;
  return (float)(2.0 * S.omega) * sinf((float)(lat * (3.14159265358979323846 / 180.0)));
}

// Philox4x32-10 (Salmon et al., SC'11): counter-based, one 128-bit block per (key, counter)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}

// One thread per point: (optionally) draw it, (optionally) sample the coarse stack at it; the [N,6] output leaves through a
// shared-memory transpose so that every warp store covers 128 contiguous bytes.
__global__ void __launch_bounds__(256) query_kernel(const DpnQueryGen G, const int draw, const DpnSampler S, const float* __restrict__ coarse,
                                                    float* __restrict__ x, float* __restrict__ y, float* __restrict__ t,
                                                    float* __restrict__ coord_data, float* __restrict__ f) {
  __shared__ float stage[8][32 * 6];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Np = draw ? G.N : S.N;
  const long long total = (long long)(draw ? G.B : S.B) * Np;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < total;
  float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float xv = 0.f, yv = 0.f, tv = 0.f;
  if (valid) {
    const int b = (int)(i / Np);
    if (draw) {
      const unsigned long long ctr = (unsigned long long)(i - (long long)b * Np) + G.offset;
      const uint4 r = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)b, 0u),
                                    make_uint2((uint32_t)G.seed, (uint32_t)(G.seed >> 32)));
      if (G.on_grid) {
        xv = (float)((double)(uint32_t)(((unsigned long long)r.x * (unsigned)G.lon_size) >> 32) * G.dx);
        yv = (float)((double)(uint32_t)(((unsigned long long)r.y * (unsigned)G.lat_size) >> 32) * G.dy);
      } else {
        xv = (float)((double)(r.x >> 8) * (1.0 / 16777216.0) * (double)(G.lon_size - 1) * G.dx);
        yv = (float)((double)(r.y >> 8) * (1.0 / 16777216.0) * (double)(G.lat_size - 1) * G.dy);
      }
      tv = (float)((double)(uint32_t)(((unsigned long long)r.z * (unsigned)G.t_steps) >> 32) * G.dt);
      x[i] = xv; y[i] = yv; t[i] = tv;
    } else {
      xv = x[i]; yv = y[i]; tv = t[i];
    }
    if (coarse) sample_point(S, coarse + (size_t)b * S.Tt * S.Hc * S.Wc * 6, xv, yv, tv, acc);
  }
  if (coarse) {
#pragma unroll
    for (int c = 0; c < 6; ++c) stage[warp][lane * 6 + c] = acc[c];
    __syncwarp();
    const long long w0 = ((long long)blockIdx.x * blockDim.x + warp * 32) * 6;       // first output word of this warp
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const long long word = w0 + c * 32 + lane;
      if (word < total * 6) coord_data[word] = stage[warp][c * 32 + lane];
    }
    if (f && valid) f[i] = coriolis(S, yv);
  }
}

// Lattice inference (dpn_decoder_lattice): one thread per node of a chunk of every sample.  The node's coordinates are computed in
// fp64 and rounded once to fp32, then clamped into the validated fp32 box: with a spacing that is not representable the last node
// could otherwise land one ulp outside the coarse stack and sample NaN; at exact lattices the clamp changes nothing.  coord_data
// comes from the same sample_point as dpn_sample_field's and leaves through the same shared-memory transpose.
__global__ void __launch_bounds__(256) lattice_kernel(const LatticeJob L, const int b0, const int nb, const int p0, const int P,
                                                      float* __restrict__ x, float* __restrict__ y, float* __restrict__ t,
                                                      float* __restrict__ coord_data) {
  __shared__ float stage[8][32 * 6];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t total = (size_t)nb * P;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (i < total) {
    const size_t b = i / P, node = (size_t)p0 + (i - b * P);
    const size_t row = node / L.g.nx;
    const double ix = (double)(node - row * L.g.nx), iy = (double)(row % L.g.ny), it = (double)(row / L.g.ny);
    const float xv = fminf(fmaxf((float)__dadd_rn(L.g.x0, __dmul_rn(ix, L.g.sx)), L.lo[0]), L.hi[0]);
    const float yv = fminf(fmaxf((float)__dadd_rn(L.g.y0, __dmul_rn(iy, L.g.sy)), L.lo[1]), L.hi[1]);
    const float tv = fminf(fmaxf((float)__dadd_rn(L.g.t0, __dmul_rn(it, L.g.st)), L.lo[2]), L.hi[2]);
    x[i] = xv; y[i] = yv; t[i] = tv;
    sample_point(L.s, L.coarse + ((size_t)b0 + b) * L.s.Tt * L.s.Hc * L.s.Wc * 6, xv, yv, tv, acc);
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) stage[warp][lane * 6 + c] = acc[c];
  __syncwarp();
  const size_t w0 = ((size_t)blockIdx.x * blockDim.x + warp * 32) * 6;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const size_t word = w0 + c * 32 + lane;
    if (word < total * 6) coord_data[word] = stage[warp][c * 32 + lane];
  }
}

// out = o * std + mean, one thread per output word: the chunk's output is contiguous per sample, and so are the rows of o.
__global__ void __launch_bounds__(256) lattice_emit_kernel(const LatticeJob L, const int nb, const int P, const float* __restrict__ o,
                                                           const size_t srow, float* __restrict__ out, const size_t out_bstride) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, per = (size_t)P * 6;
  if (i >= (size_t)nb * per) return;
  const size_t b = i / per, r = i - b * per;
  const int k = (int)(r % 6);
  out[b * out_bstride + r] = __fadd_rn(__fmul_rn(o[b * srow * 6 + r], L.sd[k]), L.mu[k]);
}

int launch_lattice(const LatticeJob& L, int b0, int nb, int p0, int P, float* x, float* y, float* t, float* coord_data, cudaStream_t st) {
  const size_t total = (size_t)nb * P;
  lattice_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(L, b0, nb, p0, P, x, y, t, coord_data);
  DPN_LAUNCH_OK();
  return 0;
}

int launch_lattice_emit(const LatticeJob& L, int nb, int P, const float* o, size_t srow, float* out, size_t out_bstride, cudaStream_t st) {
  const size_t total = (size_t)nb * P * 6;
  lattice_emit_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(L, nb, P, o, srow, out, out_bstride);
  DPN_LAUNCH_OK();
  return 0;
}

int run_sampler(const DpnSampler& S, const float* coarse, const float* x, const float* y, const float* t,
                float* coord_data, float* f, cudaStream_t st) {
  const long long total = (long long)S.B * S.N;
  DpnQueryGen none;
  memset(&none, 0, sizeof(none));
  query_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(none, 0, S, coarse, const_cast<float*>(x), const_cast<float*>(y),
                                                                const_cast<float*>(t), coord_data, f);
  DPN_LAUNCH_OK();
  return 0;
}

int run_query_gen(const DpnQueryGen& G, const DpnSampler* S, const float* coarse, float* x, float* y, float* t,
                  float* coord_data, float* f, cudaStream_t st) {
  const long long total = (long long)G.B * G.N;
  DpnSampler none;
  memset(&none, 0, sizeof(none));
  query_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(G, 1, S ? *S : none, S ? coarse : nullptr, x, y, t, coord_data, f);
  DPN_LAUNCH_OK();
  return 0;
}

}  // namespace dpn
