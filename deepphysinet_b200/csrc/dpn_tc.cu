// The hot path on the 5th-generation tensor cores (tcgen05.mma kind::f16, fp32 accumulators in TMEM), weights streamed through
// shared memory with cp.async.bulk (UBLKCP) on mbarriers: pass1_ts_kernel / pass2z_kernel / wgrad2_kernel, templated on the number
// of operand planes PL.
//
//   * PL = 2, the SPLIT MODES (DPN_MODE_F16X3 - the default -, DPN_MODE_F16X3A, DPN_MODE_BF16X3): every operand - weight images,
//     activation tiles, workspace tiles - is kept as TWO 16-bit planes, hi = rn16(v) and lo = rn16(v - hi) (22 / 16 mantissa bits
//     together; fp16 tiles carry exact power-of-two scales), and a contraction issues three MMAs into the same fp32 accumulator:
//     lo*hi + hi*lo + hi*hi (two where one operand is the exact 0 / 1 ReLU mask).
//   * PL = 1, DPN_MODE_BF16: one bf16 plane, one MMA per contraction.
//
// A operands live in TENSOR MEMORY: two 256-column regions used as ping-pong accumulators that the epilogues convert IN PLACE into the
// next A operand while the next GEMM already runs on the converted blocks (DESIGN.md section 5).
//
// Executed algorithm (DESIGN.md section 3), per tile of 128 query points and per coordinate net:
//   pass 1  G1 a1 = PE W1^T            -> h1 = relu(a1+b1), mask m1
//           G2 c  = h1 W2^T + PE6 Wd^T -> c + (b2+bd+e);  o += 2wo.c
//           G3 a3 = c Wa^T             -> g = relu(a3+ba), o += u.g (u = Wb^T wo: out_fc folded through cat_fc1.fc.2), mask m3
//           G4 y  = (u*m3) Wa + 2wo = m3 (diag(u) Wa) + 2wo    reverse sweep of the scalar output: do/dc   (the bare mask is the A operand)
//           G5 q  = y W2, qm = q*m1    do/da1
//           G6 jin = qm W1             do/dPE  -> do/dz_c = jin . dPE_c   (the 3 Jacobian columns)
//   residual kernel (fp64, shared with the fp32 mode) -> loss terms + seeds dL/do, dL/d(do/dz_c)
//   pass 2  the Z-side rows  zp = dov PE + sum_c seed_c dPE_c, zd = dov PE6, zh = dov h1 + ht, zc = dov c + ct  as the FORWARD pass of the
//           combined row zp with frozen masks and dov-scaled biases (G7', G8'); gz = dov g + gt is never formed - its column sum
//           comes out of the dWa contraction
//   wgrad   dW1 = qm^T zp, dW2 = y^T zh, dWa = diag(u) (m3^T zc), dWd = y^T zd  : K = points contractions, MN-major operands
//   colsum  bias gradients and the two vectors the folded output layer needs (vc, vg)
//
// Every [128 x Kd] 16-bit operand tile ("blob") is stored in the layout (*) of dpn_umma.cuh in shared memory (and, 32 points at a
// time, in the workspace), so a tile written once by an epilogue is (a) the K-major A operand of the next GEMM and
// (b) an MN-major operand of the weight-gradient contraction, and moves with plain 1-D bulk copies.
#include <math.h>
#include <stdlib.h>

#include <atomic>

#include "dpn_tc.cuh"
#include "dpn_umma.cuh"

namespace dpn {
namespace tc {

using namespace umma;

constexpr int TP = 128;                       // points per tile = TMEM lanes
constexpr int BLOB_H = TP * H * 2;            // 65536  [128 x 256] bf16
constexpr int BLOB_C = TP * C * 2;            // 49152  [128 x 192] bf16
constexpr int CORE_STRIDE = TP * 16;          // 2048   bytes between k-cores of a 128-row blob
constexpr int STAGE_BYTES = 8192;             // one K=16 chunk (= one MMA) of a [256 x K] weight image
#ifndef DPN_REUSE_A
#define DPN_REUSE_A 1
#endif
constexpr bool REUSE_A = DPN_REUSE_A != 0;               // consecutive MMAs on the same shared-memory A tile share one fetch (A collector)
#ifndef DPN_CLUSTER
#define DPN_CLUSTER 2
#endif
constexpr int CLUSTER = DPN_CLUSTER;                     // CTAs (tiles of the same sample) sharing every weight chunk through one multicast L2 read
constexpr int AUX_BYTES = TP * 16 * 2;        // 4096   [128 x 16] 16-bit seed tile: col 0/1/2 = the three 16-bit terms of dov
constexpr int IMG_HC = H * C * 2;             // 98304
constexpr int IMG_HH = H * H * 2;             // 131072
constexpr int GEN_IMG = 2 * IMG_HC + 2 * IMG_HH;   // per (sample, net): W1, W1T, W2, W2T
constexpr int STA_IMG = IMG_HC + 2 * IMG_HH;       // per net: Wd, Wa, (diag(u) Wa)^T
// Workspace tile of one (net, point tile):  YT QM ZH ZC | ZP ZD | AUX | MASK.  Pass 2 runs as the forward pass of the combined row
// (DESIGN.md section 3) and needs only the ReLU mask m1 of pass 1 (256 bits per point) instead of the h1 / c / g tiles (3 x 1 KB per
// point), and the weight-gradient kernel builds its J operand [a3 > 0] from the m3 mask bits instead of reading a stored tile.
constexpr int NBLOB_H = 4, NBLOB_C = 2;
enum { B_YT = 0, B_QM, B_ZH, B_ZC };
constexpr int MASK_BYTES = 2 * TP * 32;       // [m1 | m3][128 rows][8 words]

// Sizes that depend on the number of operand planes PL (1: bf16; 2: hi + lo, bf16 or scaled fp16).  Planes of one tile are
// contiguous, in shared memory and in the workspace alike.
template <int PL>
struct Geo {
  static constexpr int BH = BLOB_H * PL, BC = BLOB_C * PL;       // workspace tiles: plane p at p * BLOB_H (p * BLOB_C)
  static constexpr int GEN = GEN_IMG * PL, STA = STA_IMG * PL;
  static constexpr size_t NET_TILE = (size_t)NBLOB_H * BH + (size_t)NBLOB_C * BC + AUX_BYTES + MASK_BYTES;
  // Epilogue warps: warps w and w + 4 share the TMEM lanes 32 (w % 4) .. +31 and split the 256 columns.  8 warps: 16 (column
  // quarters, 113 registers) and 12 (blocks split 3 / 3 / 2, pass 2) were measured and lose (DESIGN.md section 9).
  static constexpr int EW = 8;
  static constexpr int ET = EW * 32;                             // epilogue threads
  static constexpr int NB = 4;                                   // 32-column blocks per thread
  static constexpr int W_PROD = EW, W_MMA = EW + 1;              // producer / MMA-issuer warps
  static constexpr int THREADS = ET + 64;
};
enum { V_B1 = 0, V_BSUM, V_BA, V_U, V_WO2, V_C2, NVEC };   // epilogue vectors staged in shared memory per net (pass 1)

struct NetScales;

// Work-skipping switches for timing experiments exist only in debug builds (-DDPN_DEBUG_BUILD, never the shipped library)
#ifdef DPN_DEBUG_BUILD
#define DPN_DBG(w, bit) (((w).dbg_flags & (bit)) != 0)
#else
#define DPN_DBG(w, bit) false
#endif

struct Work {
  // geometry of this pass
  int B, Kn, T;            // samples, nets, tiles per sample
  int P;                   // valid points per sample in this pass
  int N;                   // points per sample of the whole call (stride of the per-point inputs)
  int p0;                  // first point of this pass
  // weight images
  const uint8_t* img_gen;  // [B][Kn][GEN_IMG]
  const uint8_t* img_sta;  // [Kn][STA_IMG]
  // epilogue vectors (fp32)
  const float *b1, *bsum;  // [B][Kn][H]
  const float *ba, *uvec, *wo2, *cst;   // [Kn][H], cst [Kn]
  // per-point
  const float* coord_data; // [B*N][6]
  const float* ref;        // [B*N][Kn] residual skip, or nullptr -> coord_data[:, k]
  uint8_t* pe_blob;        // [B*T][PL][BLOB_C]
  uint8_t* pe6_blob;       // [B*T][PL][BLOB_C]
  float* pet;              // [B*T][C][TP] fp32 transposed coordinate features
  uint8_t* blobs;          // [B][Kn][T][NET_TILE_BYTES]
  float *o, *od, *dov, *dod;   // [B*T*TP][Kn], [..][Kn][3]
  float *vc, *vg, *sdo;        // [Kn][H] column sums of zc / of the never-formed gz, and [Kn] sum of dov
  const NetScales* sc;         // [B][Kn] scaling plan (fp16 variant only)
  long long* phase_dbg;        // optional [kernel(2)][8] cycle counters (debug builds with DPN_PHASE_DEBUG=1), summed over CTAs
  int xfirst;                  // cross-first accumulation of G1 - G3 (DPN_MODE_F16X3A)
  int dbg_flags;               // DEBUG BUILDS ONLY (tools/build_debug.sh, DPN_DEBUG_FLAGS): 1 = no MMAs, 2 = empty epilogues, 4 = no tile stores
  float band[NF];
};

template <int PL>
__device__ __forceinline__ uint8_t* net_tile(const Work& w, int b, int k, int tl) {
  return w.blobs + (((size_t)b * w.Kn + k) * w.T + tl) * Geo<PL>::NET_TILE;
}
template <int PL> __host__ __device__ constexpr size_t off_h(int which) { return (size_t)which * Geo<PL>::BH; }
template <int PL> __host__ __device__ constexpr size_t off_zp() { return (size_t)NBLOB_H * Geo<PL>::BH; }
template <int PL> __host__ __device__ constexpr size_t off_zd() { return off_zp<PL>() + Geo<PL>::BC; }
template <int PL> __host__ __device__ constexpr size_t off_aux() { return off_zp<PL>() + 2 * Geo<PL>::BC; }
template <int PL> __host__ __device__ constexpr size_t off_mask() { return off_aux<PL>() + AUX_BYTES; }
template <int PL> __device__ __forceinline__ uint8_t* blob_h(uint8_t* nt, int which) { return nt + off_h<PL>(which); }
template <int PL> __device__ __forceinline__ uint8_t* blob_zp(uint8_t* nt) { return nt + off_zp<PL>(); }
template <int PL> __device__ __forceinline__ uint8_t* blob_zd(uint8_t* nt) { return nt + off_zd<PL>(); }
template <int PL> __device__ __forceinline__ uint8_t* blob_aux(uint8_t* nt) { return nt + off_aux<PL>(); }
template <int PL> __device__ __forceinline__ uint8_t* blob_mask(uint8_t* nt) { return nt + off_mask<PL>(); }

// ------------------------------------------------------------------------------------------------
// Small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 pack8(const float* v) {
  return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
__device__ __forceinline__ void unpack8(const uint4& q, float* v) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}
// 16-bit operand format: bf16 (8-bit mantissa, fp32 range) or fp16 (11-bit mantissa; callers pre-scale into its range)
template <bool F16>
__device__ __forceinline__ uint4 pack8f(const float* v) {
  if (F16) return make_uint4(pack_f16(v[0], v[1]), pack_f16(v[2], v[3]), pack_f16(v[4], v[5]), pack_f16(v[6], v[7]));
  return pack8(v);
}
template <bool F16>
__device__ __forceinline__ void unpack8f(const uint4& q, float* v) {
  if (F16) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
  } else {
    unpack8(q, v);
  }
}
// v - h for a 16-bit h (fp16 / bf16) without unpacking it: one mixed-precision FMA, h * (-1) + v (SASS: FHFMA with a half selector).
// Exact: h is v rounded to 11 / 8 significant bits, so the difference fits fp32.
template <bool F16>
__device__ __forceinline__ float resid16(const uint32_t h, const float v) {
  float d;
  if (F16) asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(d) : "h"((uint16_t)h), "h"((uint16_t)0xBC00), "f"(v));
  else asm("fma.rn.f32.bf16 %0, %1, %2, %3;" : "=f"(d) : "h"((uint16_t)h), "h"((uint16_t)0xBF80), "f"(v));
  return d;
}
// 8 fp32 values -> one 16-byte piece per plane: hi = rn16(v), lo = rn16(v - hi)  (v - hi is exact in fp32).
// Per pair of values: pack, two mixed-precision FMAs, pack - the epilogues of the split modes spend a third of their instructions here.
template <int PL, bool F16 = false>
__device__ __forceinline__ void split8(const float* v, uint4 (&q)[PL]) {
  q[0] = pack8f<F16>(v);
  if (PL == 2) {
    const uint32_t hw[4] = {q[0].x, q[0].y, q[0].z, q[0].w};
    float l[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      l[2 * i] = resid16<F16>(hw[i] & 0xFFFFu, v[2 * i]);
      l[2 * i + 1] = resid16<F16>(hw[i] >> 16, v[2 * i + 1]);
    }
    q[PL - 1] = pack8f<F16>(l);
  }
}
// store a piece into a tile whose planes are `plane` bytes apart: shared memory (sts8) / workspace, streaming (stg8)
template <int PL, bool F16 = false>
__device__ __forceinline__ void sts8(uint8_t* tile, uint32_t plane, uint32_t off, const float* v) {
  uint4 q[PL];
  split8<PL, F16>(v, q);
#pragma unroll
  for (int p = 0; p < PL; ++p) *reinterpret_cast<uint4*>(tile + p * plane + off) = q[p];
}
template <int PL, bool F16 = false>
__device__ __forceinline__ void stg8(uint8_t* tile, uint32_t plane, uint32_t off, const float* v) {
  uint4 q[PL];
  split8<PL, F16>(v, q);
#pragma unroll
  for (int p = 0; p < PL; ++p) __stcs(reinterpret_cast<uint4*>(tile + p * plane + off), q[p]);
}

// ------------------------------------------------------------------------------------------------
// Scaling plan of the fp16 variant (DPN_MODE_F16X3).  fp16 carries 11 mantissa bits but only 5 exponent bits, so every
// operand tile is multiplied by a power of two (exact to apply, exact to undo in the epilogue) that maps a RIGOROUS
// bound of its magnitude to 2^15.  Bounds come from row / column L1 norms of the weights (|PE| <= 1), so no value can
// overflow whatever the weights are; the 30 binades of fp16 below the bound absorb the looseness of the bounds.
// ------------------------------------------------------------------------------------------------
struct NetScales {                       // one per (sample, net)
  float sW1, sW2, sWd, sWa;              // weight images (a matrix and its transpose share the factor)
  float sWaU;                            // the image of diag(u) Wa (B operand of G4, whose A operand is the bare m3 mask)
  float sH1, sC, sG, sUM, sY, sQ;        // tiles written by pass 1: h1, c, g, u*m3, y, q*m1
  float M1, Mc, l1W1, l1W12;             // bounds of |h1|, |c|; L1(W1), L1(W1) L1(W2)
  float rowB;                            // max(1, L1(W1), L1(W1) L1(W2)): growth of the pass-2 tangent row over its chain
  float cap;                             // largest sH1 * sW2 this (sample, net) can carry (plan_kernel takes the min over samples)
  float sZP, sZH, sZC, sZD, sDV;         // Z-side tiles and the seed tile of the CURRENT chunk (zscale_kernel)
};
constexpr float S_PE = 1024.f;           // coordinate / data features lie in [-1, 1]
constexpr float F16_TOP = 32768.f;       // bound -> 2^15 (fp16 max is 65504)

__host__ __device__ __forceinline__ float pow2_floor(float x) {           // largest power of two <= x, clamped to [2^-80, 2^80]
  if (!(x > 8.2718061e-25f)) return 8.2718061e-25f;                       // 2^-80; also catches NaN / 0 / negatives
  if (x > 1.2089258e24f) return 1.2089258e24f;                            // 2^80
#ifdef __CUDA_ARCH__
  return __uint_as_float(__float_as_uint(x) & 0x7F800000u);
#else
  uint32_t u; memcpy(&u, &x, 4); u &= 0x7F800000u; float r; memcpy(&r, &u, 4); return r;
#endif
}
__device__ __forceinline__ float scale_for(float bound) { return pow2_floor(F16_TOP / fmaxf(bound, 1e-30f)); }
// element (r, 8*kc .. 8*kc+7) of a 128-row blob
__device__ __forceinline__ uint32_t piece_off(int r, int kc) { return (uint32_t)kc * CORE_STRIDE + (uint32_t)r * 16; }
// byte offset of the 16-byte piece (row r, k-core kc) of a workspace tile of the split modes: [point quarter][k-core][32 rows][16 B],
// KC k-cores per tile.  A 32-point quarter of a tile is contiguous, which is what lets the weight-gradient kernel stream quarter
// tiles through three stages (wgrad2_kernel); a warp (32 consecutive rows) still writes 512 contiguous bytes per 16-byte store.
__device__ __forceinline__ uint32_t gp_off(const int KC, const int r, const int kc) {
  return (uint32_t)(r >> 5) * (uint32_t)(KC * 512) + (uint32_t)kc * 512u + (uint32_t)(r & 31) * 16u;
}

// Column sums over the 32 rows a warp owns: after the exchange lane l holds sum_rows v[row][l].  31 shuffles.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool up = (lane & w) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float keep = up ? v[i + w] : v[i];
      const float send = up ? v[i] : v[i + w];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
    }
  }
  return v[0];
}

// sign / partner of d(PE_j)/dz: PE[6f+c] = sin, PE[6f+3+c] = cos  ->  dPE[6f+c] = +band cos, dPE[6f+3+c] = -band sin
#define DPE_PARTNER(J) (((J) % 6) < 3 ? (J) + 3 : (J)-3)
#define DPE_SIGN(J) (((J) % 6) < 3 ? 1.0f : -1.0f)

template <int PL> __device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(Geo<PL>::ET) : "memory"); }   // the epilogue warps only

// ------------------------------------------------------------------------------------------------
// The tcgen05 pipeline of pass1_ts_kernel and pass2z_kernel (DESIGN.md section 5).  A producer warp streams the K = 16 weight chunks
// through a ring of stages (`full` / `empty` mbarriers; with a cluster, every chunk is read from L2 once and multicast); one MMA warp
// issues split contractions; two 256-column TMEM regions are ping-pong accumulators that the epilogue warps convert in place, block
// by block, into the A operand of the next GEMM (`blk[4]`: block cb of both column halves is converted, one arrival per epilogue
// warp; `acc_ready[2]`: the GEMM into region 0 / 1 has completed).  A kernel brings its ring geometry (Cfg: NS stages of STAGE bytes,
// the weight chunk first, W_BYTES at most), its barrier struct (full, empty, blk, acc_ready, tmem_base and whatever only it needs)
// and its schedule.
// ------------------------------------------------------------------------------------------------
namespace pp {
constexpr uint32_t REGION = 256;                // TMEM columns of one ping-pong region
constexpr int A_PLANE = 2 * CORE_STRIDE;        // A slice [128 x 16] of one plane that rides in a stage behind its weight chunk: 4 KB
constexpr uint16_t MC_MASK = (uint16_t)((1u << CLUSTER) - 1);
static_assert(2 * REGION == 512 && REGION == H, "TMEM map: two [128 x 256] fp32 accumulators, each converted in place into 2 x 16-bit planes");
// which of the products of a split contraction a chunk issues: all three | exact A operand (B_lo, B_hi) | the two cross terms | the main term
enum { P_ALL = 0, P_EXACT = 1, P_CROSS = 2, P_MAIN = 3 };

// K-chunk order of a TS-form GEMM: the two epilogue warp groups finish block cb of their column halves together, i.e. chunks
// 2cb, 2cb+1 (half 0) and 8+2cb, 9+2cb (half 1)
__host__ __device__ constexpr int block_order(int i) { return ((i >> 2) << 1) + (i & 1) + ((i >> 1) & 1) * 8; }
// TMEM column of the hi plane of K-chunk c of a converted region a (the lo plane is 16 columns further)
__device__ __forceinline__ uint32_t chunk_col(uint32_t a, int c) { return a + 32u * (uint32_t)(c >> 1) + 8u * (uint32_t)(c & 1); }

// mbarrier wait; with the cycle counters on (debug builds, DPN_PHASE_DEBUG=1), the cycles spent waiting are added to acc
__device__ __forceinline__ void wait(uint64_t* bar, uint32_t parity, const bool timed, long long& acc) {
  if (timed) {
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += clock64() - t0;
  } else {
    mbar_wait(bar, parity);
  }
}

struct Block {
  uint32_t tmem;    // base of the 512 TMEM columns
  uint32_t rank;    // rank of this CTA in its cluster
};
// Thread 0 initialises the ring and hand-off barriers (a kernel initialises its own extra barriers before this call), the MMA warp
// allocates all 512 TMEM columns, and no CTA goes on before the barriers of every CTA of its cluster exist (multicast copies and
// commits arrive on them).
template <int PL, int NS, class Pipe>
__device__ __forceinline__ Block block_start(Pipe& p, const int tid, const int warp) {
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(&p.full[s], 1); mbar_init(&p.empty[s], CLUSTER); }
    for (int i = 0; i < 4; ++i) mbar_init(&p.blk[i], Geo<PL>::EW);
    mbar_init(&p.acc_ready[0], 1); mbar_init(&p.acc_ready[1], 1);
    fence_barrier_init();
  }
  if (warp == Geo<PL>::W_MMA) tmem_alloc(&p.tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (CLUSTER > 1) cluster_sync_all();
  return Block{p.tmem_base, cluster_ctarank()};
}
// No CTA leaves, and no TMEM column is freed, while MMAs or the multicast commits of a peer may still arrive
template <int PL>
__device__ __forceinline__ void block_end(const uint32_t tmem, const int warp) {
  tc_fence_before();
  __syncthreads();
  if (CLUSTER > 1) cluster_sync_all();
  if (warp == Geo<PL>::W_MMA) tmem_dealloc(tmem, 512);
}

// The weight ring as one warp (producer or MMA issuer) walks it: its stage and that stage's phase
template <int PL, class Cfg>
struct Ring {
  uint8_t* ring;
  uint64_t *full, *empty;
  uint32_t rank = 0;                // producer: this CTA's rank in the cluster
  uint64_t pol = 0;                 // producer: L2 policy of the weights (evict_last: every tile of a sample re-reads them)
  uint32_t s = 0, ph = 0;
  __device__ __forceinline__ void advance() { if (++s == Cfg::NS) { s = 0; ph ^= 1; } }
  // Producer: wait for the stage to be free, then one lane starts the copies into it: the weight chunk wsrc of wbytes (with a cluster,
  // each CTA fetches 1 / CLUSTER of it and multicasts that slice) and, if asrc, the A slice of the same K-chunk behind it.
  // hi_only: only the hi planes (the first half of the chunk, one plane of the A slice).
  __device__ __forceinline__ void put(const uint8_t* wsrc, uint32_t wbytes, const uint8_t* asrc, const bool hi_only = false) {
    if (hi_only) wbytes /= 2;
    const int a_planes = hi_only ? 1 : PL;
    mbar_wait(&empty[s], ph ^ 1);
    if (elect_one()) {
      uint8_t* stg = ring + s * Cfg::STAGE;
      mbar_arrive_expect_tx(&full[s], wbytes + (asrc ? a_planes * A_PLANE : 0));
      if (CLUSTER == 1) {
        bulk_g2s_hint(stg, wsrc, wbytes, &full[s], pol);
      } else {
        const uint32_t slice = wbytes / CLUSTER;
        bulk_g2s_mc_hint(stg + rank * slice, wsrc + rank * slice, slice, &full[s], MC_MASK, pol);
      }
      if (asrc) {
        for (int p = 0; p < a_planes; ++p) bulk_g2s_hint(stg + Cfg::W_BYTES + p * A_PLANE, asrc + p * BLOB_C, A_PLANE, &full[s], pol);
      }
    }
    advance();
  }
  // MMA issuer (elected lane): the stage is free once the MMAs issued so far have read it, in every CTA of the cluster
  __device__ __forceinline__ void release() { if (CLUSTER == 1) mma_commit(&empty[s]); else mma_commit_mc(&empty[s], MC_MASK); }
};

// The MMA warp: consumer of the ring and of the epilogues' converted blocks
template <int PL, bool F16, class Cfg>
struct Mma {
  Ring<PL, Cfg> ring;
  uint64_t *blk, *acc_ready;
  uint32_t ring_addr;               // shared-memory address of stage 0
  bool timed;
  bool no_mma;                      // debug builds: the barrier protocol without the MMAs
  uint32_t bp = 0;                  // parity of the blk barriers
  long long t_full = 0, t_epi = 0;  // cycles waited for weight chunks / for converted blocks

  // One K = 16 chunk: the weights of the next stage (N = Nn) against an A operand, into the accumulator at d.  PL = 2: lo*hi + hi*lo
  // + hi*hi (`part` selects a subset); PL = 1: one product.
  // TS form: A planes in tensor memory, hi at a_hi, lo at a_lo.
  __device__ __forceinline__ void ts(const uint32_t d, const int Nn, const uint32_t a_hi, const uint32_t a_lo, const uint32_t first, const int part = P_ALL) {
    chunk(Nn, [&](const uint32_t idesc, const uint64_t bd, const uint64_t bl) {
      if (PL == 1) {
        mma_ts(d, a_hi, bd, idesc, first);
      } else {
        if (part == P_ALL || part == P_CROSS) mma_ts(d, a_lo, bd, idesc, first);   // (an exact 16-bit A operand - the 0 / 1 mask of G4 - has no lo plane)
        if (part != P_MAIN) mma_ts(d, a_hi, bl, idesc, part == P_EXACT ? first : 1u);
        if (part != P_CROSS) mma_ts(d, a_hi, bd, idesc, part == P_MAIN ? first : 1u);
      }
    });
  }
  // SS form: A planes in shared memory, descriptor ad, the lo plane al_off (>> 4) further; in_stage: the A slice rides in the stage
  // behind the weight chunk, so ad is the descriptor of stage 0's slice.  The hi plane of A is fetched once for its two MMAs.
  __device__ __forceinline__ void ss(const uint32_t d, const int Nn, const uint64_t a0, const uint32_t al_off, const bool in_stage, const uint32_t first, const int part = P_ALL) {
    const uint64_t ad = a0 + (in_stage ? ring.s * (uint32_t)(Cfg::STAGE >> 4) : 0u), al = ad + al_off;
    chunk(Nn, [&](const uint32_t idesc, const uint64_t bd, const uint64_t bl) {
      if (PL == 1 || part == P_MAIN) {
        mma_bf16(d, ad, bd, idesc, first);
      } else {
        mma_bf16(d, al, bd, idesc, first);
        if (part == P_CROSS) {
          mma_bf16(d, ad, bl, idesc, 1u);
        } else {
          mma_f16_c<REUSE_A ? A_FILL : A_DISCARD>(d, ad, bl, idesc, 1u);
          mma_f16_c<REUSE_A ? A_LAST : A_DISCARD>(d, ad, bd, idesc, 1u);
        }
      }
    });
  }
  // K = 256 GEMM into d whose A operand is region a, converted in place by the running epilogue: each block as soon as it is converted
  __device__ __forceinline__ void gemm_ts(const uint32_t d, const uint32_t a, const int Nn, const bool accumulate, const int part = P_ALL) {
    for (int cb = 0; cb < 4; ++cb) {
      wait_blk(cb);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 2 * cb + (j & 1) + (j >> 1) * 8;              // block_order(4 cb + j)
        const uint32_t ah = chunk_col(a, c);
        ts(d, Nn, ah, ah + 16, (accumulate || cb > 0 || j > 0) ? 1u : 0u, part);
      }
    }
    bp ^= 1u;
  }
  __device__ __forceinline__ void wait_blk(const int cb) { wait(&blk[cb], bp, timed, t_epi); tc_fence_after(); }
  // the GEMM into `region` is complete once the MMAs issued so far are
  __device__ __forceinline__ void ready(const uint32_t region) { if (elect_one()) mma_commit(&acc_ready[region]); }

  template <class F>
  __device__ __forceinline__ void chunk(const int Nn, F&& mmas) {
    const uint32_t idesc = idesc_16(F16, Nn, 0, 0, 128);
    const uint64_t b_base = smem_desc(ring_addr, Nn * 16, 128);
    const uint32_t b_lo = (uint32_t)(Nn * 32) >> 4;
    wait(&ring.full[ring.s], ring.ph, timed, t_full);
    tc_fence_after();
    const uint64_t bd = b_base + ring.s * (uint32_t)(Cfg::STAGE >> 4), bl = bd + b_lo;
    if (elect_one()) {
      if (!no_mma) mmas(idesc, bd, bl);
      ring.release();
    }
    ring.advance();
  }
};

// An epilogue thread (point r of the tile = TMEM lane, one column half): its side of the hand-offs
template <int PL, bool F16>
struct Epi {
  uint64_t *blk, *acc_ready;
  uint32_t lane_base;               // this warp's TMEM lanes, column 0
  int r, lane;
  bool timed;
  bool no_stores;                   // debug builds: no workspace tile stores
  uint32_t ar0 = 0, ar1 = 0;        // waits on acc_ready[0] / [1] so far
  long long t_acc = 0;              // cycles waited for accumulators

  // waits for the GEMM into `region`; returns this thread's lane address of that region
  __device__ __forceinline__ uint32_t acc_wait(const uint32_t region) {
    const uint32_t par = (region ? ar1 : ar0) & 1u;
    wait(&acc_ready[region], par, timed, t_acc);
    if (region) ++ar1; else ++ar0;
    tc_fence_after();
    return lane_base + region * REGION;
  }
  // this warp's part of block cb is in tensor memory (proxy: and its generic-proxy stores to shared memory are visible to the tensor
  // core): one arrival per warp
  __device__ __forceinline__ void blk_done(const int cb, const bool proxy = false) {
    tmem_st_wait(); tc_fence_before();
    if (proxy) fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(&blk[cb]);
  }
  // 32 columns of this row (32-column block cg): split into the planes once, then -> the workspace tile blob (if any) and / or, with
  // to_a, IN PLACE over the accumulator block they came from (blk_addr): the next A operand
  __device__ __forceinline__ void emit(const int cg, const float (&v)[32], uint8_t* blob, const bool to_a, const uint32_t blk_addr) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
      uint4 pq[PL];
      split8<PL, F16>(v + qd * 8, pq);
      if (blob && !no_stores) {
        const uint32_t off = gp_off(32, r, cg * 4 + qd);
        __stcs(reinterpret_cast<uint4*>(blob + off), pq[0]);
        if (PL == 2) __stcs(reinterpret_cast<uint4*>(blob + BLOB_H + off), pq[PL - 1]);
      }
      hi[qd * 4 + 0] = pq[0].x; hi[qd * 4 + 1] = pq[0].y; hi[qd * 4 + 2] = pq[0].z; hi[qd * 4 + 3] = pq[0].w;
      lo[qd * 4 + 0] = pq[PL - 1].x; lo[qd * 4 + 1] = pq[PL - 1].y; lo[qd * 4 + 2] = pq[PL - 1].z; lo[qd * 4 + 3] = pq[PL - 1].w;
    }
    if (to_a) {
      tmem_st16(blk_addr, hi);
      if (PL == 2) tmem_st16(blk_addr + 16, lo);
    }
  }
};
}  // namespace pp

// ------------------------------------------------------------------------------------------------
// Pass 1 of the split modes: A operands in TENSOR MEMORY (DESIGN.md section 5).
// The A operand of every GEMM but G1 / G2b is written by the epilogues with tcgen05.st and read by the TS form of tcgen05.mma; the
// PE / PE6 tiles of G1 / G2b travel through the ring as K = 16 slices next to their weight chunks; tiles kept for the backward pass
// leave with streaming 16-byte stores from registers.  No activation buffer in shared memory -> the ring holds 9 stages of 24 KB.
//
// Tensor memory = two 256-column regions R0 | R1 used as PING-PONG accumulators with IN-PLACE conversion: the epilogue of GEMM j
// reads a 32-column block of the fp32 accumulator (32 outputs of this row) and writes the two 16-bit planes of the same 32 values
// back into the SAME 32 columns (hi -> columns +0..15, lo -> +16..31; K-chunk c of the next contraction = columns 32 (c / 2) +
// 8 (c % 2), lo 16 further).  GEMM j + 1 accumulates into the OTHER region and starts on a K-chunk as soon as the epilogue has
// converted that block (one mbarrier per block, weights streamed in block order), so the tensor pipe runs under the epilogue of
// the previous GEMM instead of after it; the K-chunks without a dependence on the epilogue (PE6 Wd^T of G2, G1 of the next net)
// are issued first.  tcgen05.mma executes in issue order, so a region that was the A operand of GEMM j is safe to be the
// accumulator of GEMM j + 1.
// ------------------------------------------------------------------------------------------------
namespace ts {
constexpr int NS_MAX = 16;
template <int PL>
struct Cfg {                                    // ring geometry for PL operand planes
  static constexpr int NS = PL == 2 ? 9 : 16;
  static constexpr int W_BYTES = PL * STAGE_BYTES;         // weight chunk [256 x 16]: 8 KB per plane, hi | lo  ([192 x 16]: 6 KB per plane)
  static constexpr int STAGE = W_BYTES + PL * pp::A_PLANE; // 24 KB / 12 KB
  static constexpr int SMEM = NS * STAGE + NVEC * H * 4 + TP * 4 * 4;
};
struct PipeTS {
  uint64_t full[NS_MAX], empty[NS_MAX];
  uint64_t blk[4];          // block cb of BOTH column halves of the next A operand is in tensor memory (one arrival per epilogue warp)
  uint64_t acc_ready[2];    // the GEMM accumulating into region 0 / 1 has completed
  uint64_t drained;         // the last epilogue of a net (which hands no operand on) has read its accumulator
  uint32_t tmem_base;
};
static_assert(Cfg<2>::SMEM + (int)sizeof(PipeTS) + 1024 <= 227 * 1024 && Cfg<1>::SMEM <= Cfg<2>::SMEM, "pass1_ts_kernel: ring + vectors + row sums + barriers must fit one SM's 227 KB");
}  // namespace ts

template <int PL, bool F16, bool XF>             // PL operand planes; XF: cross-first accumulation of G1 - G3 (DPN_MODE_F16X3A)
__global__ void __cluster_dims__(CLUSTER, 1, 1) __launch_bounds__(Geo<2>::THREADS, 1) pass1_ts_kernel(const Work w, const int sweep) {
  using TS = ts::Cfg<PL>;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ ts::PipeTS pipe;
  uint8_t* ring = smem;
  float* svec = reinterpret_cast<float*>(smem + TS::NS * TS::STAGE);
  float* rowsum = svec + NVEC * H;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int b = blockIdx.x / w.T, tl = blockIdx.x % w.T;
  const size_t g = blockIdx.x;
  if (tid == 0) mbar_init(&pipe.drained, Geo<PL>::EW);
  const pp::Block cta = pp::block_start<PL, TS::NS>(pipe, tid, warp);
  const uint32_t tmem = cta.tmem;
  // DPN_MODE_F16X3A: CROSS-FIRST accumulation of the three GEMMs that decide the ReLU masks (G1 -> m1; G2, G3 -> m3).  The tensor core adds every MMA
  // into the fp32 accumulator with round-toward-zero at the accumulator's CURRENT magnitude, so the 2 x 16 cross-term MMAs of a split
  // contraction cost as much accuracy as its 16 main-term MMAs when they are interleaved.  Issued FIRST - while the accumulator holds
  // only the 2^-11-times-smaller cross sums - their truncations vanish, and a pre-activation carries 16 instead of 48 truncations:
  // 4.6e-7 instead of 1.2e-6 rms relative error for K = 256 (a CUDA-core fp32 FMA chain: 2.9e-7; DESIGN.md section 6).  The price is
  // that the hi planes of these GEMMs' chunks are fetched twice and that their main terms cannot start under the running epilogue.
  // Only when a Jacobian / backward pass follows (sweep > 0): the values themselves are continuous in the masks.
  const bool xfirst = XF && sweep > 0;

  if (warp == Geo<PL>::W_PROD) {
    // ---------------- producer: weight chunks (multicast slices) + this tile's PE slices ----------------
    // (the main-term phase of a cross-first GEMM needs only the hi planes of its chunks and A slices: hi_only)
    pp::Ring<PL, TS> wr{ring, pipe.full, pipe.empty, cta.rank, l2_policy_evict_last()};
    const uint8_t* pe_src = w.pe_blob + g * Geo<PL>::BC;
    const uint8_t* pe6_src = w.pe6_blob + g * Geo<PL>::BC;
    for (int k = 0; k < w.Kn; ++k) {
      const uint8_t* gen = w.img_gen + ((size_t)b * w.Kn + k) * Geo<PL>::GEN;
      const uint8_t* sta = w.img_sta + (size_t)k * Geo<PL>::STA;
      const uint8_t *iW1 = gen, *iW1T = gen + PL * IMG_HC, *iW2 = gen + PL * 2 * IMG_HC, *iW2T = gen + PL * (2 * IMG_HC + IMG_HH);
      const uint8_t *iWd = sta, *iWa = sta + PL * IMG_HC, *iWaT = sta + PL * (IMG_HC + IMG_HH);
      // the MMA warp's order: G1 | G2b (PE6 slices: no dependence on an epilogue, issued first) | TS-form GEMMs in block order.
      // Cross-first GEMMs (G1 - G3 when masks matter, see the MMA warp) read every chunk twice: whole chunks for the cross terms,
      // then the hi planes again for the main terms.
      for (int c = 0; c < 12; ++c) wr.put(iW1 + (size_t)c * TS::W_BYTES, TS::W_BYTES, pe_src + (size_t)c * pp::A_PLANE);
      if (xfirst) for (int c = 0; c < 12; ++c) wr.put(iW1 + (size_t)c * TS::W_BYTES, TS::W_BYTES, pe_src + (size_t)c * pp::A_PLANE, true);
      for (int c = 0; c < 12; ++c) wr.put(iWd + (size_t)c * TS::W_BYTES, TS::W_BYTES, pe6_src + (size_t)c * pp::A_PLANE);
      for (int i = 0; i < 16; ++i) wr.put(iW2 + (size_t)pp::block_order(i) * TS::W_BYTES, TS::W_BYTES, nullptr);
      if (xfirst) {
        for (int c = 0; c < 12; ++c) wr.put(iWd + (size_t)c * TS::W_BYTES, TS::W_BYTES, pe6_src + (size_t)c * pp::A_PLANE, true);
        for (int c = 0; c < 16; ++c) wr.put(iW2 + (size_t)c * TS::W_BYTES, TS::W_BYTES, nullptr, true);
      }
      for (int i = 0; i < 16; ++i) wr.put(iWa + (size_t)pp::block_order(i) * TS::W_BYTES, TS::W_BYTES, nullptr);
      if (xfirst) for (int c = 0; c < 16; ++c) wr.put(iWa + (size_t)c * TS::W_BYTES, TS::W_BYTES, nullptr, true);
      if (sweep) {
        for (int i = 0; i < 16; ++i) wr.put(iWaT + (size_t)pp::block_order(i) * TS::W_BYTES, TS::W_BYTES, nullptr);
        for (int i = 0; i < 16; ++i) wr.put(iW2T + (size_t)pp::block_order(i) * TS::W_BYTES, TS::W_BYTES, nullptr);
        if (sweep > 1)
          for (int i = 0; i < 16; ++i) wr.put(iW1T + (size_t)pp::block_order(i) * (PL * 6144), PL * 6144, nullptr);
      }
    }
  } else if (warp == Geo<PL>::W_MMA) {
    // ---------------- MMA issuer ----------------
    pp::Mma<PL, F16, TS> mma{{ring, pipe.full, pipe.empty}, pipe.blk, pipe.acc_ready, smem_u32(ring), w.phase_dbg != nullptr, DPN_DBG(w, 1)};
    uint32_t dr = 0, cur = 0;
    const long long t_begin = clock64();
    const uint64_t a_base = smem_desc(smem_u32(ring) + TS::W_BYTES, CORE_STRIDE, 128);      // the A slice of stage 0
    // G over the PE / PE6 slices of the ring into region `cur`
    auto gemm_ss = [&](const int nchunks, const int part = pp::P_ALL, const bool accumulate = false) {
      for (int c = 0; c < nchunks; ++c) mma.ss(tmem + cur * pp::REGION, H, a_base, pp::A_PLANE >> 4, true, (accumulate || c > 0) ? 1u : 0u, part);
    };
    // G whose A operand is the other region, converted in place by the running epilogue: block by block
    auto gemm_ts = [&](const int Nn, const bool accumulate, const int part = pp::P_ALL) {
      mma.gemm_ts(tmem + cur * pp::REGION, tmem + (cur ^ 1u) * pp::REGION, Nn, accumulate, part);
    };
    // main terms of a cross-first K = 256 GEMM: every block of the A operand has arrived (its cross terms are in), natural chunk order
    auto gemm_ts_main = [&]() {
      const uint32_t d = tmem + cur * pp::REGION, a = tmem + (cur ^ 1u) * pp::REGION;
      for (int c = 0; c < 16; ++c) mma.ts(d, H, pp::chunk_col(a, c), pp::chunk_col(a, c) + 16, 1u, pp::P_MAIN);
    };
    auto ready = [&]() { mma.ready(cur); cur ^= 1u; };
    for (int k = 0; k < w.Kn; ++k) {
      if (xfirst) { gemm_ss(12, pp::P_CROSS); gemm_ss(12, pp::P_MAIN, true); } else gemm_ss(12);
      ready();                                                             // G1 (A = PE slices); its region was the A operand of the previous GEMM
      if (k > 0) {                                                         // the last epilogue of the previous net has drained this region
        pp::wait(&pipe.drained, dr & 1, mma.timed, mma.t_epi);
        ++dr; tc_fence_after();
      }
      if (xfirst) {                                                        // G2b (A = PE6 slices) + G2a (A = h1): all cross terms, then all main terms
        gemm_ss(12, pp::P_CROSS); gemm_ts(H, true, pp::P_CROSS); gemm_ss(12, pp::P_MAIN, true); gemm_ts_main(); ready();
      } else {
        gemm_ss(12); gemm_ts(H, true); ready();
      }
      if (xfirst) { gemm_ts(H, false, pp::P_CROSS); gemm_ts_main(); } else gemm_ts(H, false);
      ready();                                                             // G3 (A = c)
      if (sweep) {
        gemm_ts(H, false, pp::P_EXACT); ready();                             // G4 (A = the m3 mask, B = diag(u) Wa: two MMAs per chunk)
        gemm_ts(H, false); ready();                                        // G5 (A = y)
        if (sweep > 1) { gemm_ts(C, false); ready(); }                     // G6 (A = qm, N = 192)
      }
    }
    if (mma.timed && lane == 0) {
      atomicAdd((unsigned long long*)w.phase_dbg + 0, (unsigned long long)(clock64() - t_begin));
      atomicAdd((unsigned long long*)w.phase_dbg + 1, (unsigned long long)mma.t_full);
      atomicAdd((unsigned long long*)w.phase_dbg + 2, (unsigned long long)mma.t_epi);
    }
  } else if (warp < Geo<PL>::EW) {
    // ---------------- epilogue: thread = (point r, column half) ----------------
    constexpr int NB = Geo<PL>::NB;
    const int half = warp >> 2, r = (warp & 3) * 32 + lane, c0 = half * NB;
    pp::Epi<PL, F16> epi{pipe.blk, pipe.acc_ready, tmem + ((uint32_t)((warp & 3) * 32) << 16), r, lane, w.phase_dbg != nullptr, DPN_DBG(w, 4)};
    const int p_local = tl * TP + r;
    const bool valid = p_local < w.P;
    const size_t q = (size_t)b * w.N + w.p0 + p_local;
    const size_t row = g * TP + r;
    const float* pet = w.pet + g * (size_t)(C * TP) + r;
    const uint64_t pol_keep = l2_policy_evict_last();
    uint32_t cur = 0u;
    // this warp has read the last accumulator of the net: one arrival per warp
    auto net_done = [&]() { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(&pipe.drained); };
    const long long t_begin = clock64();
    // waits for the GEMM into the current region; returns this thread's lane address of that region and flips the region
    auto acc_wait = [&]() -> uint32_t {
      const uint32_t a = epi.acc_wait(cur);
      cur ^= 1u;
      return a;
    };
    if (half == 0) { rowsum[r * 4 + 0] = 0.f; rowsum[r * 4 + 1] = 0.f; rowsum[r * 4 + 2] = 0.f; rowsum[r * 4 + 3] = 0.f; }
    for (int k = 0; k < w.Kn; ++k) {
      uint8_t* nt = net_tile<PL>(w, b, k, tl);
      // fp16 variant: an accumulator carries (A tile scale) x (weight image scale); k1 .. k6 undo that AND apply the scale of the tile
      // the epilogue produces, and the bias vectors are staged pre-multiplied by the same power of two (exact), so that
      // value -> next operand is ONE FMA per element:  h1 sH1 = max(acc k1 + b1 sH1, 0),  c sC = acc k2 + bsum sC,  y sY = acc k4 + 2wo sY
      float k1 = 1.f, k2 = 1.f, i3 = 1.f, k4 = 1.f, i5 = 1.f, i6 = 1.f, sH1 = 1.f, sC = 1.f, sY = 1.f;
      if (F16) {
        const NetScales t = w.sc[b * w.Kn + k];
        sH1 = t.sH1; sC = t.sC; sY = t.sY;
        k1 = sH1 / (S_PE * t.sW1); k2 = sC / (t.sH1 * t.sW2); i3 = 1.f / (t.sC * t.sWa); k4 = sY / t.sWaU;
        i5 = t.sQ / (t.sY * t.sW2); i6 = 1.f / (t.sQ * t.sW1);
      }
      epi_bar<PL>();
      if (tid < H) {                                                   // V_B1: b1 sH1 | V_BSUM: bsum sC | V_BA, V_U | V_WO2: 2wo / sC (epilogue 2) | V_C2: 2wo sY (epilogue 4)
        const size_t vb = ((size_t)b * w.Kn + k) * H, vk = (size_t)k * H;
        const float wo2 = __ldg(w.wo2 + vk + tid);
        svec[V_B1 * H + tid] = __ldg(w.b1 + vb + tid) * sH1;
        svec[V_BSUM * H + tid] = __ldg(w.bsum + vb + tid) * sC;
        svec[V_BA * H + tid] = __ldg(w.ba + vk + tid);
        svec[V_U * H + tid] = __ldg(w.uvec + vk + tid);
        svec[V_WO2 * H + tid] = wo2 * (1.f / sC);
        svec[V_C2 * H + tid] = wo2 * sY;
      }
      epi_bar<PL>();
      uint32_t m1w[NB];
#pragma unroll
      for (int i = 0; i < NB; ++i) m1w[i] = 0u;
      // ---- epilogue 1: h1 = relu(a1 + b1) ----
      uint32_t ra = acc_wait();
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(ra + cg * 32, v);
        uint32_t bits = 0;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(svec + V_B1 * H + cg * 32 + j4 * 4);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a = F16 ? fmaf(v[j4 * 4 + e], k1, bb[e]) : v[j4 * 4 + e] + bb[e];      // a1 sH1
            bits |= (a > 0.f ? 1u : 0u) << (j4 * 4 + e);
            v[j4 * 4 + e] = fmaxf(a, 0.f);
          }
        }
#pragma unroll
        for (int i = 0; i < NB; ++i) m1w[i] = (cb == i) ? bits : m1w[i];
        epi.emit(cg, v, nullptr, true, ra + cg * 32);                     // h1 itself is not kept: pass 2 needs only its mask
        epi.blk_done(cb);
      }
      // ---- epilogue 2: c = acc + (b2 + bd + e);  oc = 2wo.c ----
      float os0 = 0.f, os1 = 0.f;
      ra = acc_wait();
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(ra + cg * 32, v);
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(svec + V_BSUM * H + cg * 32 + j4 * 4);
          const float4 wv = *reinterpret_cast<const float4*>(svec + V_WO2 * H + cg * 32 + j4 * 4);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w}, ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float cc = F16 ? fmaf(v[j4 * 4 + e], k2, bb[e]) : v[j4 * 4 + e] + bb[e];     // c sC; ww = 2wo / sC
            if (e & 1) os1 = fmaf(ww[e], cc, os1); else os0 = fmaf(ww[e], cc, os0);
            v[j4 * 4 + e] = cc;
          }
        }
        epi.emit(cg, v, nullptr, true, ra + cg * 32);
        epi.blk_done(cb);
      }
      // ---- epilogue 3: g = relu(a3 + ba);  o = oc + u.g + cst + ref;  the mask m3 = [a3 > 0] is the A operand of G4 ----
      uint32_t m3w[NB];
#pragma unroll
      for (int i = 0; i < NB; ++i) m3w[i] = 0u;
      ra = acc_wait();
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(ra + cg * 32, v);
        uint32_t bits = 0u;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(svec + V_BA * H + cg * 32 + j4 * 4);
          const float4 uv = *reinterpret_cast<const float4*>(svec + V_U * H + cg * 32 + j4 * 4);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w}, uu[4] = {uv.x, uv.y, uv.z, uv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            const float a = F16 ? fmaf(v[j], i3, bb[e]) : v[j] + bb[e];
            const float gg = fmaxf(a, 0.f);
            if (e & 1) os1 = fmaf(uu[e], gg, os1); else os0 = fmaf(uu[e], gg, os0);
            bits |= (a > 0.f ? 1u : 0u) << j;
          }
        }
#pragma unroll
        for (int i = 0; i < NB; ++i) m3w[i] = (cb == i) ? bits : m3w[i];
        if (sweep) {                                                  // the mask as ONE exact 16-bit plane (1.0 / 0) over the accumulator block
          constexpr uint32_t ONE = F16 ? 0x3C00u : 0x3F80u;
          uint32_t mk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) mk[i] = (((bits >> (2 * i)) & 1u) ? ONE : 0u) | (((bits >> (2 * i + 1)) & 1u) ? (ONE << 16) : 0u);
          tmem_st16(ra + cg * 32, mk);
          epi.blk_done(cb);
        }
      }
      if (!sweep) net_done();
      if (sweep) {                                                     // the two ReLU masks of this (net, tile): all pass 2 needs of h1 / c / g
        uint4* mk = reinterpret_cast<uint4*>(blob_mask<PL>(nt));
        static_assert(NB == 4, "one uint4 of mask words per thread");
        mk[r * 2 + half] = make_uint4(m1w[0], m1w[1], m1w[2], m1w[3]);
        mk[(TP + r) * 2 + half] = make_uint4(m3w[0], m3w[1], m3w[2], m3w[3]);
      }
      atomicAdd(rowsum + r * 4, os0 + os1);
      epi_bar<PL>();
      if (half == 0) {
        if (valid) w.o[row * w.Kn + k] = rowsum[r * 4] + __ldg(w.cst + k) + (w.ref ? __ldg(w.ref + q * w.Kn + k) : __ldg(w.coord_data + q * 6 + k));
        rowsum[r * 4] = 0.f;
      }
      if (!sweep) continue;
      // ---- epilogue 4: y = acc + 2wo ----
      ra = acc_wait();
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(ra + cg * 32, v);
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 wv = *reinterpret_cast<const float4*>(svec + V_C2 * H + cg * 32 + j4 * 4);      // 2wo sY
          const float ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) v[j4 * 4 + e] = F16 ? fmaf(v[j4 * 4 + e], k4, ww[e]) : v[j4 * 4 + e] + ww[e];
        }
        epi.emit(cg, v, blob_h<PL>(nt, B_YT), true, ra + cg * 32);
        epi.blk_done(cb);
      }
      // ---- epilogue 5: qm = acc * m1 ----
      ra = acc_wait();
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(ra + cg * 32, v);
        uint32_t bits = 0u;
#pragma unroll
        for (int i = 0; i < NB; ++i) bits = (cb == i) ? m1w[i] : bits;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((bits >> j) & 1u) ? (F16 ? v[j] * i5 : v[j]) : 0.f;
        epi.emit(cg, v, blob_h<PL>(nt, B_QM), sweep > 1, ra + cg * 32);
        if (sweep > 1) epi.blk_done(cb);
      }
      if (sweep < 2) { net_done(); continue; }
      // ---- epilogue 6: do/dz_c = sum_j jin_j dPE_j  (j % 3 == c); N = 192: each half takes one 96-column group ----
      ra = acc_wait();
      float dz[3] = {0.f, 0.f, 0.f};
      {
        const uint32_t a6 = ra + half * 96;
        const float bsel = half ? 1.f : 0.f;
#pragma unroll
        for (int ib = 0; ib < 3; ++ib) {
          float pp[32], v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) pp[j] = ldg_f32_hint(pet + (size_t)(half * 96 + DPE_PARTNER(ib * 32 + j)) * TP, pol_keep);
          tmem_ld32(a6 + ib * 32, v);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int Jl = ib * 32 + j;
            const float bnd = bsel * w.band[16 + Jl / 6] + (1.f - bsel) * w.band[Jl / 6];
            dz[Jl % 3] = fmaf(DPE_SIGN(Jl) * bnd * v[j], pp[j], dz[Jl % 3]);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) atomicAdd(rowsum + r * 4 + 1 + c, F16 ? dz[c] * i6 : dz[c]);
      net_done();
      epi_bar<PL>();
      if (half == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if (valid) w.od[(row * w.Kn + k) * 3 + c] = rowsum[r * 4 + 1 + c];
          rowsum[r * 4 + 1 + c] = 0.f;
        }
      }
    }
    if (epi.timed && tid == 0) {
      const long long tot = clock64() - t_begin;
      atomicAdd((unsigned long long*)w.phase_dbg + 4, (unsigned long long)tot);
      atomicAdd((unsigned long long*)w.phase_dbg + 5, (unsigned long long)epi.t_acc);
      atomicAdd((unsigned long long*)w.phase_dbg + 7, (unsigned long long)(tot - epi.t_acc));
      atomicAdd((unsigned long long*)w.phase_dbg + 6, 1ull);
    }
  }
  pp::block_end<PL>(tmem, warp);
}

// 8 consecutive values of a stored tile: sum of its planes
template <int PL, bool F16 = false>
__device__ __forceinline__ void unpack_planes(const uint4 (&q)[PL], float* v) {
  unpack8f<F16>(q[0], v);
  if (PL == 2) {
    float l[8];
    unpack8f<F16>(q[PL - 1], l);
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] += l[e];
  }
}

// ------------------------------------------------------------------------------------------------
// Pass 2 of the split modes as the FORWARD PASS OF THE COMBINED ROW (DESIGN.md section 3).
// The Z-side operands of the weight gradients are  zh = dov h1 + ht,  zc = dov c + ct,  gz = dov g + gt  with the tangent chain
// ht = (xt W1^T) m1, ct = ht W2^T, gt = (ct Wa^T) m3.  Because h1 = m1 (PE W1^T + b1), c = h1 W2^T + PE6 Wd^T + bsum and
// g = m3 (c Wa^T + ba) are (masked) affine in their inputs, the sums collapse:
//        zh = m1 ( zp W1^T + dov b1 )            zp = dov PE + xt   (the operand of dW1, computed by the prologue anyway)
//        zc = zh W2^T + zd Wd^T + dov bsum       zd = dov PE6       (the operand of dWd)
//        gz = m3 ( zc Wa^T + dov ba )
// i.e. pass 2 is pass 1's value chain applied to the row zp with the FROZEN masks and dov-scaled biases.  It needs from pass 1
// one bit mask per point (32 bytes) instead of the h1 / c / g tiles (3 KB), no separate tangent row, and every tile it produces
// is at once the next A operand and the stored wgrad operand (one split instead of two).
// gz itself is never formed: it enters the gradients only through its column sum vg = sum_p gz (dWb, dwo), and
//        vg[j] = sum_i Wa[j,i] S[j,i] + ba[j] sum_p m3[p,j] dov[p],     S = m3^T zc
// where S is the contraction the weight-gradient kernel runs anyway for dWa = diag(u) S (wgrad2_kernel, layer 2) - so the third
// GEMM of the chain (zc Wa^T, K = 256) and its epilogue are not executed at all.
// Structure = pass1_ts_kernel: two 256-column TMEM regions as ping-pong accumulators, converted in place into the next A operand,
// the next GEMM starting block by block under the running epilogue.  Per net: the prologue writes zp into R1 (hi planes columns
// [0,96), lo [96,192)) while G7' (-> R0) consumes it; epilogue 7 converts R0 into zh while G8' (-> R1, first the K = 192 part whose
// A operand zd is staged in shared memory, 96 KB, layout (*)) consumes it; epilogue 8 reads R1 (zc -> workspace, column sums) and
// the next net's prologue follows in the same threads.  7 x 16 KB weight ring.
// ------------------------------------------------------------------------------------------------
namespace p2z {
enum { V2_B1 = 0, V2_BSUM, NV2 };
constexpr int NS_MAX = 14;
template <int PL>
struct Cfg {
  static constexpr int NS = PL == 2 ? 7 : 14;
  static constexpr int W_BYTES = PL * STAGE_BYTES;       // one K = 16 chunk of a [256 x K] image: 8 KB per plane, hi | lo
  static constexpr int STAGE = W_BYTES;
  static constexpr int ZD_BYTES = PL * BLOB_C;           // zd staging: one [128 x 192] tile per plane, layout (*)
  static constexpr int SMEM = NS * STAGE + ZD_BYTES + NV2 * H * 4 + H * 4 + 16;        // + column sums of zc + sum of dov
};
constexpr uint32_t ZP_LO = 96;                 // zp planes inside TMEM region R1: hi [0,96) | lo [96,192)
struct PipeZ {
  uint64_t full[NS_MAX], empty[NS_MAX];
  uint64_t blk[4];          // block i of both column halves of the next A operand is in tensor memory (one arrival per epilogue warp)
  uint64_t acc_ready[2];    // the GEMM accumulating into region 0 / 1 has completed
  uint32_t tmem_base;
};
// K-chunks of zp (K = 192) complete after prologue iteration i of both halves: a half writes 24 columns = 1.5 chunks per iteration
__host__ __device__ constexpr int zp_first(int i) { return i == 0 ? 0 : i == 1 ? 1 : i == 2 ? 3 : 4; }
__host__ __device__ constexpr int zp_count(int i) { return (i & 1) ? 2 : 1; }
static_assert(Cfg<2>::SMEM + (int)sizeof(PipeZ) + 1024 <= 227 * 1024 && Cfg<1>::SMEM <= Cfg<2>::SMEM, "pass2z_kernel: ring + zd tile + vectors must fit one SM's 227 KB");
}  // namespace p2z

template <int PL, bool F16>
__global__ void __cluster_dims__(CLUSTER, 1, 1) __launch_bounds__(Geo<2>::THREADS, 1) pass2z_kernel(const Work w) {
  using PZ = p2z::Cfg<PL>;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ p2z::PipeZ pipe;
  uint8_t* ring = smem;
  uint8_t* zdt = smem + PZ::NS * PZ::STAGE;
  float* svec = reinterpret_cast<float*>(zdt + PZ::ZD_BYTES);
  float* csum = svec + p2z::NV2 * H;                               // [H] + sdo
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int b = blockIdx.x / w.T, tl = blockIdx.x % w.T;
  const size_t g = blockIdx.x;
  const pp::Block cta = pp::block_start<PL, PZ::NS>(pipe, tid, warp);
  const uint32_t tmem = cta.tmem;

  if (warp == Geo<PL>::W_PROD) {
    // ---------------- producer: weight chunks (multicast slices) ----------------
    pp::Ring<PL, PZ> wr{ring, pipe.full, pipe.empty, cta.rank, l2_policy_evict_last()};
    for (int k = 0; k < w.Kn; ++k) {
      const uint8_t* gen = w.img_gen + ((size_t)b * w.Kn + k) * Geo<PL>::GEN;
      const uint8_t* sta = w.img_sta + (size_t)k * Geo<PL>::STA;
      const uint8_t *iW1 = gen, *iW2 = gen + PL * 2 * IMG_HC, *iWd = sta;
      // the MMA warp's order: G7' in prologue-block order | zd Wd^T (no dependence on an epilogue) | G8' in block order
      for (int i = 0; i < 4; ++i)
        for (int h = 0; h < 2; ++h)
          for (int j = 0; j < p2z::zp_count(i); ++j) wr.put(iW1 + (size_t)(6 * h + p2z::zp_first(i) + j) * PZ::W_BYTES, PZ::W_BYTES, nullptr);
      for (int c = 0; c < 12; ++c) wr.put(iWd + (size_t)c * PZ::W_BYTES, PZ::W_BYTES, nullptr);
      for (int i = 0; i < 16; ++i) wr.put(iW2 + (size_t)pp::block_order(i) * PZ::W_BYTES, PZ::W_BYTES, nullptr);
    }
  } else if (warp == Geo<PL>::W_MMA) {
    // ---------------- MMA issuer ----------------
    pp::Mma<PL, F16, PZ> mma{{ring, pipe.full, pipe.empty}, pipe.blk, pipe.acc_ready, smem_u32(ring), w.phase_dbg != nullptr, false};
    const long long t_begin = clock64();
    const uint64_t zd_base = smem_desc(smem_u32(zdt), CORE_STRIDE, 128);
    constexpr uint32_t zd_lo = BLOB_C >> 4, zd_step = (2 * CORE_STRIDE) >> 4;
    const uint32_t R0 = tmem, R1 = tmem + pp::REGION;
    for (int k = 0; k < w.Kn; ++k) {
      for (int i = 0; i < 4; ++i) {                                        // G7' = zp W1^T -> R0, under the prologue
        mma.wait_blk(i);
        for (int h = 0; h < 2; ++h)
          for (int j = 0; j < p2z::zp_count(i); ++j) {
            const uint32_t c = 6 * h + p2z::zp_first(i) + j;
            mma.ts(R0, H, R1 + 8u * c, R1 + p2z::ZP_LO + 8u * c, (i > 0 || h > 0 || j > 0) ? 1u : 0u);
          }
      }
      mma.bp ^= 1u;
      mma.ready(0);
      for (int c = 0; c < 12; ++c) mma.ss(R1, H, zd_base + (uint32_t)c * zd_step, zd_lo, false, c > 0 ? 1u : 0u);   // G8' = zd Wd^T (zd: shared memory, complete with the prologue)
      mma.gemm_ts(R1, R0, H, true); mma.ready(1);                          //       + zh W2^T, under epilogue 7
    }
    if (mma.timed && lane == 0) {
      atomicAdd((unsigned long long*)w.phase_dbg + 8, (unsigned long long)(clock64() - t_begin));
      atomicAdd((unsigned long long*)w.phase_dbg + 9, (unsigned long long)mma.t_full);
      atomicAdd((unsigned long long*)w.phase_dbg + 10, (unsigned long long)mma.t_epi);
    }
  } else if (warp < Geo<PL>::EW) {
    // ---------------- prologue + epilogues: thread = (point r, column half) ----------------
    constexpr int NB = Geo<PL>::NB;
    const int half = warp >> 2, r = (warp & 3) * 32 + lane, c0 = half * NB;
    pp::Epi<PL, F16> epi{pipe.blk, pipe.acc_ready, tmem + ((uint32_t)((warp & 3) * 32) << 16), r, lane, w.phase_dbg != nullptr, false};
    const size_t row = g * TP + r;
    const float* pet = w.pet + g * (size_t)(C * TP) + r;
    const uint8_t* pe6 = w.pe6_blob + g * Geo<PL>::BC;
    const uint64_t pol_keep = l2_policy_evict_last();
    const uint32_t R0 = epi.lane_base, R1 = epi.lane_base + pp::REGION;
    long long t_pro = 0;
    const long long t_begin = clock64();
    const bool timed = epi.timed;
    for (int i = tid; i < H + 4; i += Geo<PL>::ET) csum[i] = 0.f;
    for (int k = 0; k < w.Kn; ++k) {
      uint8_t* nt = net_tile<PL>(w, b, k, tl);
      epi_bar<PL>();                                                   // previous net's vectors / column sums are flushed
      if (tid < H) {
        const size_t vb = ((size_t)b * w.Kn + k) * H;
        svec[p2z::V2_B1 * H + tid] = __ldg(w.b1 + vb + tid);
        svec[p2z::V2_BSUM * H + tid] = __ldg(w.bsum + vb + tid);
      }
      epi_bar<PL>();
      const float dv = w.dov[row * w.Kn + k];
      float dd[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) dd[c] = w.dod[(row * w.Kn + k) * 3 + c];          // zero for the values-only backward
      const uint4 m1q = __ldg(reinterpret_cast<const uint4*>(blob_mask<PL>(nt)) + r * 2 + half);
      const uint32_t m1w[4] = {m1q.x, m1q.y, m1q.z, m1q.w};
      // fp16 variant: every tile carries one power-of-two scale per (sample, net) (zscale_kernel); accumulators carry
      // (A tile scale) x (weight image scale) and i7 / i8 undo that
      // zd exists twice: the stored tile (wgrad operand of dWd) with its own scale sZD, and the A operand of G8' whose scale is tied
      // to the accumulator it shares with zh W2^T: sZH sW2 = sZDa sWd, and plan_kernel made sH1 sW2 = S_PE sWd  =>  sZDa = sZH S_PE / sH1
      float sZP = 1.f, sZH = 1.f, sZC = 1.f, sZD = 1.f, sZDa = 1.f, sDV = 1.f, i7 = 1.f, i8 = 1.f;
      if (F16) {
        const NetScales t = w.sc[b * w.Kn + k];
        sZP = t.sZP; sZH = t.sZH; sZC = t.sZC; sZD = t.sZD; sDV = t.sDV;
        sZDa = t.sZH * (S_PE / t.sH1);
        i7 = (1.f / t.sZP) * (1.f / t.sW1); i8 = (1.f / t.sZH) * (1.f / t.sW2);
      }
      // the scale of the tile an epilogue produces is folded into its FMA (powers of two: exact): zh sZH = m1 (acc k7 + (dov sZH) b1), ...
      const float k7 = i7 * sZH, k8 = i8 * sZC, dvH = dv * sZH, dvC = dv * sZC, dvP = dv * sZP, inv_sZC = 1.f / sZC;
      const float ddP[3] = {dd[0] * sZP, dd[1] * sZP, dd[2] * sZP};
      // seed tile for the bias-gradient MMAs of the wgrad kernel: col 0/1/2 = dov split into three 16-bit terms, rest 0
      if (half == 0) {
        float a8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (F16) {
          const float x = dv * sDV;
          a8[0] = __half2float(__float2half_rn(x));
          a8[1] = __half2float(__float2half_rn(x - a8[0]));
          a8[2] = (x - a8[0]) - a8[1];
        } else {
          a8[0] = __uint_as_float(__float_as_uint(dv) & 0xFFFF0000u);
          a8[1] = __uint_as_float(__float_as_uint(dv - a8[0]) & 0xFFFF0000u);
          a8[2] = (dv - a8[0]) - a8[1];
        }
        __stcs(reinterpret_cast<uint4*>(blob_aux<PL>(nt) + gp_off(2, r, 0)), pack8f<F16>(a8));
        __stcs(reinterpret_cast<uint4*>(blob_aux<PL>(nt) + gp_off(2, r, 1)), make_uint4(0u, 0u, 0u, 0u));
      }
      // ---- prologue: zp = dov PE + sum_c dod_c dPE_c -> A operand (TMEM) + workspace;  zd = dov PE6 -> shared memory + workspace ----
      const long long t_p0 = timed ? clock64() : 0ll;
      // the loads of column group it + 1 are in flight while group it is processed (they come from L2: the tile's features are
      // re-read for every net)
      float pe_n[24];
      uint4 p6_n[3][PL];
      auto fetch = [&](const int it) {
#pragma unroll
        for (int j = 0; j < 24; ++j) pe_n[j] = ldg_f32_hint(pet + (size_t)(it * 24 + j) * TP, pol_keep);
#pragma unroll
        for (int qd = 0; qd < 3; ++qd)
#pragma unroll
          for (int p = 0; p < PL; ++p) p6_n[qd][p] = ldg_v4_hint(pe6 + p * BLOB_C + piece_off(r, it * 3 + qd), pol_keep);
      };
      fetch(half * NB);
#pragma unroll 1
      for (int it = half * NB; it < half * NB + NB; ++it) {          // 24 columns = 4 frequencies = 3 pieces = 12 packed words per plane
        float pe[24], zp[24];
        uint4 p6[3][PL];
#pragma unroll
        for (int j = 0; j < 24; ++j) pe[j] = pe_n[j];
#pragma unroll
        for (int qd = 0; qd < 3; ++qd)
#pragma unroll
          for (int p = 0; p < PL; ++p) p6[qd][p] = p6_n[qd][p];
        if (it + 1 < half * NB + NB) fetch(it + 1);
        float kb[4][3];                                               // (dod_c sZP) band_f: one product per (frequency, component) of this group
#pragma unroll
        for (int f = 0; f < 4; ++f)
#pragma unroll
          for (int c = 0; c < 3; ++c) kb[f][c] = ddP[c] * w.band[it * 4 + f];
#pragma unroll
        for (int j = 0; j < 24; ++j)                                  // it*24 is a multiple of 6: the partner stays inside the block
          zp[j] = fmaf(dvP, pe[j], (DPE_SIGN(j) * kb[j / 6][j % 3]) * pe[DPE_PARTNER(j)]);
        uint32_t hi[12], lo[12];
#pragma unroll
        for (int qd = 0; qd < 3; ++qd) {
          uint4 pq[PL];
          split8<PL, F16>(zp + qd * 8, pq);
          const uint32_t goff = gp_off(24, r, it * 3 + qd);
          __stcs(reinterpret_cast<uint4*>(blob_zp<PL>(nt) + goff), pq[0]);
          if (PL == 2) __stcs(reinterpret_cast<uint4*>(blob_zp<PL>(nt) + BLOB_C + goff), pq[PL - 1]);
          hi[qd * 4 + 0] = pq[0].x; hi[qd * 4 + 1] = pq[0].y; hi[qd * 4 + 2] = pq[0].z; hi[qd * 4 + 3] = pq[0].w;
          lo[qd * 4 + 0] = pq[PL - 1].x; lo[qd * 4 + 1] = pq[PL - 1].y; lo[qd * 4 + 2] = pq[PL - 1].z; lo[qd * 4 + 3] = pq[PL - 1].w;
          float d6[8], da[8];
          unpack_planes<PL, F16>(p6[qd], d6);
#pragma unroll
          for (int e = 0; e < 8; ++e) { da[e] = F16 ? d6[e] * (dv * (sZDa / S_PE)) : d6[e] * dv; d6[e] *= F16 ? dv * (sZD / S_PE) : dv; }
          split8<PL, F16>(d6, pq);
          __stcs(reinterpret_cast<uint4*>(blob_zd<PL>(nt) + goff), pq[0]);
          if (PL == 2) __stcs(reinterpret_cast<uint4*>(blob_zd<PL>(nt) + BLOB_C + goff), pq[PL - 1]);
          if (F16) split8<PL, F16>(da, pq);                           // (bf16 / bf16x3: no scales, the same planes serve both)
          const uint32_t soff = piece_off(r, it * 3 + qd);
          *reinterpret_cast<uint4*>(zdt + soff) = pq[0];
          if (PL == 2) *reinterpret_cast<uint4*>(zdt + BLOB_C + soff) = pq[PL - 1];
        }
        tmem_st8(R1 + it * 12, hi); tmem_st4(R1 + it * 12 + 8, hi + 8);
        if (PL == 2) { tmem_st8(R1 + p2z::ZP_LO + it * 12, lo); tmem_st4(R1 + p2z::ZP_LO + it * 12 + 8, lo + 8); }
        epi.blk_done(it - half * NB, true);               // (and its part of the zd tile is in shared memory)
      }
      if (timed) t_pro += clock64() - t_p0;
      // ---- epilogue 7: zh = m1 (acc + dov b1) ----
      epi.acc_wait(0);
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32];
        tmem_ld32(R0 + cg * 32, v);
        uint32_t bits = 0u;
#pragma unroll
        for (int i = 0; i < NB; ++i) bits = (cb == i) ? m1w[i] : bits;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(svec + p2z::V2_B1 * H + cg * 32 + j4 * 4);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            const float z = F16 ? fmaf(v[j], k7, dvH * bb[e]) : fmaf(dv, bb[e], v[j]);      // zh sZH
            v[j] = ((bits >> j) & 1u) ? z : 0.f;
          }
        }
        epi.emit(cg, v, blob_h<PL>(nt, B_ZH), true, R0 + cg * 32);
        epi.blk_done(cb, true);
      }
      // ---- epilogue 8: zc = acc + dov (b2 + bd + e) -> workspace (Z operand of dWa);  column sum -> vc ----
      epi.acc_wait(1);
#pragma unroll 1
      for (int cb = 0; cb < NB; ++cb) {
        const int cg = c0 + cb;
        float v[32], z[32];
        tmem_ld32(R1 + cg * 32, v);
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(svec + p2z::V2_BSUM * H + cg * 32 + j4 * 4);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            z[j] = v[j] = F16 ? fmaf(v[j], k8, dvC * bb[e]) : fmaf(dv, bb[e], v[j]);           // zc sZC
          }
        }
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
          uint4 pq[PL];
          split8<PL, F16>(v + qd * 8, pq);
          const uint32_t off = gp_off(32, r, cg * 4 + qd);
          __stcs(reinterpret_cast<uint4*>(blob_h<PL>(nt, B_ZC) + off), pq[0]);
          if (PL == 2) __stcs(reinterpret_cast<uint4*>(blob_h<PL>(nt, B_ZC) + BLOB_H + off), pq[PL - 1]);
        }
        const float cs = warp_colsum32(z, lane);
        atomicAdd(csum + cg * 32 + lane, cs * inv_sZC);
      }
      tc_fence_before();                                                // my reads of R1 precede the prologue's tcgen05.st of the next net
      // ---- flush this net's column sums ----
      if (half == 0) {
        float sd = dv;
#pragma unroll
        for (int m = 16; m; m >>= 1) sd += __shfl_xor_sync(0xffffffffu, sd, m);
        if (lane == 0) atomicAdd(csum + H, sd);
      }
      epi_bar<PL>();
      for (int i = tid; i < H; i += Geo<PL>::ET) {
        atomicAdd(w.vc + (size_t)k * H + i, csum[i]);
        csum[i] = 0.f;
      }
      if (tid == 0) { atomicAdd(w.sdo + k, csum[H]); csum[H] = 0.f; }
    }
    if (timed && tid == 0) {
      const long long tot = clock64() - t_begin;
      atomicAdd((unsigned long long*)w.phase_dbg + 12, (unsigned long long)tot);
      atomicAdd((unsigned long long*)w.phase_dbg + 13, (unsigned long long)epi.t_acc);
      atomicAdd((unsigned long long*)w.phase_dbg + 15, (unsigned long long)(tot - epi.t_acc));
      atomicAdd((unsigned long long*)w.phase_dbg + 11, (unsigned long long)t_pro);
      atomicAdd((unsigned long long*)w.phase_dbg + 14, 1ull);
    }
  }
  pp::block_end<PL>(tmem, warp);
}

// ------------------------------------------------------------------------------------------------
struct WgradWork {
  int B, Kn, T, splits;
  const uint8_t* blobs;
  const NetScales* sc;
  const float* uvec;       // [Kn][H] u = Wb^T wo
  const float *Wa, *ba;    // [Kn][H][H], [Kn][H] fp32 (split modes: vg = sum_p gz from the dWa contraction, see wgrad2_kernel)
  float* vg;               // [Kn][H]
  float *gW1, *gW2, *gWa, *gWd;
  float *gb1, *gb2, *ge, *gbd, *gba;
};

// ------------------------------------------------------------------------------------------------
// Weight gradients: K = points contractions of the tiles pass 1 / pass 2 stored (round 1 ran them with one 200 KB stage per SM - load
// and MMA strictly alternating, 3.8 TB/s).  The kernel is
// HBM-bound (it reads every operand tile pass 1 / pass 2 wrote), so the structure follows the bytes:
//   * tiles are stored [point quarter][k-core][32 rows][16 B] (gp_off), so a 32-point quarter of every operand is contiguous; THREE
//     stages of 73 KB: the bulk loads of quarter-tiles i+1, i+2 run under the MMAs of quarter-tile i;
//   * three kinds of work item per (sample, net):  0: dW1 = qm^T zp (+ db1);  1: dW2 = y^T zh AND dWd = y^T zd (+ db2) - the two layers
//     that share J = y run in ONE item with a 256 + 192 column accumulator, so the y tile is read once (-15 % of the kernel's bytes);
//     2: S = m3^T zc with J = [a3 > 0] as one exact 16-bit plane built from the mask bits of pass 1 (two MMAs per step instead of
//     three, no stored J tile).  Its epilogue derives three results from S and the seed product sm3 = sum_p m3 dov:
//     dWa = diag(u) S,  dba = u sm3,  and the column sum of the never-formed tile gz = m3 (zc Wa^T + dov ba):
//     vg[j] = sum_i Wa[j,i] S[j,i] + ba[j] sm3[j]  - which is why pass 2 has no third GEMM;
//   * bias gradients are seed-tile products (an N = 16 MMA of the same J planes against the three 16-bit terms of dov);
//   * the two CTAs of a cluster are the two output halves of one item: they contract against the SAME Z quarter-tiles, each fetches
//     half of every Z plane (and of the seed tile) and multicasts it to both - one L2 / DRAM read instead of two;
//   * epilogue: every thread owns one output row; it parks the scaled row in shared memory (the stages are free by then) and hands
//     it to the TMA engine as ONE bulk fp32 reduction (cp.reduce.async.bulk ... add.f32, 768 / 1024 contiguous bytes) instead of
//     192 / 256 scalar red.global.add whose 32 lanes hit 32 different rows.
// ------------------------------------------------------------------------------------------------
namespace wg2 {
constexpr int PT = 32;                              // points per stage
constexpr int J_PLANE = PT * 128 * 2;               // 8192: [16 k-cores of this out-half][32][16 B]
constexpr int ZH_PLANE = PT * H * 2;                // 16384
constexpr int ZC_PLANE = PT * C * 2;                // 12288
constexpr int X_BYTES = PT * 16 * 2;                // 1024 seed tile
constexpr int ROW_PAD = 16;                         // bytes between staged output rows: 1040-byte pitch -> conflict-free 16-byte stores
constexpr int ITEMS = 3;                            // work-item kinds per (sample, net)
constexpr int NSTG_MAX = 5;
template <int PL>
struct Cfg {                                        // stage = J planes | Z1 planes (zp / zh / zc) | Z2 planes (zd) | seed tile
  static constexpr int NSTG = PL == 2 ? 3 : 5;
  static constexpr int OFF_Z1 = PL * J_PLANE, OFF_Z2 = OFF_Z1 + PL * ZH_PLANE, OFF_X = OFF_Z2 + PL * ZC_PLANE;
  static constexpr int STAGE = OFF_X + X_BYTES;     // 74752 / 37888
  static constexpr int SMEM = NSTG * STAGE;         // 224256 / 189440
  static_assert(128 * (H * 4 + ROW_PAD) <= SMEM, "the staged [128 x 256] fp32 output must fit the (idle) stages");
  static_assert(SMEM + 1024 <= 227 * 1024, "the stages must fit one SM's 227 KB");
};
}  // namespace wg2

template <int PL, bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(192, 1) wgrad2_kernel(const WgradWork w) {
  using WG = wg2::Cfg<PL>;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t full[wg2::NSTG_MAX], empty[wg2::NSTG_MAX], acc_ready;
  __shared__ uint32_t tmem_s;
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  int item = blockIdx.x;
  const int mh = item & 1; item >>= 1;                               // output half == cluster rank
  const int split = item % w.splits; item /= w.splits;
  const int kind = item % wg2::ITEMS; item /= wg2::ITEMS;            // 0: dW1   1: dW2 + dWd   2: dWa (mask)
  const int k = item % w.Kn, b = item / w.Kn;
  const int N1 = kind == 0 ? C : H;                                   // columns of the first Z tile (zp | zh | zc)
  const bool two = kind == 1;                                         // second Z tile: zd, N = 192
  const bool build_j = kind == 2;
  const uint32_t z1plane = (uint32_t)wg2::PT * N1 * 2;                // bytes of one plane of a Z1 quarter-tile
  const int jsel = kind == 0 ? B_QM : B_YT;
  const int t0 = (int)((long long)w.T * split / w.splits), t1 = (int)((long long)w.T * (split + 1) / w.splits);
  const int nst = 4 * (t1 - t0);                                      // quarter-tiles
  if (tid == 0) {
    for (int s = 0; s < WG::NSTG; ++s) { mbar_init(&full[s], build_j ? 129 : 1); mbar_init(&empty[s], 2); }
    mbar_init(&acc_ready, 1);
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc(&tmem_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  cluster_sync_all();                                                // the peer's barriers exist before anything is multicast to them
  const uint32_t tmem = tmem_s;
  constexpr uint32_t COL_D2 = 256, COL_X = 448;                       // TMEM: D1 [0,256) | D2 (dWd) [256,448) | seed product [448,464)
  if (nst > 0) {
    if (warp == 4) {
      for (int i = 0; i < nst; ++i) {
        const int t = t0 + (i >> 2), pq = i & 3;                      // tile, point quarter
        const uint8_t* nt = w.blobs + (((size_t)b * w.Kn + k) * w.T + t) * Geo<PL>::NET_TILE;
        const uint8_t* jsrc = nt + off_h<PL>(jsel) + (size_t)pq * (BLOB_H / 4) + (size_t)mh * wg2::J_PLANE;
        const uint8_t* z1src = (kind == 0 ? nt + off_zp<PL>() : nt + off_h<PL>(kind == 1 ? B_ZH : B_ZC)) + (size_t)pq * z1plane;
        const uint32_t z1stride = kind == 0 ? BLOB_C : BLOB_H;          // plane stride of the Z1 tile in the workspace
        const uint8_t* z2src = nt + off_zd<PL>() + (size_t)pq * wg2::ZC_PLANE;
        const uint8_t* xsrc = nt + off_aux<PL>() + (size_t)pq * wg2::X_BYTES;
        const int s = i % WG::NSTG;
        uint8_t* st = smem + s * WG::STAGE;
        mbar_wait(&empty[s], ((i / WG::NSTG) & 1) ^ 1);              // BOTH CTAs are done with the previous occupant (multicast commits)
        if (elect_one()) {
          mbar_arrive_expect_tx(&full[s], (build_j ? 0 : PL * wg2::J_PLANE) + PL * z1plane + (two ? PL * wg2::ZC_PLANE : 0) + wg2::X_BYTES);
          const uint32_t zh = z1plane / 2, z2h = wg2::ZC_PLANE / 2, xh = wg2::X_BYTES / 2;
#pragma unroll
          for (int p = 0; p < PL; ++p) {
            if (!build_j) bulk_g2s(st + p * wg2::J_PLANE, jsrc + (size_t)p * BLOB_H, wg2::J_PLANE, &full[s]);
            bulk_g2s_mc(st + WG::OFF_Z1 + p * wg2::ZH_PLANE + mh * zh, z1src + (size_t)p * z1stride + mh * zh, zh, &full[s], (uint16_t)3);
            if (two) bulk_g2s_mc(st + WG::OFF_Z2 + p * wg2::ZC_PLANE + mh * z2h, z2src + (size_t)p * BLOB_C + mh * z2h, z2h, &full[s], (uint16_t)3);
          }
          bulk_g2s_mc(st + WG::OFF_X + mh * xh, xsrc + mh * xh, xh, &full[s], (uint16_t)3);
        }
      }
    } else if (warp == 5) {
      const uint32_t idesc1 = idesc_16(F16, N1, 1, 1), idesc2 = idesc_16(F16, C, 1, 1), idesc_x = idesc_16(F16, 16, 1, 1);
      // MN-major operands: 8-element groups of the M / N dimension are one k-core block of [32 points][16 B] = 512 bytes apart,
      // 8-point groups of the K dimension 128 bytes; a K = 16-point step adds 256 bytes (>> 4) to the address field
      constexpr uint32_t SBO = wg2::PT * 16;
      constexpr uint32_t a_lo = wg2::J_PLANE >> 4, b1_lo = wg2::ZH_PLANE >> 4, b2_lo = wg2::ZC_PLANE >> 4;
      for (int i = 0; i < nst; ++i) {
        const int s = i % WG::NSTG;
        const uint32_t base = smem_u32(smem + s * WG::STAGE);
        const uint64_t a_hi = smem_desc(base, 128, SBO), b1_hi = smem_desc(base + WG::OFF_Z1, 128, SBO), b2_hi = smem_desc(base + WG::OFF_Z2, 128, SBO);
        const uint64_t x_d = smem_desc(base + WG::OFF_X, 128, SBO);
        mbar_wait(&full[s], (i / WG::NSTG) & 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < wg2::PT / 16; ++ks) {
            const uint32_t first = (i > 0 || ks > 0) ? 1u : 0u;
            const uint64_t ad = a_hi + ks * 16, b1 = b1_hi + ks * 16, b2 = b2_hi + ks * 16, xd = x_d + ks * 16;
            // every J plane is fetched from shared memory once per step for all MMAs that read it (A collector)
            if (PL == 1) {                                   // one plane per operand: J Z1 (+ J Z2) + J seeds
              mma_f16_c<A_FILL>(tmem, ad, b1, idesc1, first);
              if (two) mma_f16_c<A_USE>(tmem + COL_D2, ad, b2, idesc2, first);
              mma_f16_c<A_LAST>(tmem + COL_X, ad, xd, idesc_x, first);
            } else if (build_j) {                            // exact one-plane J (the mask): J Z_lo + J Z_hi + J seeds
              mma_f16_c<A_FILL>(tmem, ad, b1 + b1_lo, idesc1, first);
              mma_f16_c<A_USE>(tmem, ad, b1, idesc1, 1u);
              mma_f16_c<A_LAST>(tmem + COL_X, ad, xd, idesc_x, first);
            } else if (two) {                                // J = y against zh (D1) and zd (D2)
              mma_f16_c<A_FILL>(tmem, ad + a_lo, b1, idesc1, first);
              mma_f16_c<A_USE>(tmem + COL_D2, ad + a_lo, b2, idesc2, first);
              mma_f16_c<A_LAST>(tmem + COL_X, ad + a_lo, xd, idesc_x, first);
              mma_f16_c<A_FILL>(tmem, ad, b1 + b1_lo, idesc1, 1u);
              mma_f16_c<A_USE>(tmem, ad, b1, idesc1, 1u);
              mma_f16_c<A_USE>(tmem + COL_D2, ad, b2 + b2_lo, idesc2, 1u);
              mma_f16_c<A_USE>(tmem + COL_D2, ad, b2, idesc2, 1u);
              mma_f16_c<A_LAST>(tmem + COL_X, ad, xd, idesc_x, 1u);
            } else {
              mma_f16_c<A_FILL>(tmem, ad + a_lo, b1, idesc1, first);
              mma_f16_c<A_LAST>(tmem + COL_X, ad + a_lo, xd, idesc_x, first);
              mma_f16_c<A_FILL>(tmem, ad, b1 + b1_lo, idesc1, 1u);
              mma_f16_c<A_USE>(tmem, ad, b1, idesc1, 1u);
              mma_f16_c<A_LAST>(tmem + COL_X, ad, xd, idesc_x, 1u);
            }
          }
          mma_commit_mc(&empty[s], (uint16_t)3);                      // the stage is free in BOTH CTAs' eyes only when both have read it
        }
      }
      if (elect_one()) mma_commit(&acc_ready);
    } else if (warp < 4) {
      if (build_j) {
        // J quarter-tile = [16 k-cores][32 points][8 features], one plane: thread = (point, 32-feature group gq): 4 pieces from one mask word
        const int pt = tid & 31, gq = tid >> 5;
        for (int i = 0; i < nst; ++i) {
          const int t = t0 + (i >> 2), pq = i & 3, s = i % WG::NSTG;
          const uint8_t* nt = w.blobs + (((size_t)b * w.Kn + k) * w.T + t) * Geo<PL>::NET_TILE;
          const uint32_t mw = __ldg(reinterpret_cast<const uint32_t*>(nt + off_mask<PL>() + MASK_BYTES / 2) + (size_t)(pq * wg2::PT + pt) * 8 + mh * 4 + gq);
          uint8_t* st = smem + s * WG::STAGE;
          mbar_wait(&empty[s], ((i / WG::NSTG) & 1) ^ 1);            // both CTAs' MMAs are done with the previous occupant of the stage
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t bits = (mw >> (j * 8)) & 0xFFu;
            constexpr uint32_t ONE = F16 ? 0x3C00u : 0x3F80u;                 // 1.0 in the operand format
            uint32_t hi[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) hi[e] = (((bits >> (2 * e)) & 1u) ? ONE : 0u) | (((bits >> (2 * e + 1)) & 1u) ? (ONE << 16) : 0u);
            const uint32_t off = (uint32_t)(gq * 4 + j) * (wg2::PT * 16) + (uint32_t)pt * 16;
            *reinterpret_cast<uint4*>(st + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          }
          fence_proxy_async();                                         // generic-proxy stores -> visible to the tensor core's reads
          mbar_arrive(&full[s]);
        }
      }
      mbar_wait(&acc_ready, 0);                                        // every MMA has completed: all stages are idle
      tc_fence_after();
      const size_t gk = ((size_t)b * w.Kn + k);
      const int out = mh * TP + tid;
      float un1 = 1.f, un2 = 1.f, un_x = 1.f;                          // fp16 variant: undo (J tile scale) x (Z tile / seed scale)
      if (F16) {
        const NetScales t = w.sc[gk];
        const float sj = kind == 0 ? t.sQ : (kind == 2 ? 1.f : t.sY);        // (the mask carries no scale)
        const float sz1 = kind == 0 ? t.sZP : (kind == 1 ? t.sZH : t.sZC);
        un1 = (1.f / sj) * (1.f / sz1); un2 = (1.f / sj) * (1.f / t.sZD); un_x = (1.f / sj) * (1.f / t.sDV);   // separately: sj * sz may leave the fp32 range
      }
      // kind 2: this row of S = m3^T zc gives dWa[out,:] = u[out] S and the dot product with Wa[out,:] that vg needs
      const float urow = build_j ? __ldg(w.uvec + (size_t)k * H + out) : 1.f;
      const float* warow = w.Wa + ((size_t)k * H + out) * H;
      float dot0 = 0.f, dot1 = 0.f;
      uint8_t* myrow = smem + (size_t)tid * (H * 4 + wg2::ROW_PAD);
      const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
      float v[32];
      {
        float* dst = (kind == 0 ? w.gW1 + gk * H * C : kind == 1 ? w.gW2 + gk * H * H : w.gWa + (size_t)k * H * H) + (size_t)out * N1;
        const float sc = un1 * urow;
        for (int cb = 0; cb < N1 / 32; ++cb) {
          tmem_ld32(lane_base + cb * 32, v);
          if (build_j) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 wv = __ldg(reinterpret_cast<const float4*>(warow + cb * 32) + j4);
              dot0 = fmaf(v[j4 * 4], wv.x, dot0); dot1 = fmaf(v[j4 * 4 + 1], wv.y, dot1);
              dot0 = fmaf(v[j4 * 4 + 2], wv.z, dot0); dot1 = fmaf(v[j4 * 4 + 3], wv.w, dot1);
            }
          }
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            *reinterpret_cast<float4*>(myrow + cb * 128 + j4 * 16) =
                (F16 || build_j) ? make_float4(v[j4 * 4] * sc, v[j4 * 4 + 1] * sc, v[j4 * 4 + 2] * sc, v[j4 * 4 + 3] * sc)
                                 : make_float4(v[j4 * 4], v[j4 * 4 + 1], v[j4 * 4 + 2], v[j4 * 4 + 3]);
        }
        fence_proxy_async();                                           // my generic-proxy row -> visible to the bulk engine
        bulk_red_add_f32(dst, myrow, (uint32_t)N1 * 4u);
        bulk_commit();
      }
      if (two) {                                                       // second output of the merged item: dWd rows (the staging row is reused)
        float* dst = w.gWd + (size_t)k * H * C + (size_t)out * C;
        bulk_wait_read_all();
        for (int cb = 0; cb < C / 32; ++cb) {
          tmem_ld32(lane_base + COL_D2 + cb * 32, v);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            *reinterpret_cast<float4*>(myrow + cb * 128 + j4 * 16) =
                F16 ? make_float4(v[j4 * 4] * un2, v[j4 * 4 + 1] * un2, v[j4 * 4 + 2] * un2, v[j4 * 4 + 3] * un2)
                    : make_float4(v[j4 * 4], v[j4 * 4 + 1], v[j4 * 4 + 2], v[j4 * 4 + 3]);
        }
        fence_proxy_async();
        bulk_red_add_f32(dst, myrow, (uint32_t)C * 4u);
        bulk_commit();
      }
      {
        float x[16];
        tmem_ld16(lane_base + COL_X, x);
        const float bsum = (x[0] + x[1] + x[2]) * un_x;                // the three 16-bit terms of the seed
        if (kind == 0) {
          atomicAdd(w.gb1 + gk * H + out, bsum);
        } else if (kind == 2) {                                        // bsum = sum_p m3[p,out] dov[p]
          atomicAdd(w.gba + (size_t)k * H + out, urow * bsum);
          atomicAdd(w.vg + (size_t)k * H + out, fmaf(__ldg(w.ba + (size_t)k * H + out), bsum, (dot0 + dot1) * un1));
        } else {
          atomicAdd(w.gb2 + gk * H + out, bsum);
          atomicAdd(w.ge + gk * H + out, bsum);
          atomicAdd(w.gbd + (size_t)k * H + out, bsum);
        }
      }
      bulk_wait_read_all();                                            // the engine has read my row: shared memory may go away
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                                // nobody leaves while the peer's commits may still arrive on its barriers
  if (warp == 5) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// SIMT helpers of the tensor-core mode
// ------------------------------------------------------------------------------------------------
// ---- scaling plan of the fp16 variant -------------------------------------------------------------
__device__ __forceinline__ float block_max256(float v, float* red) {      // 256 threads; every thread gets the result
#pragma unroll
  for (int w = 16; w; w >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, w));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float m = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
  return m;
}

// One block per (sample, net): L1 norms / maxima of its matrices -> activation bounds and tile scales.
__global__ void __launch_bounds__(1024) bounds_kernel(int Kn, const float* __restrict__ W1, const float* __restrict__ b1,
                                                     const float* __restrict__ W2, const float* __restrict__ Wd,
                                                     const float* __restrict__ Wa, const float* __restrict__ ba,
                                                     const float* __restrict__ bsum, const float* __restrict__ uvec,
                                                     const float* __restrict__ wo2, NetScales* __restrict__ tab) {
  __shared__ float red[8];
  __shared__ float srow[8][H];                                       // per matrix row: L1 norm / maximum of W1, Wd, W2, Wa
  // 1024 threads: the block reads ~1.4 MB and one SM's memory-level parallelism is what bounds it (48 blocks on 148 SMs)
  __shared__ float scol[2][4][H];                                    // partial column L1 norms of W2, Wa
  const int bk = blockIdx.x, k = bk % Kn, j = threadIdx.x & 255, part = threadIdx.x >> 8, lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const float* w1m = W1 + (size_t)bk * H * C;
  const float* w2 = W2 + (size_t)bk * H * H;
  const float* wdm = Wd + (size_t)k * H * C;
  const float* wa = Wa + (size_t)k * H * H;
  // row-wise quantities: one warp per row, lanes along the row (coalesced), shuffle reduction
  for (int row = wrp; row < H; row += 32) {
    float a1 = 0.f, x1 = 0.f, ad = 0.f, xd = 0.f, a2 = 0.f, x2 = 0.f, aa = 0.f, xa = 0.f;
    for (int i = lane; i < C; i += 32) {
      const float a = fabsf(w1m[(size_t)row * C + i]), d = fabsf(wdm[(size_t)row * C + i]);
      a1 += a; x1 = fmaxf(x1, a); ad += d; xd = fmaxf(xd, d);
    }
    for (int i = lane; i < H; i += 32) {
      const float a = fabsf(w2[(size_t)row * H + i]), c = fabsf(wa[(size_t)row * H + i]);
      a2 += a; x2 = fmaxf(x2, a); aa += c; xa = fmaxf(xa, c);
    }
#pragma unroll
    for (int m = 16; m; m >>= 1) {
      a1 += __shfl_xor_sync(0xffffffffu, a1, m); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, m));
      ad += __shfl_xor_sync(0xffffffffu, ad, m); xd = fmaxf(xd, __shfl_xor_sync(0xffffffffu, xd, m));
      a2 += __shfl_xor_sync(0xffffffffu, a2, m); x2 = fmaxf(x2, __shfl_xor_sync(0xffffffffu, x2, m));
      aa += __shfl_xor_sync(0xffffffffu, aa, m); xa = fmaxf(xa, __shfl_xor_sync(0xffffffffu, xa, m));
    }
    if (lane == 0) {
      srow[0][row] = a1; srow[1][row] = x1; srow[2][row] = ad; srow[3][row] = xd;
      srow[4][row] = a2; srow[5][row] = x2; srow[6][row] = aa; srow[7][row] = xa;
    }
  }
  // column-wise L1 norms: thread (part, j) walks down a quarter of column j (coalesced across the block)
  float c2 = 0.f, ca = 0.f;
  for (int i0 = part * 64; i0 < part * 64 + 64; i0 += 16) {          // 32 independent loads in flight per thread
    float t2[16], ta[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) { t2[u] = __ldg(w2 + (size_t)(i0 + u) * H + j); ta[u] = __ldg(wa + (size_t)(i0 + u) * H + j); }
#pragma unroll
    for (int u = 0; u < 16; ++u) { c2 += fabsf(t2[u]); ca += fabsf(ta[u]); }
  }
  scol[0][part][j] = c2; scol[1][part][j] = ca;
  __syncthreads();
  if (threadIdx.x >= H) return;                                      // (exited threads do not take part in later barriers)
  c2 = (scol[0][0][j] + scol[0][1][j]) + (scol[0][2][j] + scol[0][3][j]);
  ca = (scol[1][0][j] + scol[1][1][j]) + (scol[1][2][j] + scol[1][3][j]);
  const float r1 = srow[0][j], m1 = srow[1][j], rd = srow[2][j], md = srow[3][j];
  const float r2 = srow[4][j], m2 = srow[5][j], ra = srow[6][j], ma = srow[7][j];
  const float l1W1 = block_max256(r1, red), M1 = block_max256(r1 + fabsf(b1[(size_t)bk * H + j]), red);
  const float l1W2 = block_max256(r2, red), l1Wd = block_max256(rd, red), l1Wa = block_max256(ra, red);
  const float cW2 = block_max256(c2, red), cWa = block_max256(ca, red);
  const float mW1 = block_max256(m1, red), mW2 = block_max256(m2, red), mWd = block_max256(md, red), mWa = block_max256(ma, red);
  const float mBs = block_max256(fabsf(bsum[(size_t)bk * H + j]), red), mBa = block_max256(fabsf(ba[(size_t)k * H + j]), red);
  const float Mu = block_max256(fabsf(uvec[(size_t)k * H + j]), red), mWo2 = block_max256(fabsf(wo2[(size_t)k * H + j]), red);
  const float mWaU = block_max256(fabsf(uvec[(size_t)k * H + j]) * ma, red);       // max |u_j Wa_ji|
  if (j == 0) {
    NetScales t;
    const float Mc = l1W2 * M1 + l1Wd + mBs, Mg = l1Wa * Mc + mBa;
    const float My = Mu * cWa + mWo2, Mq = My * cW2;
    t.sW1 = scale_for(mW1 * 32.f);                   // weights: maximum -> 2^10
    t.sWa = scale_for(mWa * 32.f);
    t.sWaU = scale_for(mWaU * 32.f);
    t.sWd = scale_for(mWd * 32.f);                   // preliminary: plan_kernel couples sWd, sH1 and sW2
    t.sW2 = scale_for(mW2);                          // preliminary: the LARGEST admissible factor
    t.sH1 = scale_for(M1); t.sC = scale_for(Mc); t.sG = scale_for(Mg);
    t.sUM = scale_for(Mu); t.sY = scale_for(My); t.sQ = scale_for(Mq);
    t.M1 = M1; t.Mc = Mc; t.l1W1 = l1W1; t.l1W12 = l1W1 * l1W2;
    t.rowB = fmaxf(1.f, fmaxf(l1W1, l1W1 * l1W2));
    t.cap = t.sH1 * t.sW2;
    t.sZP = t.sZH = t.sZC = t.sZD = t.sDV = 1.f;
    tab[bk] = t;
  }
}

// G2 accumulates h1 W2^T and PE6 Wd^T in ONE accumulator: (sH1 sW2) must equal (S_PE sWd), and the Wd image is shared by
// all samples.  Per net: T2 = min(S_PE * sWd, min over samples of their capacity); then sWd = T2 / S_PE, sW2 = T2 / sH1.
__global__ void plan_kernel(int B, int Kn, NetScales* __restrict__ tab) {
  const int k = threadIdx.x;
  if (k >= Kn) return;
  float T2 = S_PE * tab[k].sWd;
  for (int b = 0; b < B; ++b) T2 = fminf(T2, tab[b * Kn + k].cap);
  for (int b = 0; b < B; ++b) {
    NetScales& t = tab[b * Kn + k];
    t.sWd = T2 / S_PE;
    t.sW2 = T2 / t.sH1;
  }
}

// max |dov| and max |dod| per (sample, net) over the rows of this chunk -> seedmax[bk][2] (non-negative floats order like ints)
__global__ void __launch_bounds__(256) seedmax_kernel(int Kn, size_t rows_per_sample, const float* __restrict__ dov,
                                                      const float* __restrict__ dod, int* __restrict__ seedmax) {
  const int b = blockIdx.y;
  float mv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, md[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows_per_sample; r += (size_t)gridDim.x * blockDim.x) {
    const size_t row = (size_t)b * rows_per_sample + r;
    for (int k = 0; k < Kn; ++k) {
      mv[k] = fmaxf(mv[k], fabsf(dov[row * Kn + k]));
#pragma unroll
      for (int c = 0; c < 3; ++c) md[k] = fmaxf(md[k], fabsf(dod[(row * Kn + k) * 3 + c]));
    }
  }
  for (int k = 0; k < Kn; ++k) {
    float a = mv[k], d = md[k];
#pragma unroll
    for (int w = 16; w; w >>= 1) { a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, w)); d = fmaxf(d, __shfl_xor_sync(0xffffffffu, d, w)); }
    if ((threadIdx.x & 31) == 0) {
      if (a > 0.f && isfinite(a)) atomicMax(seedmax + ((size_t)b * Kn + k) * 2, __float_as_int(a));
      if (d > 0.f && isfinite(d)) atomicMax(seedmax + ((size_t)b * Kn + k) * 2 + 1, __float_as_int(d));
    }
  }
}

// Z-side scales of this chunk from the seed maxima: zp = dov PE + xt, zh = dov h1 + ht, zc = dov c + ct, zd = dov PE6
__global__ void zscale_kernel(int n, const int* __restrict__ seedmax, NetScales* __restrict__ tab) {
  const int bk = blockIdx.x * blockDim.x + threadIdx.x;
  if (bk >= n) return;
  NetScales& t = tab[bk];
  const float DV = __int_as_float(seedmax[bk * 2]), RR = 16.f * __int_as_float(seedmax[bk * 2 + 1]);   // |dPE/dz| <= 2^4
  t.sZP = scale_for(DV + RR);
  t.sZH = scale_for(DV * t.M1 + RR * t.l1W1);
  t.sZC = scale_for(DV * t.Mc + RR * t.l1W12);
  t.sZD = scale_for(DV);
  t.sDV = scale_for(DV);
}

// fp32 weight matrix [R_src x K_src] -> bf16 image in layout (*) ; transpose = image rows are source columns.
// The image is a sequence of K = 16 chunks (two k-cores, rows*32 bytes per plane); with PL planes a chunk is
// [hi plane | lo plane], so the producer still fetches one contiguous block per chunk.
template <int PL, bool F16>
__global__ void image_kernel(const float* __restrict__ src, size_t src_stride, uint8_t* __restrict__ dst,
                             size_t dst_stride, int rows, int kd, int transpose, const NetScales* __restrict__ tab, int which,
                             const float* __restrict__ kscale) {        // kscale [batch][kd]: image of S diag(kscale) (or nullptr)
  const float* S = src + blockIdx.y * src_stride;
  uint8_t* D = dst + blockIdx.y * dst_stride;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;             // 16-byte piece index
  if (q >= rows * kd / 8) return;
  const int kc = q / rows, r = q % rows;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = transpose ? S[(size_t)(kc * 8 + e) * rows + r] : S[(size_t)r * kd + kc * 8 + e];
  if (kscale) {
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] *= kscale[(size_t)blockIdx.y * kd + kc * 8 + e];
  }
  if (F16) {                                                         // entry blockIdx.y: (sample, net) for generated weights, (0, net) for static ones
    const NetScales& t = tab[blockIdx.y];
    const float sc = which == 0 ? t.sW1 : (which == 1 ? t.sW2 : (which == 2 ? t.sWd : (which == 3 ? t.sWa : t.sWaU)));
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] *= sc;
  }
  uint4 pq[PL];
  split8<PL, F16>(v, pq);
  // chunk = [hi plane | lo plane], each plane two k-cores of rows x 16 bytes
  const size_t base = (size_t)(kc >> 1) * PL * rows * 32 + (size_t)(kc & 1) * rows * 16 + (size_t)r * 16;
#pragma unroll
  for (int p = 0; p < PL; ++p) *reinterpret_cast<uint4*>(D + base + (size_t)p * rows * 32) = pq[p];
}

// coordinate / data features of one tile: bf16 blobs (GEMM operands) and the fp32 transposed copy (epilogues)
template <int PL, bool F16>
__global__ void __launch_bounds__(TP) encode_kernel(const DevConsts K, const Work w, const float* __restrict__ x,
                                                    const float* __restrict__ y, const float* __restrict__ t,
                                                    const float* __restrict__ coord_pe) {
  const size_t g = blockIdx.x;
  const int b = blockIdx.x / w.T, tl = blockIdx.x % w.T, r = threadIdx.x;
  const int p_local = tl * TP + r;
  const bool valid = p_local < w.P;
  const size_t q = (size_t)b * w.N + w.p0 + p_local;
  float z[3] = {0.f, 0.f, 0.f}, d[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (valid) {
    if (!coord_pe) { z[0] = (x[q] / K.dxf) / K.wm1; z[1] = (y[q] / K.dyf) / K.hm1; z[2] = t[q] / K.t_span; }
#pragma unroll
    for (int c = 0; c < 6; ++c) d[c] = w.coord_data[q * 6 + c];
  }
  uint8_t* pe = w.pe_blob + g * Geo<PL>::BC;
  uint8_t* pe6 = w.pe6_blob + g * Geo<PL>::BC;
  float* pet = w.pet + g * (size_t)(C * TP) + r;
  float buf[24];
#pragma unroll 1
  for (int it = 0; it < 8; ++it) {                                   // 4 frequencies x (3 sin, 3 cos)
#pragma unroll
    for (int ff = 0; ff < 4; ++ff) {
      const float band = K.band[it * 4 + ff];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float s = 0.f, co = 0.f;
        if (valid && !coord_pe) sincosf(z[c] * band, &s, &co);
        buf[ff * 6 + c] = s;
        buf[ff * 6 + 3 + c] = co;
      }
    }
    if (coord_pe && valid) {                                           // PhysicsNet.forward surface: the caller's encoding (values only)
#pragma unroll
      for (int j4 = 0; j4 < 6; ++j4) {
        const float4 pv = __ldg(reinterpret_cast<const float4*>(coord_pe + q * C + it * 24) + j4);
        buf[j4 * 4] = pv.x; buf[j4 * 4 + 1] = pv.y; buf[j4 * 4 + 2] = pv.z; buf[j4 * 4 + 3] = pv.w;
      }
    }
#pragma unroll
    for (int j = 0; j < 24; ++j) pet[(size_t)(it * 24 + j) * TP] = buf[j];
    if (F16) {
#pragma unroll
      for (int j = 0; j < 24; ++j) buf[j] *= S_PE;
    }
#pragma unroll
    for (int qd = 0; qd < 3; ++qd) sts8<PL, F16>(pe, BLOB_C, piece_off(r, it * 3 + qd), buf + qd * 8);      // (plain global stores)
  }
#pragma unroll 1
  for (int it = 0; it < 8; ++it) {                                   // 2 frequencies x (6 sin, 6 cos)
#pragma unroll
    for (int ff = 0; ff < 2; ++ff) {
      const float band = K.band6[it * 2 + ff];
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        float s = 0.f, co = 0.f;
        if (valid) sincosf(d[c] * band, &s, &co);
        buf[ff * 12 + c] = F16 ? s * S_PE : s;
        buf[ff * 12 + 6 + c] = F16 ? co * S_PE : co;
      }
    }
#pragma unroll
    for (int qd = 0; qd < 3; ++qd) sts8<PL, F16>(pe6, BLOB_C, piece_off(r, it * 3 + qd), buf + qd * 8);
  }
}

__global__ void seed_copy_kernel(const Work w, const float* __restrict__ d_o, float scale) {
  // values-only backward: dov[row][k] = d_o[q][k] * scale for valid rows
  const size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= (size_t)w.B * w.T * TP) return;
  const int tile = (int)(row / TP), r = (int)(row % TP);
  const int b = tile / w.T, tl = tile % w.T;
  const int p_local = tl * TP + r;
  for (int k = 0; k < w.Kn; ++k)
    w.dov[row * w.Kn + k] = p_local < w.P ? d_o[((size_t)b * w.N + w.p0 + p_local) * w.Kn + k] * scale : 0.f;
}

__global__ void gather_o_kernel(const Work w, float* __restrict__ o_out) {
  const size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= (size_t)w.B * w.T * TP) return;
  const int tile = (int)(row / TP), r = (int)(row % TP);
  const int b = tile / w.T, tl = tile % w.T;
  const int p_local = tl * TP + r;
  if (p_local >= w.P) return;
  for (int k = 0; k < w.Kn; ++k) o_out[((size_t)b * w.N + w.p0 + p_local) * w.Kn + k] = w.o[row * w.Kn + k];
}

// ------------------------------------------------------------------------------------------------
// Workspace and driver
// ------------------------------------------------------------------------------------------------
struct Carve {
  uint8_t *img_gen, *img_sta, *pe_blob, *pe6_blob, *blobs;
  float *pet, *o, *od, *dov, *dod, *uvec, *wo2, *cst, *bsum, *vc, *vg, *sdo;
  float *lx, *ly, *lt, *lcd;    // lattice staging (values-only carve only)
  long long* dbg;
  NetScales* sc;
  int* seedmax;
  size_t bytes;
};

static inline size_t al(size_t n) { return (n + 1023) & ~(size_t)1023; }

// What a values-only pass (sweep 0) touches comes first; what only the reverse sweep, the residual or the backward touches follows.
// values_only: the prefix plus the staging of the lattice job's per-point inputs, in place of the rest.
static Carve carve(uint8_t* base, int chunk, int Kn, int B, int pl, bool values_only = false) {
  Carve c;
  memset(&c, 0, sizeof(c));
  const size_t T = ((size_t)(chunk + TP - 1) / TP + CLUSTER - 1) / CLUSTER * CLUSTER, rows = (size_t)B * T * TP;
  size_t off = 0;
  auto take = [&](size_t bytes) { uint8_t* p = base + off; off += al(bytes); return p; };
  c.img_gen = take((size_t)B * Kn * GEN_IMG * pl);
  c.img_sta = take((size_t)Kn * STA_IMG * pl);
  c.pe_blob = take((size_t)B * T * BLOB_C * pl);
  c.pe6_blob = take((size_t)B * T * BLOB_C * pl);
  c.pet = reinterpret_cast<float*>(take((size_t)B * T * C * TP * 4));
  c.o = reinterpret_cast<float*>(take(rows * Kn * 4));
  c.uvec = reinterpret_cast<float*>(take((size_t)Kn * H * 4));
  c.wo2 = reinterpret_cast<float*>(take((size_t)Kn * H * 4));
  c.cst = reinterpret_cast<float*>(take((size_t)Kn * 4));
  c.bsum = reinterpret_cast<float*>(take((size_t)B * Kn * H * 4));
  c.dbg = reinterpret_cast<long long*>(take(16 * 8));
  c.sc = reinterpret_cast<NetScales*>(take((size_t)B * Kn * sizeof(NetScales)));
  if (values_only) {
    const size_t pts = (size_t)B * chunk;
    c.lx = reinterpret_cast<float*>(take(pts * 4));
    c.ly = reinterpret_cast<float*>(take(pts * 4));
    c.lt = reinterpret_cast<float*>(take(pts * 4));
    c.lcd = reinterpret_cast<float*>(take(pts * 24));
    c.bytes = off;
    return c;
  }
  c.blobs = take((size_t)B * Kn * T * (pl == 2 ? Geo<2>::NET_TILE : Geo<1>::NET_TILE));
  c.od = reinterpret_cast<float*>(take(rows * Kn * 12));
  c.dov = reinterpret_cast<float*>(take(rows * Kn * 4));
  c.dod = reinterpret_cast<float*>(take(rows * Kn * 12));
  c.vc = reinterpret_cast<float*>(take((size_t)Kn * H * 4));
  c.vg = reinterpret_cast<float*>(take((size_t)Kn * H * 4));
  c.sdo = reinterpret_cast<float*>(take((size_t)Kn * 4));
  c.seedmax = reinterpret_cast<int*>(take((size_t)B * Kn * 2 * sizeof(int)));
  c.bytes = off;
  return c;
}

int default_chunk(int B, int planes) {
  int c = DEFAULT_POINTS_IN_FLIGHT / planes / (B > 0 ? B : 1);
  c = c / TP * TP;
  return c < TP ? TP : c;
}

size_t workspace_bytes(int chunk, int Kn, int B, int planes) { return carve(nullptr, chunk, Kn, B, planes).bytes; }
size_t lattice_workspace_bytes(int chunk, int Kn, int B, int planes) { return carve(nullptr, chunk, Kn, B, planes, true).bytes; }

template <int PL, bool F16>
static int make_images(const DpnWeights& Wt, const Carve& c, int B, int Kn, cudaStream_t st) {
  struct Spec { const float* src; size_t sstride; size_t doff; size_t dstride; int rows, kd, tr, batches; uint8_t* dst; int which; const float* kscale; };
  // the transposed Wa image carries u (G4: y = m3 (diag(u) Wa) + 2wo with the bare mask as A operand)
  const float* ku = c.uvec;
  const Spec specs[] = {
      {Wt.W1, (size_t)H * C, 0, GEN_IMG, H, C, 0, B * Kn, c.img_gen, 0, nullptr},              // W1  : rows = out, k = in
      {Wt.W1, (size_t)H * C, IMG_HC, GEN_IMG, C, H, 1, B * Kn, c.img_gen, 0, nullptr},         // W1T : rows = in,  k = out
      {Wt.W2, (size_t)H * H, 2 * IMG_HC, GEN_IMG, H, H, 0, B * Kn, c.img_gen, 1, nullptr},
      {Wt.W2, (size_t)H * H, 2 * IMG_HC + IMG_HH, GEN_IMG, H, H, 1, B * Kn, c.img_gen, 1, nullptr},
      {Wt.Wd, (size_t)H * C, 0, STA_IMG, H, C, 0, Kn, c.img_sta, 2, nullptr},
      {Wt.Wa, (size_t)H * H, IMG_HC, STA_IMG, H, H, 0, Kn, c.img_sta, 3, nullptr},
      {Wt.Wa, (size_t)H * H, IMG_HC + IMG_HH, STA_IMG, H, H, 1, Kn, c.img_sta, ku ? 5 : 3, ku},
  };
  for (const Spec& s : specs) {
    if (s.batches == 0) continue;
    const int pieces = s.rows * s.kd / 8;
    image_kernel<PL, F16><<<dim3((pieces + 255) / 256, s.batches), 256, 0, st>>>(s.src, s.sstride, s.dst + s.doff * PL, s.dstride * PL,
                                                                                 s.rows, s.kd, s.tr, c.sc, s.which, s.kscale);
    DPN_LAUNCH_OK();
  }
  return 0;
}

template <int PL, bool F16>
static int run_planes(const Job& J, cudaStream_t st) {
  const int B = J.shape.B, N = J.shape.N, Kn = J.shape.K, chunk = J.chunk;
  {
    // function attributes are per device: set them once for every device this process drives (bit d of the mask)
    static std::atomic<unsigned long long> attr_done_mask{0ull};
    int dev = 0;
    DPN_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !((attr_done_mask.load(std::memory_order_acquire) >> dev) & 1ull)) {
      DPN_CUDA_OK(cudaFuncSetAttribute(pass1_ts_kernel<PL, F16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ts::Cfg<PL>::SMEM));
      if constexpr (PL == 2) DPN_CUDA_OK(cudaFuncSetAttribute(pass1_ts_kernel<PL, F16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ts::Cfg<PL>::SMEM));
      DPN_CUDA_OK(cudaFuncSetAttribute(pass2z_kernel<PL, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, p2z::Cfg<PL>::SMEM));
      DPN_CUDA_OK(cudaFuncSetAttribute(wgrad2_kernel<PL, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg2::Cfg<PL>::SMEM));
      if (dev >= 0 && dev < 64) attr_done_mask.fetch_or(1ull << dev, std::memory_order_release);
    }
  }
  const bool lattice = J.kind == JOB_LATTICE;
  Carve c = carve(reinterpret_cast<uint8_t*>(J.workspace), chunk, Kn, B, PL, lattice);
  const DpnWeights& Wt = *J.w;
  const bool pde = J.kind == JOB_PDE;
  const bool want_bwd = J.grads != nullptr;
  const int sweep = pde ? 2 : (J.kind == JOB_DEC_BWD ? 1 : 0);
  const double inv_n = 1.0 / (double)(J.shape.n_norm > 0 ? J.shape.n_norm : N);
  const double seed_scale = J.shape.seed_scale != 0.f ? (double)J.shape.seed_scale : 1.0;
  int rc;
#ifdef DPN_DEBUG_BUILD                                                 // cycle counters + a stream synchronisation: never in the release library
  static const bool phase_debug = getenv("DPN_PHASE_DEBUG") != nullptr;
  if (phase_debug) DPN_CUDA_OK(cudaMemsetAsync(c.dbg, 0, 16 * 8, st));
#else
  constexpr bool phase_debug = false;
#endif
  if ((rc = f32::launch_prep(B, Kn, Wt, c.uvec, c.wo2, c.cst, c.bsum, st))) return rc;
  if (F16) {                                                          // scaling plan before anything is converted to fp16
    bounds_kernel<<<B * Kn, 1024, 0, st>>>(Kn, Wt.W1, Wt.b1, Wt.W2, Wt.Wd, Wt.Wa, Wt.ba, c.bsum, c.uvec, c.wo2, c.sc);
    DPN_LAUNCH_OK();
    plan_kernel<<<1, 32, 0, st>>>(B, Kn, c.sc);
    DPN_LAUNCH_OK();
  }
  if ((rc = make_images<PL, F16>(Wt, c, B, Kn, st))) return rc;
  if (pde) DPN_CUDA_OK(cudaMemsetAsync(J.out->loss_terms, 0, sizeof(double) * 6 * B, st));
  if (pde && J.margin) DPN_CUDA_OK(cudaMemsetAsync(J.margin->loss, 0, sizeof(double) * B, st));
  if (want_bwd) {
    const DpnGrads& G = *J.grads;
    const size_t BKn = (size_t)B * Kn;
    DPN_CUDA_OK(cudaMemsetAsync(G.W1, 0, BKn * H * C * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.b1, 0, BKn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.W2, 0, BKn * H * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.b2, 0, BKn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.e, 0, BKn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.Wd, 0, (size_t)Kn * H * C * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.bd, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.Wa, 0, (size_t)Kn * H * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(G.ba, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(c.vc, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(c.vg, 0, (size_t)Kn * H * 4, st));
    DPN_CUDA_OK(cudaMemsetAsync(c.sdo, 0, (size_t)Kn * 4, st));
  }
  for (int p0 = 0; p0 < N; p0 += chunk) {
    const int P = min(chunk, N - p0);
    const int T = ((P + TP - 1) / TP + CLUSTER - 1) / CLUSTER * CLUSTER;   // clusters pair tiles of the same sample
    const size_t rows = (size_t)B * T * TP;
    Work w;
    memset(&w, 0, sizeof(w));
    w.B = B; w.Kn = Kn; w.T = T; w.P = P; w.N = N; w.p0 = p0;
    w.img_gen = c.img_gen; w.img_sta = c.img_sta;
    w.b1 = Wt.b1; w.bsum = c.bsum; w.ba = Wt.ba; w.uvec = c.uvec; w.wo2 = c.wo2; w.cst = c.cst;
    const float *px, *py, *pt, *ppe = nullptr;
    if (lattice) {                                                    // staged inputs of this chunk: [B][P], so q = b P + p_local
      if ((rc = launch_lattice(J.lat, 0, B, p0, P, c.lx, c.ly, c.lt, c.lcd, st))) return rc;
      w.N = P; w.p0 = 0;
      w.coord_data = c.lcd; w.ref = nullptr;
      px = c.lx; py = c.ly; pt = c.lt;
    } else {
      w.coord_data = J.pts->coord_data; w.ref = J.pts->ref;
      px = J.pts->x; py = J.pts->y; pt = J.pts->t; ppe = J.pts->coord_pe;
    }
    w.pe_blob = c.pe_blob; w.pe6_blob = c.pe6_blob; w.pet = c.pet; w.blobs = c.blobs;
    w.o = c.o; w.od = c.od; w.dov = c.dov; w.dod = c.dod;
    w.vc = c.vc; w.vg = c.vg; w.sdo = c.sdo;
    w.sc = c.sc;
    w.xfirst = J.shape.mode == DPN_MODE_F16X3A ? 1 : 0;
    w.phase_dbg = phase_debug ? c.dbg : nullptr;
#ifdef DPN_DEBUG_BUILD
    w.dbg_flags = getenv("DPN_DEBUG_FLAGS") ? atoi(getenv("DPN_DEBUG_FLAGS")) : 0;
#endif
    memcpy(w.band, J.dc.band, sizeof(w.band));
    const int tiles = B * T;
    encode_kernel<PL, F16><<<tiles, TP, 0, st>>>(J.dc, w, px, py, pt, ppe);
    DPN_LAUNCH_OK();
    if constexpr (PL == 2) {
      if (w.xfirst) pass1_ts_kernel<PL, F16, true><<<tiles, Geo<PL>::THREADS, ts::Cfg<PL>::SMEM, st>>>(w, sweep);
      else pass1_ts_kernel<PL, F16, false><<<tiles, Geo<PL>::THREADS, ts::Cfg<PL>::SMEM, st>>>(w, sweep);
    } else {
      pass1_ts_kernel<PL, F16, false><<<tiles, Geo<PL>::THREADS, ts::Cfg<PL>::SMEM, st>>>(w, sweep);
    }
    DPN_LAUNCH_OK();
    if (lattice) {
      if ((rc = launch_lattice_emit(J.lat, B, P, c.o, (size_t)T * TP, J.o + (size_t)p0 * 6, (size_t)N * 6, st))) return rc;
      continue;
    }
    if (J.kind == JOB_DEC_FWD) {
      gather_o_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(w, J.o);
      DPN_LAUNCH_OK();
      continue;
    }
    if (want_bwd || pde) {
      DPN_CUDA_OK(cudaMemsetAsync(c.dov, 0, rows * Kn * 4, st));
      DPN_CUDA_OK(cudaMemsetAsync(c.dod, 0, rows * Kn * 12, st));
    }
    if (pde) {                                                        // all samples in one launch (blockIdx.y = sample)
      const size_t srow = (size_t)T * TP, q0 = (size_t)p0;
      if ((rc = f32::launch_residual(J.dc, B, P, srow, (size_t)N, c.o, c.od, J.pts->f + q0, inv_n, seed_scale, J.out->loss_terms,
                                     c.dov, c.dod, J.out->vals ? J.out->vals + q0 * 6 : nullptr,
                                     J.out->jac ? J.out->jac + q0 * 18 : nullptr, st)))
        return rc;
      if (J.margin && (rc = f32::launch_margin(B, P, srow, (size_t)N, c.o, J.margin->target + q0 * 6, *J.margin, inv_n, seed_scale,
                                               J.margin->loss, c.dov, J.margin->o ? J.margin->o + q0 * 6 : nullptr, st)))
        return rc;
    } else {
      seed_copy_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(w, J.d_o, (float)seed_scale);
      DPN_LAUNCH_OK();
    }
    if (!want_bwd) continue;
    const DpnGrads& G = *J.grads;
    if (F16) {                                                        // Z-side scales of this chunk from the seeds' maxima
      DPN_CUDA_OK(cudaMemsetAsync(c.seedmax, 0, (size_t)B * Kn * 2 * sizeof(int), st));
      seedmax_kernel<<<dim3(64, B), 256, 0, st>>>(Kn, (size_t)T * TP, c.dov, c.dod, c.seedmax);
      DPN_LAUNCH_OK();
      zscale_kernel<<<(B * Kn + 63) / 64, 64, 0, st>>>(B * Kn, c.seedmax, c.sc);
      DPN_LAUNCH_OK();
    }
    pass2z_kernel<PL, F16><<<tiles, Geo<PL>::THREADS, p2z::Cfg<PL>::SMEM, st>>>(w);
    DPN_LAUNCH_OK();
    WgradWork ww;
    ww.B = B; ww.Kn = Kn; ww.T = T; ww.blobs = c.blobs; ww.sc = c.sc; ww.uvec = c.uvec;
    ww.Wa = Wt.Wa; ww.ba = Wt.ba; ww.vg = c.vg;
    ww.gW1 = G.W1; ww.gW2 = G.W2; ww.gWa = G.Wa; ww.gWd = G.Wd;
    ww.gb1 = G.b1; ww.gb2 = G.b2; ww.ge = G.e; ww.gbd = G.bd; ww.gba = G.ba;
    const int items = B * Kn * 2 * wg2::ITEMS;                            // x 2 output halves
    // point-splits per (sample, net, layer, out-half): fill whole waves of resident CTAs (148 SMs x CTAs per SM); every split
    // adds one fp32 red.add pass over the gradient tile, so prefer the smallest count within 2 % of the best wave efficiency
    int splits = 1;
    {
      const double slots = 148.0;
      double best = 0.0;
      for (int sp = 1; sp <= 8 && sp <= T; ++sp) {
        const double waves = items * sp / slots, eff = waves / ceil(waves);
        if (eff > best + 0.02) { best = eff; splits = sp; }
      }
      // The tensor core adds into its fp32 accumulator with round-toward-zero: a bias of ~2^-25 of the running sum per MMA.  One CTA
      // issues 24 MMAs per tile (split modes), so the error of a weight-gradient tile grows with the tiles it accumulates (measured
      // against an fp64 oracle at 65 536 points: 1e-4 with 64 tiles per CTA, 7e-6 with 4).  The split modes therefore flush to the
      // fp32 red.add sums (round-to-nearest) every `wgrad_tiles` tiles (32: 1.7e-5 at no measurable cost; 16: 1.2e-5 for +2 % time).
      static const int wgrad_tiles = getenv("DPN_WGRAD_TILES") ? atoi(getenv("DPN_WGRAD_TILES")) : 32;
      if (wgrad_tiles > 0 && (T + splits - 1) / splits > wgrad_tiles) splits = (T + wgrad_tiles - 1) / wgrad_tiles;
    }
    ww.splits = splits;
    wgrad2_kernel<PL, F16><<<items * splits, 192, wg2::Cfg<PL>::SMEM, st>>>(ww);
    DPN_LAUNCH_OK();
  }
#ifdef DPN_DEBUG_BUILD
  if (phase_debug) {
    long long h[16];
    DPN_CUDA_OK(cudaStreamSynchronize(st));
    DPN_CUDA_OK(cudaMemcpy(h, c.dbg, sizeof(h), cudaMemcpyDeviceToHost));
    const double n1 = h[6] > 0 ? (double)h[6] : 1.0, n2 = h[14] > 0 ? (double)h[14] : 1.0;
    fprintf(stderr, "[dpn phase] pass1 per CTA (cycles): mma-thread total %.0f | wait weights %.0f | wait epilogue %.0f | wait A tile %.0f || "
                    "epilogue-thread total %.0f | wait accumulator %.0f | acc ready -> tile handed over %.0f\n", h[0] / n1, h[1] / n1, h[2] / n1, h[3] / n1, h[4] / n1, h[5] / n1, h[7] / n1);
    fprintf(stderr, "[dpn phase] pass2 per CTA (cycles): mma-thread total %.0f | wait weights %.0f | wait epilogue %.0f || "
                    "epilogue-thread total %.0f | wait accumulator %.0f | compute %.0f (of which prologue %.0f)\n", h[8] / n2, h[9] / n2, h[10] / n2, h[12] / n2, h[13] / n2, h[15] / n2, h[11] / n2);
  }
#endif
  if (want_bwd) {
    if ((rc = f32::launch_finalize(Kn, Wt, c.vc, c.vg, c.sdo, *J.grads, st))) return rc;
  }
  return 0;
}

int run(const Job& J, cudaStream_t st) {
  // (a single scaled fp16 plane - run_planes<1, true> - was measured too: 12.1 ms per call against 10.8 ms for bf16, Jacobian /
  //  gradient errors 1e-2..3e-2 against 5e-2: ReLU-mask flips dominate both, not worth a fifth mode)
  if (J.shape.mode == DPN_MODE_F16X3 || J.shape.mode == DPN_MODE_F16X3A) return run_planes<2, true>(J, st);
  if (J.shape.mode == DPN_MODE_BF16X3) return run_planes<2, false>(J, st);
  return run_planes<1, false>(J, st);
}

}  // namespace tc
}  // namespace dpn
