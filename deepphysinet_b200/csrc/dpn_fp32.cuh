// DPN_MODE_FP32 internals (see dpn_fp32.cu) and the job description shared by both modes.
#pragma once
#include "dpn_common.cuh"

namespace dpn {

// JOB_JAC_FWD / JOB_JAC_BWD: dpn_decoder_jac_fwd / _bwd - values and Jacobian out, caller seeds on both in.
enum JobKind { JOB_PDE = 0, JOB_DEC_FWD = 1, JOB_DEC_BWD = 2, JOB_LATTICE = 3, JOB_JAC_FWD = 4, JOB_JAC_BWD = 5 };

// dpn_decoder_lattice, validated by dpn_api.cu: the lattice, the coarse stack it samples and the de-normalisation of the output.
struct LatticeJob {
  DpnLattice g;
  DpnSampler s;
  const float* coarse;       // [B][Tt][Hc][Wc][6]
  float lo[3], hi[3];        // x, y, t are clamped to this fp32 box inside the coarse stack (the validated domain)
  float sd[6], mu[6];        // std, mean rounded double -> fp32: out = o * sd + mu with two roundings, as torch's o * std + mean
};

// Per chunk (dpn_sampler.cu): staged x, y, t [nb][P] and coord_data [nb][P][6] of nodes p0 .. p0 + P - 1 of samples b0 .. b0 + nb - 1;
// then out[b * out_bstride + p * 6 + k] = o[(b * srow + p) * 6 + k] * sd[k] + mu[k] for the same nodes (out at sample b0, node p0).
int launch_lattice(const LatticeJob& L, int b0, int nb, int p0, int P, float* x, float* y, float* t, float* coord_data, cudaStream_t st);
int launch_lattice_emit(const LatticeJob& L, int nb, int P, const float* o, size_t srow, float* out, size_t out_bstride, cudaStream_t st);

// One library call, validated and normalised by dpn_api.cu.
struct Job {
  JobKind kind;
  DpnShape shape;
  DevConsts dc;
  const DpnPoints* pts;
  const DpnWeights* w;
  const DpnPdeOut* out;     // JOB_PDE
  const DpnMargin* margin;  // JOB_PDE, optional: supervised SmoothL1 data loss on the same points
  const DpnGrads* grads;    // JOB_PDE (optional), JOB_DEC_BWD, JOB_JAC_BWD
  float* o;                 // JOB_DEC_FWD, JOB_JAC_FWD: normalised [B*N][K];  JOB_LATTICE: physical [B][N][6]
  float* jac;               // JOB_JAC_FWD: [B*N][K][3] d o / d(x, y, t)
  LatticeJob lat;           // JOB_LATTICE
  const float* d_o;         // JOB_DEC_BWD; JOB_JAC_BWD (may be NULL)
  const float* d_jac;       // JOB_JAC_BWD (may be NULL): [B*N][K][3]
  void* workspace;
  size_t workspace_bytes;
  int chunk;                // points per sample per internal pass
};

namespace f32 {

enum { NT = 0, NN = 1, TN = 2 };

struct Gemm {
  int M, N, K;
  const float* A; int lda; size_t sA;
  const float* B; int ldb; size_t sB;
  const float* bias; size_t sBias;
  const float* mask; size_t sMask;
  const float* addsrc; size_t sAdd;
  const float* rowscale; int sRow; int ldRow;
  float* out; size_t sOut;
  float* out2; size_t sOut2;
  int relu, accumulate, atomic, ksplit;
};

struct Workspace {
  float *pe, *pe6, *o, *od, *dov, *dod;
  float *H1, *CC, *GG, *UM, *YT, *QM, *HT, *CT, *ZH, *ZC, *GZ;
  float *JIN, *ZP, *ZD;
  float *uvec, *wo2, *cst, *bsum, *vc, *vg, *sdo;
  float *lx, *ly, *lt, *lcd;  // lattice staging (values-only carve only)
  size_t bytes;
};

constexpr int DEFAULT_CHUNK = 16384;

size_t workspace_bytes(int P, int Kn, int B);
size_t lattice_workspace_bytes(int P, int Kn, int B);
int launch_gemm(const Gemm& g, int layout, int batches, cudaStream_t st);
int run(const Job& job, cudaStream_t st);

// pieces reused by the tensor-core mode
int launch_prep(int B, int Kn, const DpnWeights& Wt, float* uvec, float* wo2, float* cst, float* bsum, cudaStream_t st);
int launch_residual(const DevConsts& DC, int B, int P, size_t srow, size_t sq, const float* o, const float* od, const float* f,
                    double inv_n, double seed_scale, double* loss6, float* dov, float* dod, float* vals, float* jac, cudaStream_t st);
int launch_margin(int B, int P, size_t srow, size_t sq, const float* o, const float* target, const DpnMargin& M, double inv_n,
                  double seed_scale, double* loss, float* dov, float* o_out, cudaStream_t st);
// Caller seeds of P points per sample (samples srow workspace rows / sq caller points apart) -> dov [..][Kn], dod [..][Kn][3]
// (dod may be NULL: values-only backward); a NULL d_o / d_jac is a zero seed.
int launch_seed_in(const DevConsts& DC, int B, int P, int Kn, size_t srow, size_t sq, const float* d_o, const float* d_jac,
                   double seed_scale, float* dov, float* dod, cudaStream_t st);
// o [..][Kn], od [..][Kn][3] of the workspace -> the caller's o [B*N][Kn] and jac = od (sx, sy, st) [B*N][Kn][3].
int launch_fields(const DevConsts& DC, int B, int P, int Kn, size_t srow, size_t sq, const float* o, const float* od, float* o_out,
                  float* jac, cudaStream_t st);
int launch_finalize(int Kn, const DpnWeights& Wt, const float* vc, const float* vg, const float* sdo, const DpnGrads& G,
                    cudaStream_t st);

}  // namespace f32
}  // namespace dpn
