/*
 * dpn_b200.h - C ABI of libdpn_b200.so: the decoder-query + PDE-residual hot path of
 * flyakon/DeepPhysiNet, hand-written for NVIDIA B200 (sm_100a).
 *
 * The reference has no FFI / plugin layer: the boundary it offers is two Python call signatures,
 *     PhysicsNet.forward(field_x, coord_x, coord_data, forecast_h)        DeepPhysiNet/model/physics_net.py:41-55
 *     InterfacePhysics.place_one_batch(x, y, t, f, field_data, ...)       DeepPhysiNet/interface/interface_physics.py:271-320
 * This library is what a ctypes binding underneath those two methods calls (INTEGRATION.md shows the
 * stub).  Every entry point takes plain pointers and sizes; all pointers are DEVICE pointers unless
 * the name says host; the caller owns every buffer including the workspace; nothing is allocated or
 * synchronised inside a call; work is enqueued on the given CUDA stream.
 *
 * Layout conventions (all row-major, fp32 unless stated):
 *   B  = samples (independent encoder outputs / weight sets),  N = query points per sample,
 *   K  = coordinate nets (6 for the PDE path: u, v, p, T, q, rho = coord_data column order,
 *        physics_net.py:49-54),  H = 256 hidden, C = 192 encoded-coordinate width.
 *   Generated (hyper-network) tensors are per sample:  W1 [B,K,H,C]  b1 [B,K,H]  W2 [B,K,H,H]  b2 [B,K,H]
 *   (variable_net.py:57-65) and e [B,K,H] = fore_h_fc(PE(fore_h)) (variable_net.py:75-78).
 *   Static tensors are shared by all samples:  Wd [K,H,C] bd [K,H] (data_input_fc), Wa [K,H,H] ba [K,H]
 *   (cat_fc1.fc.0), Wb [K,H,H] bb [K,H] (cat_fc1.fc.2), wo [K,H] bo [K] (out_fc).
 *
 * Return value: 0 on success, otherwise a cudaError_t-style / DPN_E_* code; dpn_last_error() gives text.
 */
#ifndef DPN_B200_H_
#define DPN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPN_ABI_VERSION 2

#define DPN_H 256
#define DPN_C 192
#define DPN_MAX_NETS 6

/* Arithmetic of the dense contractions. */
enum {
  DPN_MODE_FP32 = 0,  /* CUDA-core fp32 FMA everywhere: the 1e-4 parity mode                              */
  DPN_MODE_BF16 = 1,  /* tcgen05 kind::f16 (bf16 operands, fp32 TMEM accumulators); tolerance in DESIGN.md */
  DPN_MODE_BF16X3 = 2,/* tcgen05, every operand split into bf16 hi + lo (16 mantissa bits), three MMAs per
                         contraction (lo*hi + hi*lo + hi*hi); tolerance in DESIGN.md                        */
  DPN_MODE_F16X3 = 3, /* same with fp16 hi + lo (22 mantissa bits) and exact power-of-two scaling of every
                         operand tile from rigorous L1-norm bounds: fp32-class results on the tensor cores */
  DPN_MODE_F16X3A = 4 /* F16X3 with CROSS-FIRST accumulation of the three GEMMs that decide the ReLU masks: their
                         lo*hi / hi*lo products are issued before any hi*hi product, so the tensor core's
                         round-toward-zero accumulation truncates 16 instead of 48 times per pre-activation (2.6x
                         smaller error, values at 7e-8); 6 % slower (DESIGN.md section 6)                  */
};

enum {
  DPN_OK = 0,
  DPN_E_INVALID = 10001,    /* bad argument (null pointer, unsupported size, misaligned buffer) */
  DPN_E_WORKSPACE = 10002,  /* workspace too small: call dpn_workspace_bytes                    */
  DPN_E_UNSUPPORTED = 10003 /* device is not sm_100 / mode not built                           */
};

/* Problem shape.  n_norm is the divisor of the per-sample mean (MSELoss, losses/builder.py:10): the
 * total number of points of the sample, which exceeds N when one sample's points are sharded across
 * GPUs (SURVEY 8(e) level 2).  seed_scale multiplies dL/d(theta) (1/B for the DDP sample mean). */
typedef struct DpnShape {
  int32_t B;
  int32_t N;
  int32_t K;
  int32_t mode;
  int64_t n_norm;     /* 0 -> N */
  float seed_scale;   /* 0 -> 1 */
  int32_t chunk;      /* points per sample processed per internal pass; 0 -> library default */
} DpnShape;

/* Geometry, normalisation and physics constants.  Defaults: configs/DeepPhysiNet_NCEP_cfg.py:64-83,
 * :93-95,:139-148 and interface_physics.py:126,146,177,322-332.  Order of the 6-arrays: u,v,p,T,q,rho;
 * order of factor[]: motion_u, motion_v, continuous, energy, vapor, gas. */
typedef struct DpnConsts {
  double dx, dy;          /* grid spacing [m]                                                     */
  int32_t lat_size, lon_size;
  double t_span;          /* pred_t_span [s]                                                      */
  int32_t with_clip;      /* InterfacePhysics.with_clip (interface_physics.py:258-261)            */
  int32_t pad_;
  double mean[6], std[6], lo[6], hi[6];
  double factor[6];
  double c_p, L, R_v, R_d;
  /* fp32 frequency buffers of SineCosPE (utils/position_encoding.py:27,33): the coordinate instance
   * (interface_physics.py:44, 32 bands) and the data instance (variable_net.py:45, 16 bands).
   * band_coord[0] == 0 -> the library fills in 2**linspace(0,4,n) itself. */
  float band_coord[32];
  float band_data[16];
} DpnConsts;

/* Per-point inputs.  Either (x,y,t) or coord_pe is given:
 *   x,y,t  [B*N]       physical coordinates (metres, seconds) - required for anything involving d/dx,dy,dt
 *   coord_pe [B*N,C]   already encoded coordinates (PhysicsNet.forward surface) - values only
 *   f      [B*N]       Coriolis parameter (dataset/physics_dataset.py:521-526); PDE path only
 *   coord_data [B*N,6] interpolated coarse field (dataset/physics_dataset.py:477-486)
 *   ref    [B*N,K]     residual skip; NULL -> coord_data[:, k] (physics_net.py:49-54)                */
typedef struct DpnPoints {
  const float *x, *y, *t, *f;
  const float *coord_pe;
  const float *coord_data;
  const float *ref;
} DpnPoints;

typedef struct DpnWeights {
  const float *W1, *b1, *W2, *b2, *e;            /* generated, per sample */
  const float *Wd, *bd, *Wa, *ba, *Wb, *bb, *wo, *bo; /* static              */
} DpnWeights;

/* Gradients, same shapes as DpnWeights; the library OVERWRITES them (zero-fills first). */
typedef struct DpnGrads {
  float *W1, *b1, *W2, *b2, *e;
  float *Wd, *bd, *Wa, *ba, *Wb, *bb, *wo, *bo;
} DpnGrads;

/* Outputs of the PDE path.
 *   loss_terms [B,6] double: factor_e * sum_p r_e^2 / n_norm   (interface_physics.py:285-299)
 *   vals [B*N,6]   physical values after inverse_norm (+clip)    - optional (NULL to skip)
 *   jac  [B*N,6,3] d(vals)/d(x,y,t) as InterfacePhysics.gradient - optional (NULL to skip)            */
typedef struct DpnPdeOut {
  double *loss_terms;
  float *vals;
  float *jac;
} DpnPdeOut;

int dpn_abi_version(void);

/* Copies the last error text of the calling thread into buf (NUL-terminated); returns its length. */
size_t dpn_last_error(char *buf, size_t cap);

/* Bytes of device workspace the calls below need for this shape (256-byte aligned base required). */
int dpn_workspace_bytes(const DpnShape *shape, size_t *bytes);

/* Replaces InterfacePhysics.place_one_batch (interface_physics.py:271-320) followed by
 * train_loss.backward() (:506/:1056) for the decoder part: per sample, six residual loss terms and
 * d(sum of terms)/d(every DpnWeights tensor) * seed_scale.  grads may be NULL (forward/loss only). */
int dpn_pde_fwd_bwd(const DpnShape *shape, const DpnConsts *consts, const DpnPoints *pts,
                    const DpnWeights *w, const DpnPdeOut *out, const DpnGrads *grads,
                    void *workspace, size_t workspace_bytes, void *cuda_stream);

/* The supervised data loss of the train loop on the SAME points as a PDE call (SURVEY 8(f) N1): the reference evaluates the
 * margin (label) points twice per step - values only for WeightSmoothL1Loss (interface_physics.py:464-474,
 * losses/weights_loss.py:12-20) and again inside place_one_batch for their PDE residual (:489-496).  With `margin` set the
 * PDE call adds, per sample,  loss[b] = factor * mean_{N x 6} smooth_l1(o - target; beta)  (o = the six NORMALISED net outputs,
 * exactly what PhysicsNet.forward returns) and the gradients it writes are d(sum of the six PDE terms + loss[b]) / d(weights):
 * one forward, one reverse sweep, one backward for both losses. */
typedef struct DpnMargin {
  const float *target;  /* [B*N,6] normalised observations (margin_data), u,v,p,T,q,rho order            */
  double beta;          /* SmoothL1 transition (cfg train_cfg.losses: beta = 0.1)                        */
  double factor;        /* margin_factor (cfg: 1e6)                                                      */
  double *loss;         /* out [B]                                                                       */
  float *o;             /* out [B*N,6] normalised values, optional (NULL to skip)                         */
} DpnMargin;

int dpn_pde_margin_fwd_bwd(const DpnShape *shape, const DpnConsts *consts, const DpnPoints *pts,
                           const DpnWeights *w, const DpnMargin *margin, const DpnPdeOut *out,
                           const DpnGrads *grads, void *workspace, size_t workspace_bytes, void *cuda_stream);

/* Replaces the six VariableNet.forward calls of PhysicsNet.forward (physics_net.py:49-54,
 * variable_net.py:67-87): normalised outputs o [B*N,K].  Values only (dense-grid inference,
 * interface_physics.py:538-563, and the supervised margin loss :467-474). */
int dpn_decoder_fwd(const DpnShape *shape, const DpnConsts *consts, const DpnPoints *pts,
                    const DpnWeights *w, float *o, void *workspace, size_t workspace_bytes,
                    void *cuda_stream);

/* Backward of dpn_decoder_fwd: given d_o [B*N,K] = dL/do, writes dL/d(every DpnWeights tensor) * seed_scale. */
int dpn_decoder_bwd(const DpnShape *shape, const DpnConsts *consts, const DpnPoints *pts,
                    const DpnWeights *w, const float *d_o, const DpnGrads *grads,
                    void *workspace, size_t workspace_bytes, void *cuda_stream);

/* Query-point producer (SURVEY 8(f) N2).  Replaces the CPU xarray trilinear interpolation of the normalised coarse
 * field stack (dataset/physics_dataset.py:477-486, :406-415, :567-576) and get_coriolis (:521-526).
 *   coarse     [B, Tt, Hc, Wc, 6]  normalised coarse field, channel-last (u10,v10,pres,t2,q2,rio)
 *   x, y, t    [B*N]   query coordinates in the units of DpnPoints (x = fine-cell index * dx, t in seconds)
 *   coord_data [B*N,6] out;   f [B*N] out (may be NULL): 2 omega sin(begin_lat + (y/dy) deg_per_cell)
 * Values only: the reference never differentiates through this interpolation. */
typedef struct DpnSampler {
  int32_t B, N;
  int32_t Tt, Hc, Wc;          /* 5, 37, 65 in the reference configuration */
  int32_t pad_;
  double dx, dy;               /* fine grid spacing [m] */
  double cells_per_coarse;     /* fine cells per coarse cell: 4 (0.25 deg over 1 deg) */
  double t_step;               /* seconds between coarse time slices: 6 h */
  double begin_lat, deg_per_cell, omega;
} DpnSampler;

int dpn_sample_field(const DpnSampler *s, const float *coarse, const float *x, const float *y, const float *t,
                     float *coord_data, float *f, void *cuda_stream);

/* Query-point generator (SURVEY 8(f) N2, the other half of the producer): replaces the numpy draws of
 * dataset/physics_dataset.py:442-446 (interior points: x = U[0,1) (W-1) dx, y = U[0,1) (H-1) dy, t = randint(0, t_steps) dt) and
 * :334-338 (margin points: x = randint(0, W) dx, y = randint(0, H) dy - grid nodes) with a counter-based generator on the GPU:
 * Philox4x32-10, key = seed, counter = (point index + offset, sample, 0): one 128-bit block per point, words 0/1/2 -> x/y/t.
 * U[0,1) = (word >> 8) 2^-24; randint(0, n) = (word * n) >> 32.  Same distributions as the reference, NOT the same stream as
 * numpy's MT19937 (oracle/query_oracle.py restates the generator bit for bit).  With `sampler` and `coarse` given the same kernel
 * also interpolates coord_data and evaluates f for the points it just drew (dpn_sample_field semantics), so a training step's
 * per-point inputs are produced by ONE launch and never exist on the host.
 *   x, y, t [B*N] out;  coord_data [B*N,6], f [B*N] out (NULL with sampler == NULL). */
typedef struct DpnQueryGen {
  int32_t B, N;
  int32_t lat_size, lon_size;  /* fine grid nodes: 145, 257                                                   */
  int32_t t_steps;             /* exclusive upper bound of the time draw: input_time_step * nums + 1 = 25      */
  int32_t on_grid;             /* 0: interior (continuous x, y)   1: margin (integer grid nodes)               */
  double dx, dy, dt;           /* metres per fine cell, seconds per time unit (3600)                           */
  uint64_t seed, offset;
} DpnQueryGen;

int dpn_generate_queries(const DpnQueryGen *g, const DpnSampler *sampler, const float *coarse, float *x, float *y,
                         float *t, float *coord_data, float *f, void *cuda_stream);

/* Lattice inference: the six decoders on a regular space-time lattice, for B samples, as physical fields.  Generalises the
 * dense forward of interface_physics.py:538-606 and physics_dataset.get_margin_grid :528-588 to any spacing, sub-region and
 * lead times.  Node (k, j, i) of every sample sits at
 *   x = x0 + i sx,  y = y0 + j sy  (metres, DpnPoints units),  t = t0 + k st  (seconds);  i < nx, j < ny, k < nt.
 * Output order is [B, nt, ny, nx, 6]: t slowest, x fastest. */
typedef struct DpnLattice {
  int32_t nx, ny, nt, pad_;
  double x0, y0, t0;
  double sx, sy, st;
} DpnLattice;

/* Bytes of device workspace dpn_decoder_lattice needs for this shape: the values-only part of the dpn_workspace_bytes carve
 * (weight images, coordinate / data features, outputs) plus per-point staging of x, y, t and coord_data - about 2.3 KB per point
 * in flight in the split modes against 41 KB for dpn_workspace_bytes. */
int dpn_lattice_workspace_bytes(const DpnShape *shape, size_t *bytes);

/* out[b, k, j, i, :] = o * std + mean (inverse_norm WITHOUT clip, as the reference's dense forward :533) of the six nets at node
 * (k, j, i) of sample b.  Per chunk of nodes the library generates the coordinates (fp64, rounded once to fp32) and samples
 * coord_data from coarse [B,Tt,Hc,Wc,6] with dpn_sample_field's interpolation; nothing per point exists on the host.
 *   shape  B samples, N = nx ny nt (must fit int32), K = 6, any mode; chunk honoured as elsewhere
 *   s      coarse-stack geometry exactly as in dpn_sample_field; s->B, s->N must equal shape->B, shape->N; Coriolis fields unused
 *   w      generated weights per sample, as everywhere;  out [B, nt, ny, nx, 6] physical values
 * DPN_E_INVALID (with dpn_last_error text) for zero sizes, non-positive spacing, a first or last node outside the coarse stack in
 * x, y or t, B / N mismatches and NULL pointers.  Values only. */
int dpn_decoder_lattice(const DpnShape *shape, const DpnConsts *consts, const DpnLattice *g, const DpnSampler *s,
                        const float *coarse, const DpnWeights *w, float *out,
                        void *workspace, size_t workspace_bytes, void *cuda_stream);

/* Introspection for tests and bench: number of kernels the last call on this thread launched. */
int dpn_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DPN_B200_H_ */
