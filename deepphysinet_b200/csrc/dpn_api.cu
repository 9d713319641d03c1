// extern "C" surface of libdpn_b200.so (include/dpn_b200.h): argument validation, mode dispatch.
#include <math.h>
#include <stdarg.h>

#include <atomic>

#include "dpn_fp32.cuh"
#include "dpn_tc.cuh"

namespace dpn {

int run_sampler(const DpnSampler& S, const float* coarse, const float* x, const float* y, const float* t,
                float* coord_data, float* f, cudaStream_t st);

int run_query_gen(const DpnQueryGen& G, const DpnSampler* S, const float* coarse, float* x, float* y, float* t,
                  float* coord_data, float* f, cudaStream_t st);

static thread_local char g_err[1024] = "";
thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int f32_chunk(const DpnShape& s) {
  int c = s.chunk > 0 ? s.chunk : f32::DEFAULT_CHUNK;
  return c < s.N ? c : s.N;
}

static int planes(const DpnShape& s) { return (s.mode == DPN_MODE_BF16X3 || s.mode == DPN_MODE_F16X3 || s.mode == DPN_MODE_F16X3A) ? 2 : 1; }

static int tc_chunk(const DpnShape& s) {
  int c = s.chunk > 0 ? (s.chunk + 127) / 128 * 128 : tc::default_chunk(s.B, planes(s));
  const int n = (s.N + 127) / 128 * 128;
  return c < n ? c : n;
}

static int check_shape(const DpnShape* s) {
  if (!s) { set_error("shape is NULL"); return DPN_E_INVALID; }
  if (s->B <= 0 || s->N <= 0 || s->K <= 0 || s->K > DPN_MAX_NETS) {
    set_error("bad shape B=%d N=%d K=%d (need B>0, N>0, 1<=K<=6)", s->B, s->N, s->K);
    return DPN_E_INVALID;
  }
  if (s->mode < DPN_MODE_FP32 || s->mode > DPN_MODE_F16X3A) {
    set_error("unknown mode %d", s->mode);
    return DPN_E_INVALID;
  }
  return 0;
}

static int check_device() {
  // cudaGetDeviceProperties costs milliseconds per call: ask for the one attribute, once per device
  static std::atomic<int> major_of[64];                               // zero-initialised; threads (one per GPU) may race to fill an entry
  int dev = 0;
  DPN_CUDA_OK(cudaGetDevice(&dev));
  int major = (dev >= 0 && dev < 64) ? major_of[dev].load(std::memory_order_relaxed) : 0;
  if (major == 0) {
    DPN_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (dev >= 0 && dev < 64) major_of[dev].store(major, std::memory_order_relaxed);
  }
  if (major != 10) {
    set_error("libdpn_b200 is built for sm_100a only; device %d has compute capability major %d", dev, major);
    return DPN_E_UNSUPPORTED;
  }
  return 0;
}

static size_t ws_bytes(const DpnShape& s) {
  if (s.mode == DPN_MODE_FP32) return f32::workspace_bytes(f32_chunk(s), s.K, s.B);
  return tc::workspace_bytes(tc_chunk(s), s.K, s.B, planes(s));
}

static size_t lattice_ws_bytes(const DpnShape& s) {
  if (s.mode == DPN_MODE_FP32) return f32::lattice_workspace_bytes(f32_chunk(s), s.K, s.B);
  return tc::lattice_workspace_bytes(tc_chunk(s), s.K, s.B, planes(s));
}

static int dispatch(Job& job, void* stream) {
  g_launches = 0;
  int rc = check_device();
  if (rc) return rc;
  const size_t need = job.kind == JOB_LATTICE ? lattice_ws_bytes(job.shape) : ws_bytes(job.shape);
  if (!job.workspace || job.workspace_bytes < need) {
    set_error("workspace too small: have %zu bytes, need %zu", job.workspace_bytes, need);
    return DPN_E_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(job.workspace) & 255) != 0) {
    set_error("workspace must be 256-byte aligned");
    return DPN_E_INVALID;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // `mode` is honoured on every surface: pre-encoded coordinates (coord_pe), an explicit skip (ref) and K < 6 nets run on the
  // tensor cores as well (tc::encode_kernel takes the caller's encoding; the epilogues take ref)
  const bool tensor = job.shape.mode != DPN_MODE_FP32;
  job.chunk = tensor ? tc_chunk(job.shape) : f32_chunk(job.shape);
  return tensor ? tc::run(job, st) : f32::run(job, st);
}

static int check_weights(const DpnWeights* w) {
  const void* ws[] = {w->W1, w->b1, w->W2, w->b2, w->e, w->Wd, w->bd, w->Wa, w->ba, w->Wb, w->bb, w->wo, w->bo};
  for (const void* q : ws)
    if (!q || (reinterpret_cast<uintptr_t>(q) & 15)) { set_error("a weight pointer is NULL or not 16-byte aligned"); return DPN_E_INVALID; }
  return 0;
}

static int check_common(const DpnShape* s, const DpnConsts* c, const DpnPoints* p, const DpnWeights* w) {
  int rc = check_shape(s);
  if (rc) return rc;
  if (!c || !p || !w) { set_error("consts / points / weights is NULL"); return DPN_E_INVALID; }
  if ((rc = check_weights(w))) return rc;
  if (!p->coord_data) { set_error("coord_data is NULL"); return DPN_E_INVALID; }
  if (!p->coord_pe && !(p->x && p->y && p->t)) { set_error("need either coord_pe or x,y,t"); return DPN_E_INVALID; }
  return 0;
}

static bool sampler_ok(const DpnSampler* s) {
  return s->B > 0 && s->N > 0 && s->Tt >= 2 && s->Hc >= 2 && s->Wc >= 2 && s->cells_per_coarse > 0 && s->t_step > 0 &&
         s->dx > 0 && s->dy > 0;
}

// The first and last node of one lattice axis, in fp64, must lie in the coarse stack [0, (n - 1) cell] with the tolerance of
// sample_point (1e-9 coarse cells); the fp32 box the kernel clamps to is [0, largest float <= the far edge].
static int check_axis(const char* name, double v0, double step, int n, double cell, int ncoarse, float* lo, float* hi) {
  const double first = v0, last = v0 + (double)(n - 1) * step, edge = (double)(ncoarse - 1) * cell;
  constexpr double EPS = 1e-9;
  if (!(first / cell >= -EPS && last / cell <= (double)(ncoarse - 1) + EPS)) {
    set_error("dpn_decoder_lattice: lattice %s range [%.9g, %.9g] lies outside the coarse stack [0, %.9g]", name, first, last, edge);
    return DPN_E_INVALID;
  }
  float e = (float)edge;
  if ((double)e > edge) e = nextafterf(e, 0.f);
  *lo = 0.f;
  *hi = e;
  return 0;
}

static int check_grads(const DpnGrads* g) {
  const void* gs[] = {g->W1, g->b1, g->W2, g->b2, g->e, g->Wd, g->bd, g->Wa, g->ba, g->Wb, g->bb, g->wo, g->bo};
  for (const void* q : gs)
    if (!q || (reinterpret_cast<uintptr_t>(q) & 15)) { set_error("a gradient pointer is NULL or not 16-byte aligned"); return DPN_E_INVALID; }
  return 0;
}

}  // namespace dpn

using namespace dpn;

extern "C" {

int dpn_abi_version(void) { return DPN_ABI_VERSION; }

size_t dpn_last_error(char* buf, size_t cap) {
  if (!buf || cap == 0) return strlen(g_err);
  strncpy(buf, g_err, cap - 1);
  buf[cap - 1] = 0;
  return strlen(buf);
}

int dpn_last_launch_count(void) { return g_launches; }

int dpn_workspace_bytes(const DpnShape* shape, size_t* bytes) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!bytes) { set_error("bytes is NULL"); return DPN_E_INVALID; }
  *bytes = ws_bytes(*shape);
  return 0;
}

int dpn_pde_margin_fwd_bwd(const DpnShape* shape, const DpnConsts* consts, const DpnPoints* pts, const DpnWeights* w,
                           const DpnMargin* margin, const DpnPdeOut* out, const DpnGrads* grads, void* workspace,
                           size_t workspace_bytes, void* cuda_stream) {
  int rc = check_common(shape, consts, pts, w);
  if (rc) return rc;
  if (shape->K != 6) { set_error("the PDE residual needs K = 6 nets (u,v,p,T,q,rho), got %d", shape->K); return DPN_E_INVALID; }
  if (!(pts->x && pts->y && pts->t && pts->f)) { set_error("the PDE path needs x, y, t and f"); return DPN_E_INVALID; }
  if (pts->coord_pe || pts->ref) { set_error("the PDE path derives the encoding from x,y,t and the skip from coord_data"); return DPN_E_INVALID; }
  if (!out || !out->loss_terms) { set_error("out->loss_terms is NULL"); return DPN_E_INVALID; }
  if (grads && (rc = check_grads(grads))) return rc;
  Job job;
  memset(&job, 0, sizeof(job));
  job.kind = JOB_PDE; job.shape = *shape; job.dc = make_dev_consts(*consts);
  if (margin && (!margin->target || !margin->loss || !(margin->beta > 0.0))) {
    set_error("margin needs target, loss and beta > 0");
    return DPN_E_INVALID;
  }
  job.pts = pts; job.w = w; job.out = out; job.grads = grads; job.margin = margin;
  job.workspace = workspace; job.workspace_bytes = workspace_bytes;
  return dispatch(job, cuda_stream);
}

int dpn_pde_fwd_bwd(const DpnShape* shape, const DpnConsts* consts, const DpnPoints* pts, const DpnWeights* w,
                    const DpnPdeOut* out, const DpnGrads* grads, void* workspace, size_t workspace_bytes,
                    void* cuda_stream) {
  return dpn_pde_margin_fwd_bwd(shape, consts, pts, w, nullptr, out, grads, workspace, workspace_bytes, cuda_stream);
}

int dpn_decoder_fwd(const DpnShape* shape, const DpnConsts* consts, const DpnPoints* pts, const DpnWeights* w,
                    float* o, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_common(shape, consts, pts, w);
  if (rc) return rc;
  if (!o) { set_error("o is NULL"); return DPN_E_INVALID; }
  if (!pts->ref && shape->K != 6) { set_error("ref may only be NULL for K = 6"); return DPN_E_INVALID; }
  Job job;
  memset(&job, 0, sizeof(job));
  job.kind = JOB_DEC_FWD; job.shape = *shape; job.dc = make_dev_consts(*consts);
  job.pts = pts; job.w = w; job.o = o;
  job.workspace = workspace; job.workspace_bytes = workspace_bytes;
  return dispatch(job, cuda_stream);
}

int dpn_decoder_bwd(const DpnShape* shape, const DpnConsts* consts, const DpnPoints* pts, const DpnWeights* w,
                    const float* d_o, const DpnGrads* grads, void* workspace, size_t workspace_bytes,
                    void* cuda_stream) {
  int rc = check_common(shape, consts, pts, w);
  if (rc) return rc;
  if (!d_o || !grads) { set_error("d_o / grads is NULL"); return DPN_E_INVALID; }
  if (!pts->ref && shape->K != 6) { set_error("ref may only be NULL for K = 6"); return DPN_E_INVALID; }
  if ((rc = check_grads(grads))) return rc;
  Job job;
  memset(&job, 0, sizeof(job));
  job.kind = JOB_DEC_BWD; job.shape = *shape; job.dc = make_dev_consts(*consts);
  job.pts = pts; job.w = w; job.d_o = d_o; job.grads = grads;
  job.workspace = workspace; job.workspace_bytes = workspace_bytes;
  return dispatch(job, cuda_stream);
}

int dpn_lattice_workspace_bytes(const DpnShape* shape, size_t* bytes) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!bytes) { set_error("bytes is NULL"); return DPN_E_INVALID; }
  *bytes = lattice_ws_bytes(*shape);
  return 0;
}

int dpn_decoder_lattice(const DpnShape* shape, const DpnConsts* consts, const DpnLattice* g, const DpnSampler* s,
                        const float* coarse, const DpnWeights* w, float* out, void* workspace, size_t workspace_bytes,
                        void* cuda_stream) {
  int rc = check_shape(shape);
  if (rc) return rc;
  if (!consts || !g || !s || !coarse || !w || !out) { set_error("dpn_decoder_lattice: NULL argument"); return DPN_E_INVALID; }
  if ((rc = check_weights(w))) return rc;
  if (shape->K != 6) { set_error("dpn_decoder_lattice: needs K = 6 nets (u,v,p,T,q,rho), got %d", shape->K); return DPN_E_INVALID; }
  if (g->nx <= 0 || g->ny <= 0 || g->nt <= 0) {
    set_error("dpn_decoder_lattice: lattice sizes must be positive, got nx=%d ny=%d nt=%d", g->nx, g->ny, g->nt);
    return DPN_E_INVALID;
  }
  if (!(g->sx > 0 && g->sy > 0 && g->st > 0) || !isfinite(g->sx) || !isfinite(g->sy) || !isfinite(g->st)) {
    set_error("dpn_decoder_lattice: lattice spacing must be positive and finite, got sx=%g sy=%g st=%g", g->sx, g->sy, g->st);
    return DPN_E_INVALID;
  }
  const long long n = (long long)g->nx * g->ny * g->nt;
  if (n > 2147483647LL) { set_error("dpn_decoder_lattice: nx ny nt = %lld nodes does not fit int32", n); return DPN_E_INVALID; }
  if (n != shape->N) { set_error("dpn_decoder_lattice: shape N = %d but the lattice has nx ny nt = %lld nodes", shape->N, n); return DPN_E_INVALID; }
  if (!sampler_ok(s)) {
    set_error("dpn_decoder_lattice: bad sampler shape B=%d N=%d T=%d H=%d W=%d", s->B, s->N, s->Tt, s->Hc, s->Wc);
    return DPN_E_INVALID;
  }
  if (s->B != shape->B || s->N != shape->N) {
    set_error("dpn_decoder_lattice: sampler B=%d N=%d does not match shape B=%d N=%d", s->B, s->N, shape->B, shape->N);
    return DPN_E_INVALID;
  }
  Job job;
  memset(&job, 0, sizeof(job));
  LatticeJob& L = job.lat;
  if ((rc = check_axis("x", g->x0, g->sx, g->nx, s->dx * s->cells_per_coarse, s->Wc, &L.lo[0], &L.hi[0]))) return rc;
  if ((rc = check_axis("y", g->y0, g->sy, g->ny, s->dy * s->cells_per_coarse, s->Hc, &L.lo[1], &L.hi[1]))) return rc;
  if ((rc = check_axis("t", g->t0, g->st, g->nt, s->t_step, s->Tt, &L.lo[2], &L.hi[2]))) return rc;
  L.g = *g; L.s = *s; L.coarse = coarse;
  for (int k = 0; k < 6; ++k) { L.sd[k] = (float)consts->std[k]; L.mu[k] = (float)consts->mean[k]; }
  job.kind = JOB_LATTICE; job.shape = *shape; job.dc = make_dev_consts(*consts);
  job.w = w; job.o = out;
  job.workspace = workspace; job.workspace_bytes = workspace_bytes;
  return dispatch(job, cuda_stream);
}

int dpn_sample_field(const DpnSampler* s, const float* coarse, const float* x, const float* y, const float* t,
                     float* coord_data, float* f, void* cuda_stream) {
  if (!s || !coarse || !x || !y || !t || !coord_data) { set_error("dpn_sample_field: NULL argument"); return DPN_E_INVALID; }
  if (s->B <= 0 || s->N <= 0 || s->Tt < 2 || s->Hc < 2 || s->Wc < 2 || !(s->cells_per_coarse > 0) || !(s->t_step > 0)) {
    set_error("dpn_sample_field: bad sampler shape B=%d N=%d T=%d H=%d W=%d", s->B, s->N, s->Tt, s->Hc, s->Wc);
    return DPN_E_INVALID;
  }
  g_launches = 0;
  int rc = check_device();
  if (rc) return rc;
  return run_sampler(*s, coarse, x, y, t, coord_data, f, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int dpn_generate_queries(const DpnQueryGen* g, const DpnSampler* s, const float* coarse, float* x, float* y, float* t,
                         float* coord_data, float* f, void* cuda_stream) {
  if (!g || !x || !y || !t) { set_error("dpn_generate_queries: NULL argument"); return DPN_E_INVALID; }
  if (g->B <= 0 || g->N <= 0 || g->lat_size < 2 || g->lon_size < 2 || g->t_steps < 1) {
    set_error("dpn_generate_queries: bad generator B=%d N=%d grid %dx%d t_steps=%d", g->B, g->N, g->lat_size, g->lon_size, g->t_steps);
    return DPN_E_INVALID;
  }
  if (s) {
    if (!coarse || !coord_data) { set_error("dpn_generate_queries: sampler given without coarse / coord_data"); return DPN_E_INVALID; }
    if (s->B != g->B || s->N != g->N || s->Tt < 2 || s->Hc < 2 || s->Wc < 2 || !(s->cells_per_coarse > 0) || !(s->t_step > 0)) {
      set_error("dpn_generate_queries: sampler shape does not match the generator");
      return DPN_E_INVALID;
    }
  }
  g_launches = 0;
  int rc = check_device();
  if (rc) return rc;
  return run_query_gen(*g, s, coarse, x, y, t, coord_data, f, reinterpret_cast<cudaStream_t>(cuda_stream));
}

}  // extern "C"
