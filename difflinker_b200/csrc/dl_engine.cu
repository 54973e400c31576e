// difflinker_b200 engine: C-ABI (include/difflinker_b200.h), weight packing, workspace, launch sequences,
// CUDA-graph replay of the reverse-diffusion loop. Kernels live in kernels_simt.cuh / kernels_tc.cuh.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <map>
#include <string>
#include <vector>

#include "../../include/difflinker_b200.h"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_node_tc.cuh"
#include "kernels_edge_v3.cuh"
#include "diffusion_loss.cuh"

using namespace dl;

static thread_local char g_err[1024] = "";
static void set_err(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess) {                                                              \
      set_err("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));       \
      return DL_ERR_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

namespace {

struct Workspace {
  int B = 0, N = 0;
  float *nm = nullptr, *x0 = nullptr, *xa = nullptr, *xb = nullptr, *h = nullptr, *ABg = nullptr, *ABc = nullptr,
        *agg = nullptr, *z = nullptr, *ABgmax = nullptr, *ABcmax = nullptr, *eps = nullptr;
  float* eps_hat = nullptr;   // dl_diffusion_loss: the Dynamics.forward output on z_t (z holds z_t, eps holds eps_t)
  int* cls = nullptr;
  // cut-off graphs on the tcgen05 path: per-row neighbour lists and packed tile records of the current call (k_nbr)
  int *nbr = nullptr, *recs = nullptr, *xrecs = nullptr, *n_recs = nullptr;
  float4 *x04 = nullptr, *xa4 = nullptr, *xb4 = nullptr;
  int *rowidx = nullptr, *colidx = nullptr, *xrowidx = nullptr, *nr = nullptr, *nc = nullptr, *nxr = nullptr,
      *n_items = nullptr, *xmols = nullptr, *n_xmols = nullptr, *n_xitems = nullptr;
  int4* items = nullptr;
  int4* xitems = nullptr;
  int* tile_ctr = nullptr;
  void* tc_scratch = nullptr;
  // third-generation GCL kernel (kernels_edge_v3.cuh): FC graphs with N <= 64; tensor map of ABg's B halves
  bool v3 = false;
  CUtensorMap tm_abg, tm_abc;
  // per-tile tables of the v3 kernel (tc3::TileTables): set 0 = GCL tiles (plan.items), set 1 = COORD tiles (plan.xitems)
  uint8_t* ts[2] = {nullptr, nullptr};
  int2* tij[2] = {nullptr, nullptr};
  float *td[2] = {nullptr, nullptr}, *td0[2] = {nullptr, nullptr}, *tdmax[2] = {nullptr, nullptr}, *td0max[2] = {nullptr, nullptr};
  float* tcd = nullptr;
  int* cta_begin[2] = {nullptr, nullptr};   // cost-balanced slices of the two tile lists over the v3 kernels' CTAs
  std::vector<void*> allocs;
};

struct HostStage {  // device staging for the *_host entry points
  size_t cap = 0;
  char* buf = nullptr;
};

}  // namespace

struct dl_engine {
  dl_config cfg{};
  int D = 0;
  int num_sms = 0;
  int max_threads_per_sm = 2048;
  int slice_B_full = 0, slice_b0 = 0;   // dl_set_noise_slice: this engine samples rows [b0, b0 + B) of a B_full batch
  bool finalized = false;
  std::map<std::string, std::vector<float>> raw;
  float* wblob = nullptr;      // packed fp32 weights
  void* wblob_tc = nullptr;    // packed fp16 hi/lo tiles
  std::vector<GclW> gcl;       // [L*S]
  std::vector<EqW> eq;         // [L]
  const float *We_t = nullptr, *be = nullptr, *Wo = nullptr, *bo = nullptr;
  Workspace ws;
  cudaStream_t loop_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
  float* coef_dev = nullptr;
  int coef_cap = 0;
  int* step_ctr = nullptr;     // [2]: step_prep, step_fin
  int64_t launches = 0;
  HostStage stage;
  bool use_tc = false;
  bool allow_v3 = true;        // DL_EDGE_V3=0 keeps the second-generation kernel (A/B measurements)
  bool allow_v3_coord = true;  // DL_EDGE_V3_COORD=0: coordinate update on the second-generation kernel
  // pointers of the most recent forward (for dl_time_edge_kernel)
  const int8_t* last_edge_mask = nullptr;
  const float* last_linker_mask = nullptr;
  int last_B = 0, last_N = 0;
};

namespace {

// DL_TIME_KERNELS=1: CUDA-event time of every launch of a (non-captured) forward, accumulated per kernel label and printed
// when the engine is destroyed -- the live (warm-cache, back-to-back) counterpart of the ncu launch list.
struct KernelTimes {
  bool on = false;
  struct Rec { const char* label; cudaEvent_t a, b; };
  std::vector<Rec> pending;
  std::map<std::string, std::pair<double, long>> acc;
  void begin(cudaStream_t st, const char* label) {
    if (!on) return;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) return;
    Rec r{label, nullptr, nullptr};
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
    pending.push_back(r);
  }
  void end(cudaStream_t st) {
    if (!on || pending.empty() || pending.back().b == nullptr) return;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) return;
    cudaEventRecord(pending.back().b, st);
  }
  void collect(cudaStream_t st) {
    if (!on || pending.empty()) return;
    cudaStreamSynchronize(st);
    for (auto& r : pending) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { auto& a = acc[r.label]; a.first += ms; a.second += 1; }
      cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    pending.clear();
  }
  void report() {
    if (!on || acc.empty()) return;
    double tot = 0;
    for (auto& kv : acc) tot += kv.second.first;
    for (auto& kv : acc)
      fprintf(stderr, "[dl times] %-22s %6ld launches  avg %8.2f us  share %5.1f%%\n", kv.first.c_str(), kv.second.second,
              1e3 * kv.second.first / kv.second.second, 100.0 * kv.second.first / tot);
  }
};
KernelTimes g_times;
#define TIMED(label, stream, stmt) do { g_times.begin(stream, label); stmt; g_times.end(stream); } while (0)

struct ExpectedParam {
  std::string name;
  int64_t numel;
};

std::vector<ExpectedParam> expected_params(const dl_config& c) {
  const int D = c.in_node_nf + c.context_node_nf + (c.condition_time ? 1 : 0);
  const int Hh = c.hidden_nf;
  std::vector<ExpectedParam> v;
  v.push_back({"dynamics.embedding.weight", (int64_t)Hh * D});
  v.push_back({"dynamics.embedding.bias", Hh});
  v.push_back({"dynamics.embedding_out.weight", (int64_t)D * Hh});
  v.push_back({"dynamics.embedding_out.bias", D});
  char buf[160];
  for (int l = 0; l < c.n_layers; ++l) {
    for (int s = 0; s < c.inv_sublayers; ++s) {
      snprintf(buf, sizeof(buf), "dynamics.e_block_%d.gcl_%d.", l, s);
      std::string p(buf);
      v.push_back({p + "edge_mlp.0.weight", (int64_t)Hh * (2 * Hh + 2)});
      v.push_back({p + "edge_mlp.0.bias", Hh});
      v.push_back({p + "edge_mlp.2.weight", (int64_t)Hh * Hh});
      v.push_back({p + "edge_mlp.2.bias", Hh});
      v.push_back({p + "node_mlp.0.weight", (int64_t)Hh * 2 * Hh});
      v.push_back({p + "node_mlp.0.bias", Hh});
      v.push_back({p + "node_mlp.2.weight", (int64_t)Hh * Hh});
      v.push_back({p + "node_mlp.2.bias", Hh});
    }
    snprintf(buf, sizeof(buf), "dynamics.e_block_%d.gcl_equiv.", l);
    std::string p(buf);
    v.push_back({p + "coord_mlp.0.weight", (int64_t)Hh * (2 * Hh + 2)});
    v.push_back({p + "coord_mlp.0.bias", Hh});
    v.push_back({p + "coord_mlp.2.weight", (int64_t)Hh * Hh});
    v.push_back({p + "coord_mlp.2.bias", Hh});
    v.push_back({p + "coord_mlp.4.weight", Hh});
  }
  return v;
}

// Host-side packer: appends 16-byte aligned segments to one blob and remembers offsets.
struct Packer {
  std::vector<float> blob;
  size_t add(const std::vector<float>& seg) {
    while (blob.size() % 4) blob.push_back(0.f);
    size_t off = blob.size();
    blob.insert(blob.end(), seg.begin(), seg.end());
    return off;
  }
};

// (out,in) row-major sub-block [0:out) x [c0:c0+k) -> k-major [k][out]
std::vector<float> transpose_block(const std::vector<float>& W, int out, int in_stride, int c0, int k) {
  std::vector<float> t((size_t)k * out);
  for (int o = 0; o < out; ++o)
    for (int i = 0; i < k; ++i) t[(size_t)i * out + o] = W[(size_t)o * in_stride + c0 + i];
  return t;
}
std::vector<float> column(const std::vector<float>& W, int out, int in_stride, int c) {
  std::vector<float> t(out);
  for (int o = 0; o < out; ++o) t[o] = W[(size_t)o * in_stride + c];
  return t;
}

template <typename T>
dl_status dev_alloc(Workspace& ws, T** p, size_t count) {
  void* q = nullptr;
  CK(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
  ws.allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return DL_OK;
}

void free_workspace(Workspace& ws) {
  for (void* p : ws.allocs) cudaFree(p);
  ws = Workspace();
}

Geom make_geom(const dl_engine* e, int B, int N);

dl_status ensure_workspace(dl_engine* e, int B, int N) {
  Workspace& ws = e->ws;
  if (ws.B == B && ws.N == N) return DL_OK;
  free_workspace(ws);
  const size_t n = (size_t)B * N;
  const int xd = 3 + e->cfg.in_node_nf;
  dl_status s;
#define WSA(field, cnt) if ((s = dev_alloc(ws, &ws.field, (cnt))) != DL_OK) return s
  WSA(nm, n); WSA(x0, n * 3); WSA(xa, n * 3); WSA(xb, n * 3); WSA(h, n * H); WSA(ABg, n * 2 * H); WSA(ABc, n * 2 * H);
  WSA(agg, n * H); WSA(z, n * xd); WSA(eps, n * xd); WSA(eps_hat, n * xd); WSA(cls, n); WSA(x04, n); WSA(xa4, n); WSA(xb4, n); WSA(ABgmax, n * 2); WSA(ABcmax, n * 2);
  WSA(rowidx, n); WSA(colidx, n); WSA(xrowidx, n); WSA(nr, B); WSA(nc, B); WSA(nxr, B); WSA(n_items, 1);
  WSA(xmols, B); WSA(n_xmols, 1); WSA(items, n); WSA(xitems, n); WSA(n_xitems, 1); WSA(tile_ctr, 64);
  if (e->use_tc && e->cfg.graph_type != 0) { WSA(nbr, n * N); WSA(recs, n * CUT_REC); WSA(xrecs, n * CUT_REC); WSA(n_recs, 2); }
#undef WSA
  ws.B = B; ws.N = N;
  ws.v3 = false;
  if (e->use_tc && e->allow_v3 && tc3::supports(make_geom(e, B, N))) {
    if (tc3::make_panel_map(&ws.tm_abg, ws.ABg, B, N) != DL_OK || tc3::make_panel_map(&ws.tm_abc, ws.ABc, B, N) != DL_OK) {
      set_err("cuTensorMapEncodeTiled failed for the projection buffers"); return DL_ERR_CUDA;
    }
    dl_status s2;
    for (int k = 0; k < 2; ++k)                              // at most one tile per live row
      if ((s2 = dev_alloc(ws, &ws.ts[k], n * tc3::TS_BYTES)) != DL_OK || (s2 = dev_alloc(ws, &ws.tij[k], n * tc::TN)) != DL_OK ||
          (s2 = dev_alloc(ws, &ws.td[k], n * tc::TN)) != DL_OK || (s2 = dev_alloc(ws, &ws.td0[k], n * tc::TN)) != DL_OK ||
          (s2 = dev_alloc(ws, &ws.tdmax[k], n)) != DL_OK || (s2 = dev_alloc(ws, &ws.td0max[k], n)) != DL_OK)
        return s2;
    if ((s2 = dev_alloc(ws, &ws.tcd, n * 3 * tc::TN)) != DL_OK) return s2;
    if ((s2 = dev_alloc(ws, &ws.cta_begin[0], (size_t)e->num_sms + 1)) != DL_OK || (s2 = dev_alloc(ws, &ws.cta_begin[1], (size_t)e->num_sms + 1)) != DL_OK) return s2;
    ws.v3 = true;
  }
  return DL_OK;
}

Plan make_plan(const Workspace& ws) {
  Plan p;
  p.rowidx = ws.rowidx; p.colidx = ws.colidx; p.xrowidx = ws.xrowidx; p.nr = ws.nr; p.nc = ws.nc; p.nxr = ws.nxr;
  p.items = ws.items; p.n_items = ws.n_items; p.xmols = ws.xmols; p.n_xmols = ws.n_xmols;
  p.xitems = ws.xitems; p.n_xitems = ws.n_xitems;
  return p;
}

Geom make_geom(const dl_engine* e, int B, int N) {
  Geom g;
  g.B = B; g.N = N; g.F = e->cfg.in_node_nf; g.C = e->cfg.context_node_nf; g.D = e->D;
  g.graph_type = e->cfg.graph_type; g.norm_constant = e->cfg.norm_constant;
  g.normalization_factor = e->cfg.normalization_factor;
  return g;
}

#define LAUNCH_CHECK()                                                                    \
  do {                                                                                    \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      set_err("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e));   \
      return DL_ERR_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

// Masks are constant over a whole sample_chain: build the work plan once.
dl_status build_plan(dl_engine* e, int B, int N, const int8_t* node_mask, const float* linker_mask,
                     const int8_t* edge_mask, cudaStream_t st) {
  Workspace& ws = e->ws;
  CK(cudaMemsetAsync(ws.agg, 0, (size_t)B * N * H * sizeof(float), st));  // dead rows aggregate to exactly 0
  k_plan_mol<<<B, 256, 2 * N * sizeof(int), st>>>(N, e->cfg.graph_type, edge_mask, node_mask, linker_mask, ws.rowidx,
                                                  ws.colidx, ws.xrowidx, ws.nr, ws.nc, ws.nxr);
  LAUNCH_CHECK();
  const int tile_edges = e->use_tc ? tc::TN : ET;
  const int max_rows = e->use_tc ? tc::MAXR : MAXR;
  // GCL items of the v3 kernel: rows padded to a multiple of four columns, at most MAXR3 rows per tile
  k_plan_items<<<1, 1, 0, st>>>(B, tile_edges, max_rows, ws.v3 ? 4 : 1, ws.v3 ? tc3::MAXR3 : max_rows, ws.nr, ws.nc, ws.nxr,
                                ws.items, ws.n_items, ws.xmols, ws.n_xmols, ws.xitems, ws.n_xitems, ws.v3 ? e->num_sms : 0,
                                ws.cta_begin[0], ws.cta_begin[1]);
  LAUNCH_CHECK();
  e->launches += 2;
  if (ws.v3) {
    tc3::k_tiles_static<<<B * N, tc::TN, 0, st>>>(N, ws.items, ws.n_items, ws.rowidx, ws.colidx, edge_mask, ws.ts[0], ws.tij[0]);
    LAUNCH_CHECK();
    tc3::k_tiles_static<<<B * N, tc::TN, 0, st>>>(N, ws.xitems, ws.n_xitems, ws.xrowidx, ws.colidx, edge_mask, ws.ts[1], ws.tij[1]);
    LAUNCH_CHECK();
    e->launches += 2;
  }
  return DL_OK;
}

tc3::TileTables make_tile_tables(const Workspace& ws, bool coord) {
  tc3::TileTables t;
  const int k = coord ? 1 : 0;
  t.ts = ws.ts[k]; t.td = ws.td[k]; t.td0 = ws.td0[k]; t.tdmax = ws.tdmax[k]; t.td0max = ws.td0max[k];
  t.tcd = coord ? ws.tcd : nullptr;
  t.items = coord ? ws.xitems : ws.items; t.n_items = coord ? ws.n_xitems : ws.n_items; t.rowidx = coord ? ws.xrowidx : ws.rowidx;
  t.cta_begin = ws.cta_begin[k];
  static const int stream_tasks = [] { const char* v = getenv("DL_V3_STREAM_TASKS"); return v ? atoi(v) : 1; }();
  t.stream_tasks = stream_tasks;
  return t;
}

struct FwdIO {
  // Dynamics.forward mode
  const float* xh = nullptr; const float* t = nullptr; int t_numel = 0; float* out = nullptr;
  // common
  const int8_t* node_mask = nullptr; const float* linker_mask = nullptr; const int8_t* edge_mask = nullptr;
  const float* context = nullptr; int* nan_flags = nullptr;
  // sampler mode
  bool sampler = false; bool inpaint = false; const float* xh0 = nullptr; const float* upd_linker_mask = nullptr;
  const float* fragment_mask = nullptr; const float* noise = nullptr; float* chain = nullptr;
  NoiseRng rng{};
  int T = 0; float norm0 = 1.f, norm1 = 1.f, bias1 = 0.f;
};

ProjW proj_of(const GclW& w) { return ProjW{w.W1a_t, w.W1b_t, w.b1}; }
ProjW proj_of(const EqW& w) { return ProjW{w.W1a_t, w.W1b_t, w.b1}; }

dl_status launch_edge(dl_engine* e, const Geom& gm, const EdgeArgs& ea, bool coord, const void* w2_tc,
                      cudaStream_t st, const void* w2_v3 = nullptr) {
  if (e->use_tc && e->ws.v3 && w2_v3 != nullptr) {
    tc3::launch_edge_v3(gm, ea, coord, w2_v3, coord ? e->ws.tm_abc : e->ws.tm_abg, make_tile_tables(e->ws, coord), e->num_sms, st);
  } else if (e->use_tc) {
    dl_status s = tc::launch_edge_tc(gm, ea, coord, w2_tc, e->num_sms, st);
    if (s != DL_OK) return s;
  } else {
    if (coord) k_edge_simt<true><<<e->num_sms, 256, EDGE_SIMT_SMEM, st>>>(gm, ea);
    else k_edge_simt<false><<<e->num_sms, 256, EDGE_SIMT_SMEM, st>>>(gm, ea);
  }
  LAUNCH_CHECK();
  e->launches += 1;
  return DL_OK;
}

// One Dynamics.forward worth of launches (1 + L*(2S+2) + 1 kernels).
dl_status enqueue_forward(dl_engine* e, int B, int N, const FwdIO& io, cudaStream_t st) {
  Workspace& ws = e->ws;
  const Geom gm = make_geom(e, B, N);
  const int n = B * N;
  const int L = e->cfg.n_layers, S = e->cfg.inv_sublayers;
  const int node_blocks = (n + NODE_TM - 1) / NODE_TM;
  const size_t node_smem = 3 * NODE_TM * LDX * sizeof(float);

  PrepArgs pa{};
  pa.xh = io.sampler ? ws.z : io.xh;
  pa.node_mask = io.node_mask; pa.linker_mask = io.linker_mask;
  pa.t = io.t; pa.t_numel = io.t_numel; pa.context = io.context;
  pa.We_t = e->We_t; pa.be = e->be; pa.proj = proj_of(e->gcl[0]);
  pa.nm = ws.nm; pa.x0 = ws.x0; pa.x = ws.xa; pa.x04 = e->use_tc ? ws.x04 : nullptr; pa.x4 = e->use_tc ? ws.xa4 : nullptr; pa.cls = ws.cls; pa.h = ws.h;
  pa.AB = e->use_tc ? nullptr : ws.ABg; pa.ABmax = ws.ABgmax;
  pa.coef = io.sampler ? e->coef_dev : nullptr;
  pa.step_prep = io.sampler ? e->step_ctr : nullptr;
  pa.step_fin = io.sampler ? e->step_ctr + 1 : nullptr;
  TIMED("k_prep", st, (launch_chain(k_prep, dim3(node_blocks), dim3(256), 0, st, gm, pa)));
  LAUNCH_CHECK();
  e->launches += 1;
  if (e->use_tc) {
    // A | B projections of block 0 / gcl 0 from the embedded h, on the tensor cores
    const GclW& w0 = e->gcl[0];
    tcn::NodeTcArgs ta{};
    ta.h = ws.h; ta.agg = ws.h; ta.nm = ws.nm; ta.proj_only = 1;
    ta.w3 = reinterpret_cast<const __half*>(w0.W3_tc); ta.w4 = reinterpret_cast<const __half*>(w0.W4_tc);
    ta.b3 = w0.b3; ta.b4 = w0.b4; ta.w3_descale = 1.f; ta.w4_descale = 1.f;
    ta.n_proj = 1; ta.pw[0] = reinterpret_cast<const __half*>(w0.W1_tc); ta.pb1[0] = w0.b1_u;
    ta.p_descale[0] = w0.w1_descale; ta.AB[0] = ws.ABg; ta.ABmax[0] = ws.ABgmax;
    ta.tile_nodes = tcn::pick_tile_nodes(n, e->num_sms);
    TIMED("k_node_tc(proj only)", st, (tcn::launch_node(n, ta, st, nullptr)));
    LAUNCH_CHECK();
    e->launches += 1;
  }

  if (ws.nbr != nullptr) {
    // the cut-off graph of this call (a function of its input coordinates): neighbour lists + packed tiles
    CK(cudaMemsetAsync(ws.n_recs, 0, 2 * sizeof(int), st));
    k_nbr<<<B, 512, (size_t)N * CUT_SMEM_PER_NODE, st>>>(N, e->cfg.graph_type, ws.x04, ws.cls, ws.rowidx, ws.colidx,
                                                        ws.xrowidx, ws.nr, ws.nc, ws.nxr, ws.nbr, ws.recs, ws.xrecs,
                                                        ws.n_recs);
    LAUNCH_CHECK();
    e->launches += 1;
  }

  float* xin = ws.xa;
  float* xout = ws.xb;
  float4* xin4 = ws.xa4;
  float4* xout4 = ws.xb4;
  const Plan plan = make_plan(ws);
  const float ksc = e->use_tc ? 1.4426950408889634f : 1.0f;   // log2-domain first layer on the tcgen05 path
  e->last_edge_mask = io.edge_mask; e->last_linker_mask = io.linker_mask; e->last_B = B; e->last_N = N;
  for (int l = 0; l < L; ++l) {
    if (ws.v3) {
      // tile tables of this block (squared distances from the block's coordinates; block 0 also fills the input-distance
      // table: x == x0 there) + the x -> x_next copy that precedes the block's coordinate update
      tc3::TileDSet s0{ws.n_items, ws.tij[0], ws.td[0], ws.tdmax[0], ws.td0[0], ws.td0max[0], nullptr, nullptr};
      tc3::TileDSet s1{ws.n_xitems, ws.tij[1], ws.td[1], ws.tdmax[1], ws.td0[1], ws.td0max[1], ws.ts[1], ws.tcd};
      TIMED("k_tiles_d", st, (launch_chain(tc3::k_tiles_d, dim3(e->num_sms * 8, 2), dim3(tc::TN), 0, st, s0, s1, xin4, l == 0 ? 1 : 0, gm.norm_constant, n * 3, xin, xout, xin4, xout4)));
      LAUNCH_CHECK();
      e->launches += 1;
    }
    for (int s = 0; s < S; ++s) {
      const GclW& w = e->gcl[l * S + s];
      EdgeArgs ea{};
      ea.AB = ws.ABg; ea.ABmax = ws.ABgmax; ea.w2_descale = w.w2_descale; ea.wdmax = w.wdmax * ksc; ea.w0max = w.w0max * ksc;
      ea.x = xin; ea.x0 = ws.x0; ea.x4 = xin4; ea.x04 = ws.x04; ea.x4_out = nullptr;
      ea.edge_mask = io.edge_mask; ea.cls = ws.cls; ea.nm = ws.nm;
      ea.linker_mask = io.linker_mask; ea.W2_t = w.W2_t; ea.b2 = w.b2; ea.wd = e->use_tc ? w.wd_u : w.wd; ea.w0 = e->use_tc ? w.w0_u : w.w0; ea.w5 = nullptr;
      ea.plan = plan; ea.agg = ws.agg; ea.x_out = nullptr; ea.nbr = ws.nbr; ea.recs = ws.recs; ea.n_recs = ws.n_recs;
      g_times.begin(st, "edge GCL");
      dl_status st2 = launch_edge(e, gm, ea, false, w.W2_tc, st, w.W2_v3);
      g_times.end(st);
      if (st2 != DL_OK) return st2;

      const bool last_sub = s + 1 >= S;
      if (e->use_tc) {
        tcn::NodeTcArgs ta{};
        ta.h = ws.h; ta.agg = ws.agg; ta.nm = ws.nm;
        ta.w3 = reinterpret_cast<const __half*>(w.W3_tc); ta.w4 = reinterpret_cast<const __half*>(w.W4_tc);
        ta.b3 = w.b3; ta.b4 = w.b4; ta.w3_descale = w.w3_descale; ta.w4_descale = w.w4_descale;
        if (!last_sub) {
          const GclW& nx = e->gcl[l * S + s + 1];
          ta.n_proj = 1; ta.pw[0] = reinterpret_cast<const __half*>(nx.W1_tc); ta.pb1[0] = nx.b1_u;
          ta.p_descale[0] = nx.w1_descale; ta.AB[0] = ws.ABg; ta.ABmax[0] = ws.ABgmax;
        } else {
          const EqW& q = e->eq[l];
          ta.n_proj = 1; ta.pw[0] = reinterpret_cast<const __half*>(q.W1_tc); ta.pb1[0] = q.b1_u;
          ta.p_descale[0] = q.w1_descale; ta.AB[0] = ws.ABc; ta.ABmax[0] = ws.ABcmax;
          if (l + 1 < L) {
            const GclW& nx = e->gcl[(l + 1) * S];
            ta.n_proj = 2; ta.pw[1] = reinterpret_cast<const __half*>(nx.W1_tc); ta.pb1[1] = nx.b1_u;
            ta.p_descale[1] = nx.w1_descale; ta.AB[1] = ws.ABg; ta.ABmax[1] = ws.ABgmax;
          }
        }
        static int node_prof_left = getenv("DL_PROFILE_NODE") ? 3 : 0;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (node_prof_left > 0) cudaStreamIsCapturing(st, &cap);
        if (node_prof_left > 0 && cap == cudaStreamCaptureStatusNone) { --node_prof_left; tcn::profile_node(n, ta, st); }
        else {
          ta.tile_nodes = tcn::pick_tile_nodes(n, e->num_sms);
          TIMED(ta.n_proj == 2 ? "k_node_tc(2 proj)" : "k_node_tc(1 proj)", st,
                (tcn::launch_node(n, ta, st, nullptr)));
        }
      } else {
        NodeArgs na{};
        na.h = ws.h; na.agg = ws.agg; na.nm = ws.nm; na.W3_t = w.W3_t; na.b3 = w.b3; na.W4_t = w.W4_t; na.b4 = w.b4;
        if (!last_sub) {
          na.proj1 = proj_of(e->gcl[l * S + s + 1]); na.AB1 = ws.ABg; na.ABmax1 = ws.ABgmax; na.AB2 = nullptr;
        } else {
          na.proj1 = proj_of(e->eq[l]); na.AB1 = ws.ABc; na.ABmax1 = ws.ABcmax;
          if (l + 1 < L) { na.proj2 = proj_of(e->gcl[(l + 1) * S]); na.AB2 = ws.ABg; na.ABmax2 = ws.ABgmax; }
          else na.AB2 = nullptr;
        }
        k_node<ACT_SILU><<<node_blocks, 256, node_smem, st>>>(n, na);
      }
      LAUNCH_CHECK();
      e->launches += 1;
    }
    if (!ws.v3) {
      k_copy_x<<<(n * 3 + 255) / 256, 256, 0, st>>>(n * 3, xin, xout, e->use_tc ? xin4 : nullptr, xout4);
      LAUNCH_CHECK();
      e->launches += 1;
    }
    const EqW& w = e->eq[l];
    EdgeArgs ea{};
    ea.AB = ws.ABc; ea.ABmax = ws.ABcmax; ea.w2_descale = w.w2_descale; ea.wdmax = w.wdmax * ksc; ea.w0max = w.w0max * ksc;
    ea.x = xin; ea.x0 = ws.x0; ea.x4 = xin4; ea.x04 = ws.x04; ea.x4_out = xout4;
    ea.edge_mask = io.edge_mask; ea.cls = ws.cls; ea.nm = ws.nm;
    ea.linker_mask = io.linker_mask; ea.W2_t = w.W2_t; ea.b2 = w.b2; ea.wd = e->use_tc ? w.wd_u : w.wd; ea.w0 = e->use_tc ? w.w0_u : w.w0; ea.w5 = w.w5;
    ea.plan = plan; ea.agg = nullptr; ea.x_out = xout; ea.nbr = ws.nbr; ea.recs = ws.xrecs; ea.n_recs = ws.n_recs ? ws.n_recs + 1 : nullptr;
    g_times.begin(st, "edge COORD");
    dl_status st2 = launch_edge(e, gm, ea, true, w.W2_tc, st, e->allow_v3_coord ? w.W2_v3 : nullptr);
    g_times.end(st);
    if (st2 != DL_OK) return st2;
    std::swap(xin, xout);
    std::swap(xin4, xout4);
  }

  FinishArgs fa{};
  fa.h = ws.h; fa.x = xin; fa.x0 = ws.x0; fa.nm = ws.nm; fa.Wo = e->Wo; fa.bo = e->bo;
  fa.nan_flags = io.nan_flags;
  const bool fused_update = io.sampler && !io.inpaint;
  fa.out = fused_update ? nullptr : (io.sampler ? ws.eps : io.out);
  if (fused_update) {
    fa.z = ws.z; fa.fragment_mask = io.fragment_mask; fa.linker_mask = io.linker_mask; fa.noise = io.noise; fa.rng = io.rng;
    fa.coef = e->coef_dev; fa.step_fin = e->step_ctr + 1; fa.step_prep = e->step_ctr; fa.T = io.T;
    fa.norm0 = io.norm0; fa.norm1 = io.norm1; fa.bias1 = io.bias1; fa.chain = io.chain;
  } else if (io.sampler) {
    fa.tag_step = e->step_ctr + 1;
  }
  TIMED("k_finish", st, (launch_chain(k_finish, dim3((n + 15) / 16), dim3(256), 0, st, gm, fa)));
  LAUNCH_CHECK();
  e->launches += 1;
  if (e->cfg.centering || io.inpaint) {
    // per-molecule stage of inpainting models: centring of the velocity (egnn.py:444-445) and, in the sampler,
    // the whole reverse step incl. the centre-of-mass projection (edm.py:549-612)
    InpaintArgs ia{};
    ia.mode = io.inpaint ? 1 : 0;
    ia.eps = io.inpaint ? ws.eps : io.out; ia.nm = ws.nm; ia.z = ws.z; ia.xh0 = io.xh0;
    ia.fragment_mask = io.fragment_mask; ia.linker_mask = io.upd_linker_mask; ia.noise = io.noise; ia.coef = e->coef_dev;
    ia.step_prep = e->step_ctr; ia.step_fin = e->step_ctr + 1; ia.T = io.T;
    ia.norm0 = io.norm0; ia.norm1 = io.norm1; ia.bias1 = io.bias1; ia.chain = io.chain;
    k_inpaint<<<B, 256, 0, st>>>(gm, ia);
    LAUNCH_CHECK();
    e->launches += 1;
  }
  return DL_OK;
}

dl_status check_shapes(const dl_engine* e, int B, int N) {
  if (!e || !e->finalized) { set_err("engine not finalized (dl_finalize_weights)"); return DL_ERR_INVALID; }
  if (B <= 0 || N <= 0) { set_err("B and N must be positive (got %d, %d)", B, N); return DL_ERR_INVALID; }
  if ((int64_t)B * N * N > (int64_t)1 << 40) { set_err("B*N*N too large"); return DL_ERR_INVALID; }
  if (e->use_tc && e->cfg.graph_type != 0 && N > 4000) {
    set_err("cut-off graphs: N = %d exceeds the neighbour-list kernel's shared-memory staging (N <= 4000)", N);
    return DL_ERR_INVALID;
  }
  return DL_OK;
}

dl_status stage_reserve(dl_engine* e, size_t bytes) {
  if (e->stage.cap >= bytes) return DL_OK;
  if (e->stage.buf) cudaFree(e->stage.buf);
  e->stage.buf = nullptr; e->stage.cap = 0;
  CK(cudaMalloc((void**)&e->stage.buf, bytes));
  e->stage.cap = bytes;
  return DL_OK;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

const char* dl_version(void) { return "difflinker_b200 0.1 (sm_100a)"; }
const char* dl_last_error(void) { return g_err; }

dl_status dl_create(const dl_config* cfg, dl_engine** out) {
  if (!cfg || !out) { set_err("null argument"); return DL_ERR_INVALID; }
  if (cfg->hidden_nf != H) { set_err("hidden_nf must be %d (got %d)", H, cfg->hidden_nf); return DL_ERR_UNSUPPORTED; }
  if (cfg->n_dims != 3) { set_err("n_dims must be 3"); return DL_ERR_UNSUPPORTED; }
  const int D = cfg->in_node_nf + cfg->context_node_nf + (cfg->condition_time ? 1 : 0);
  if (D > MAX_DIN || cfg->in_node_nf < 1 || 3 + cfg->in_node_nf > MAX_XHD) {
    set_err("unsupported feature widths F=%d C=%d", cfg->in_node_nf, cfg->context_node_nf);
    return DL_ERR_UNSUPPORTED;
  }
  if (cfg->n_layers < 1 || cfg->inv_sublayers < 1) { set_err("n_layers/inv_sublayers must be >= 1"); return DL_ERR_INVALID; }
  if (cfg->graph_type < 0 || cfg->graph_type > 3) { set_err("bad graph_type"); return DL_ERR_INVALID; }
  if (cfg->graph_type != DL_GRAPH_FC && cfg->context_node_nf < 2) {
    set_err("pocket graphs need fragment_only/pocket_only context columns"); return DL_ERR_INVALID;
  }
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) { set_err("device %d not available (%d devices)", cfg->device, ndev); return DL_ERR_INVALID; }
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) {
    set_err("difflinker_b200 is built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
    return DL_ERR_UNSUPPORTED;
  }
  dl_engine* e = new dl_engine();
  e->cfg = *cfg;
  e->D = D;
  e->num_sms = prop.multiProcessorCount;
  e->max_threads_per_sm = prop.maxThreadsPerMultiProcessor;
  e->use_tc = tc::AVAILABLE && cfg->edge_impl != DL_EDGE_SIMT;
  CK(cudaStreamCreateWithFlags(&e->loop_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming));
  CK(cudaEventCreate(&e->ev_t0));
  CK(cudaEventCreate(&e->ev_t1));
  CK(cudaMalloc((void**)&e->step_ctr, 2 * sizeof(int)));
  CK(cudaFuncSetAttribute(k_node<ACT_SILU>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * NODE_TM * LDX * sizeof(float)));
  CK(cudaFuncSetAttribute(k_edge_simt<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EDGE_SIMT_SMEM));
  CK(cudaFuncSetAttribute(k_edge_simt<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EDGE_SIMT_SMEM));
  CK(cudaFuncSetAttribute(k_nbr, cudaFuncAttributeMaxDynamicSharedMemorySize, 4000 * CUT_SMEM_PER_NODE));
  if (getenv("DL_TIME_KERNELS")) g_times.on = true;
  if (const char* v = getenv("DL_EDGE_V3")) e->allow_v3 = atoi(v) != 0;
  if (const char* v = getenv("DL_WAIT_MODE")) { const int m = atoi(v); cudaMemcpyToSymbol(tc::c_wait_mode, &m, sizeof(int)); }
  if (const char* v = getenv("DL_CHAIN_OVERLAP")) chain_overlap_enabled() = atoi(v) != 0;   // 0: plain stream order between kernels
  if (const char* v = getenv("DL_EDGE_V3_COORD")) e->allow_v3_coord = atoi(v) != 0;
  dl_status s = tc::configure();
  if (s == DL_OK) s = tcn::configure_node();
  if (s == DL_OK) s = tc3::configure3();
  if (s != DL_OK) { set_err("cudaFuncSetAttribute failed for the tcgen05 kernels"); delete e; return s; }
  *out = e;
  return DL_OK;
}

dl_status dl_destroy(dl_engine* e) {
  if (!e) return DL_OK;
  g_times.report();
  g_times.acc.clear();
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  free_workspace(e->ws);
  if (e->wblob) cudaFree(e->wblob);
  if (e->wblob_tc) cudaFree(e->wblob_tc);
  if (e->coef_dev) cudaFree(e->coef_dev);
  if (e->step_ctr) cudaFree(e->step_ctr);
  if (e->stage.buf) cudaFree(e->stage.buf);
  if (e->loop_stream) cudaStreamDestroy(e->loop_stream);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  if (e->ev_t0) cudaEventDestroy(e->ev_t0);
  if (e->ev_t1) cudaEventDestroy(e->ev_t1);
  delete e;
  return DL_OK;
}

int64_t dl_expected_param_count(const dl_engine* e) {
  if (!e) return 0;
  int64_t n = 0;
  for (auto& p : expected_params(e->cfg)) n += p.numel;
  return n;
}

dl_status dl_set_weight(dl_engine* e, const char* name, const float* data, int64_t numel) {
  if (!e || !name || !data) { set_err("null argument"); return DL_ERR_INVALID; }
  for (auto& p : expected_params(e->cfg)) {
    if (p.name == name) {
      if (p.numel != numel) {
        set_err("weight %s: expected %lld elements, got %lld", name, (long long)p.numel, (long long)numel);
        return DL_ERR_WEIGHTS;
      }
      e->raw[p.name].assign(data, data + numel);
      e->finalized = false;
      return DL_OK;
    }
  }
  set_err("unexpected weight name %s", name);
  return DL_ERR_WEIGHTS;
}

dl_status dl_finalize_weights(dl_engine* e) {
  if (!e) { set_err("null engine"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  for (auto& p : expected_params(e->cfg))
    if (!e->raw.count(p.name)) { set_err("missing weight %s", p.name.c_str()); return DL_ERR_WEIGHTS; }
  const int L = e->cfg.n_layers, S = e->cfg.inv_sublayers, D = e->D;
  const int IN1 = 2 * H + 2;
  Packer pk;
  std::vector<__half> tcblob;
  struct GOff { size_t W1a, W1b, b1, wd, w0, W2, b2, W3, b3, W4, b4, w5, tc, tc1, tc3, tc4, b1u, wdu, w0u, v3; float descale, wdmax, w0max, d1, d3, d4; };
  // log2-domain copies for the tcgen05 path (kernels_tc.cuh pack_w2): everything that feeds the first Linear of an edge MLP
  auto scaled = [](const std::vector<float>& v) { std::vector<float> o(v.size()); for (size_t i = 0; i < v.size(); ++i) o[i] = (float)((double)v[i] * tc::NEG_LOG2E); return o; };
  auto absmax = [](const std::vector<float>& v) { float m = 0.f; for (float x : v) m = std::max(m, std::fabs(x)); return m; };
  std::vector<GOff> goff(L * S), eoff(L);
  auto R = [&](const std::string& k) -> const std::vector<float>& { return e->raw[k]; };
  size_t oWe = pk.add(transpose_block(R("dynamics.embedding.weight"), H, D, 0, D));
  size_t obe = pk.add(R("dynamics.embedding.bias"));
  size_t oWo = pk.add(R("dynamics.embedding_out.weight"));
  size_t obo = pk.add(R("dynamics.embedding_out.bias"));
  char buf[160];
  for (int l = 0; l < L; ++l) {
    for (int s = 0; s < S; ++s) {
      snprintf(buf, sizeof(buf), "dynamics.e_block_%d.gcl_%d.", l, s);
      std::string p(buf);
      GOff& o = goff[l * S + s];
      const auto& W1 = R(p + "edge_mlp.0.weight");
      o.W1a = pk.add(transpose_block(W1, H, IN1, 0, H));
      o.W1b = pk.add(transpose_block(W1, H, IN1, H, H));
      o.b1 = pk.add(R(p + "edge_mlp.0.bias"));
      o.wd = pk.add(column(W1, H, IN1, 2 * H));
      o.w0 = pk.add(column(W1, H, IN1, 2 * H + 1));
      o.W2 = pk.add(transpose_block(R(p + "edge_mlp.2.weight"), H, H, 0, H));
      o.b2 = pk.add(R(p + "edge_mlp.2.bias"));
      o.W3 = pk.add(transpose_block(R(p + "node_mlp.0.weight"), H, 2 * H, 0, 2 * H));
      o.b3 = pk.add(R(p + "node_mlp.0.bias"));
      o.W4 = pk.add(transpose_block(R(p + "node_mlp.2.weight"), H, H, 0, H));
      o.b4 = pk.add(R(p + "node_mlp.2.bias"));
      o.tc = tc::pack_w2(R(p + "edge_mlp.2.weight"), tcblob, &o.descale);
      { float d3v = 0.f; o.v3 = tc3::pack_w2_v3(R(p + "edge_mlp.2.weight"), tcblob, &d3v); }   // same scale rule as pack_w2
      o.tc1 = tcn::pack_blocks(scaled(W1), IN1, 2, tcblob, &o.d1);
      o.b1u = pk.add(scaled(R(p + "edge_mlp.0.bias")));
      o.wdu = pk.add(scaled(column(W1, H, IN1, 2 * H)));
      o.w0u = pk.add(scaled(column(W1, H, IN1, 2 * H + 1)));
      o.tc3 = tcn::pack_blocks(R(p + "node_mlp.0.weight"), 2 * H, 2, tcblob, &o.d3);
      o.tc4 = tcn::pack_blocks(R(p + "node_mlp.2.weight"), H, 1, tcblob, &o.d4);
      o.wdmax = absmax(column(W1, H, IN1, 2 * H)); o.w0max = absmax(column(W1, H, IN1, 2 * H + 1));
    }
    snprintf(buf, sizeof(buf), "dynamics.e_block_%d.gcl_equiv.", l);
    std::string p(buf);
    GOff& o = eoff[l];
    const auto& W1 = R(p + "coord_mlp.0.weight");
    o.W1a = pk.add(transpose_block(W1, H, IN1, 0, H));
    o.W1b = pk.add(transpose_block(W1, H, IN1, H, H));
    o.b1 = pk.add(R(p + "coord_mlp.0.bias"));
    o.wd = pk.add(column(W1, H, IN1, 2 * H));
    o.w0 = pk.add(column(W1, H, IN1, 2 * H + 1));
    o.W2 = pk.add(transpose_block(R(p + "coord_mlp.2.weight"), H, H, 0, H));
    o.b2 = pk.add(R(p + "coord_mlp.2.bias"));
    o.w5 = pk.add(R(p + "coord_mlp.4.weight"));
    o.tc = tc::pack_w2(R(p + "coord_mlp.2.weight"), tcblob, &o.descale);
    { float d3v = 0.f; o.v3 = tc3::pack_w2_v3(R(p + "coord_mlp.2.weight"), tcblob, &d3v); }
    o.tc1 = tcn::pack_blocks(scaled(W1), IN1, 2, tcblob, &o.d1);
    o.b1u = pk.add(scaled(R(p + "coord_mlp.0.bias")));
    o.wdu = pk.add(scaled(column(W1, H, IN1, 2 * H)));
    o.w0u = pk.add(scaled(column(W1, H, IN1, 2 * H + 1)));
    o.wdmax = absmax(column(W1, H, IN1, 2 * H)); o.w0max = absmax(column(W1, H, IN1, 2 * H + 1));
  }
  if (e->wblob) { cudaFree(e->wblob); e->wblob = nullptr; }
  if (e->wblob_tc) { cudaFree(e->wblob_tc); e->wblob_tc = nullptr; }
  CK(cudaMalloc((void**)&e->wblob, pk.blob.size() * sizeof(float)));
  CK(cudaMemcpy(e->wblob, pk.blob.data(), pk.blob.size() * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMalloc(&e->wblob_tc, std::max<size_t>(tcblob.size(), 1) * sizeof(__half)));
  CK(cudaMemcpy(e->wblob_tc, tcblob.data(), tcblob.size() * sizeof(__half), cudaMemcpyHostToDevice));
  const float* base = e->wblob;
  const __half* tbase = reinterpret_cast<const __half*>(e->wblob_tc);
  e->We_t = base + oWe; e->be = base + obe; e->Wo = base + oWo; e->bo = base + obo;
  e->gcl.assign(L * S, GclW{});
  e->eq.assign(L, EqW{});
  for (int i = 0; i < L * S; ++i) {
    const GOff& o = goff[i];
    e->gcl[i] = GclW{base + o.W1a, base + o.W1b, base + o.b1, base + o.wd, base + o.w0, base + o.W2, base + o.b2,
                     base + o.W3,  base + o.b3,  base + o.W4, base + o.b4, tbase + o.tc, o.descale, o.wdmax, o.w0max,
                     tbase + o.tc1, tbase + o.tc3, tbase + o.tc4, o.d1, o.d3, o.d4,
                     base + o.b1u, base + o.wdu, base + o.w0u, tbase + o.v3};
  }
  for (int l = 0; l < L; ++l) {
    const GOff& o = eoff[l];
    e->eq[l] = EqW{base + o.W1a, base + o.W1b, base + o.b1, base + o.wd, base + o.w0,
                   base + o.W2,  base + o.b2,  base + o.w5, tbase + o.tc, o.descale, o.wdmax, o.w0max, tbase + o.tc1, o.d1,
                   base + o.b1u, base + o.wdu, base + o.w0u, tbase + o.v3};
  }
  e->finalized = true;
  return DL_OK;
}

dl_status dl_dynamics_forward(dl_engine* e, int32_t B, int32_t N, const float* t, int32_t t_numel, const float* xh,
                              const int8_t* node_mask, const float* linker_mask, const int8_t* edge_mask,
                              const float* context, float* out, int32_t* nan_flags, void* stream) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (!xh || !node_mask || !out) { set_err("xh/node_mask/out must not be null"); return DL_ERR_INVALID; }
  if (e->cfg.condition_time && (!t || (t_numel != 1 && t_numel != B))) { set_err("t must hold 1 or B values"); return DL_ERR_INVALID; }
  if (e->cfg.context_node_nf > 0 && !context) { set_err("context required (context_node_nf=%d)", e->cfg.context_node_nf); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if ((s = ensure_workspace(e, B, N)) != DL_OK) return s;
  CK(cudaEventRecord(e->ev_t0, st));
  if (nan_flags) CK(cudaMemsetAsync(nan_flags, 0, B * sizeof(int32_t), st));
  if ((s = build_plan(e, B, N, node_mask, linker_mask, edge_mask, st)) != DL_OK) return s;
  FwdIO io;
  io.xh = xh; io.t = t; io.t_numel = t_numel; io.out = out; io.node_mask = node_mask; io.linker_mask = linker_mask;
  io.edge_mask = edge_mask; io.context = context; io.nan_flags = nan_flags;
  if ((s = enqueue_forward(e, B, N, io, st)) != DL_OK) return s;
  CK(cudaEventRecord(e->ev_t1, st));
  g_times.collect(st);
  return DL_OK;
}

dl_status dl_dynamics_forward_host(dl_engine* e, int32_t B, int32_t N, const float* t, int32_t t_numel,
                                   const float* xh, const int8_t* node_mask, const float* linker_mask,
                                   const int8_t* edge_mask, const float* context, float* out, int32_t* nan_flags) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  CK(cudaSetDevice(e->cfg.device));
  const size_t n = (size_t)B * N;
  const int xd = 3 + e->cfg.in_node_nf, C = e->cfg.context_node_nf;
  const size_t o_t = 0, o_xh = o_t + align256(sizeof(float) * std::max(t_numel, 1)), o_nm = o_xh + align256(n * xd * 4),
               o_lm = o_nm + align256(n), o_em = o_lm + align256(n * 4), o_ctx = o_em + align256(n * N),
               o_out = o_ctx + align256(n * std::max(C, 1) * 4), o_fl = o_out + align256(n * xd * 4),
               total = o_fl + align256(B * 4);
  if ((s = stage_reserve(e, total)) != DL_OK) return s;
  char* d = e->stage.buf;
  cudaStream_t st = e->loop_stream;
  if (t) CK(cudaMemcpyAsync(d + o_t, t, sizeof(float) * t_numel, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_xh, xh, n * xd * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_nm, node_mask, n, cudaMemcpyHostToDevice, st));
  if (linker_mask) CK(cudaMemcpyAsync(d + o_lm, linker_mask, n * 4, cudaMemcpyHostToDevice, st));
  if (edge_mask && e->cfg.graph_type == DL_GRAPH_FC) CK(cudaMemcpyAsync(d + o_em, edge_mask, n * N, cudaMemcpyHostToDevice, st));
  if (context) CK(cudaMemcpyAsync(d + o_ctx, context, n * C * 4, cudaMemcpyHostToDevice, st));
  s = dl_dynamics_forward(e, B, N, t ? (const float*)(d + o_t) : nullptr, t_numel, (const float*)(d + o_xh),
                          (const int8_t*)(d + o_nm), linker_mask ? (const float*)(d + o_lm) : nullptr,
                          (edge_mask && e->cfg.graph_type == DL_GRAPH_FC) ? (const int8_t*)(d + o_em) : nullptr,
                          context ? (const float*)(d + o_ctx) : nullptr, (float*)(d + o_out), (int32_t*)(d + o_fl), st);
  if (s != DL_OK) return s;
  std::vector<int32_t> flags(B);
  CK(cudaMemcpyAsync(out, d + o_out, n * xd * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(flags.data(), d + o_fl, B * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  bool any = false;
  for (int i = 0; i < B; ++i) { any |= flags[i] != 0; if (nan_flags) nan_flags[i] = flags[i]; }
  return any ? DL_NAN_DETECTED : DL_OK;
}

// torch's launch geometry for randn(numel) on this device (see NoiseRng)
static void randn_geometry(const dl_engine* e, long long numel, int* S, unsigned long long* consumed) {
  long long grid = (numel + 255) / 256;
  grid = std::min<long long>(grid, (long long)e->num_sms * (e->max_threads_per_sm / 256));
  grid = std::max<long long>(grid, 1);
  *S = (int)(256 * grid);
  *consumed = (unsigned long long)(((numel - 1) / (4LL * *S) + 1) * 4);
}
static NoiseRng make_rng(const dl_engine* e, int B, int N, uint64_t seed, uint64_t offset) {
  NoiseRng q{};
  const int F = e->cfg.in_node_nf;
  unsigned long long cx = 0, ch = 0;
  const int B_full = e->slice_B_full > 0 ? e->slice_B_full : B;   // geometry of the FULL batch's randn calls
  randn_geometry(e, (long long)B_full * N * 3, &q.Sx, &cx);
  randn_geometry(e, (long long)B_full * N * F, &q.Sh, &ch);
  q.seed = seed; q.offset = offset; q.cx = cx; q.per_draw = cx + ch; q.F = F; q.on = 1;
  q.g0 = e->slice_B_full > 0 ? e->slice_b0 * N : 0;
  return q;
}

static dl_status sample_chain_impl(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                                   const float* xh, const int8_t* node_mask, const float* fragment_mask,
                                   const float* linker_mask, const int8_t* edge_mask, const float* context,
                                   const float* noise, const NoiseRng* rng, const dl_step_coef* coef, const float* norm,
                                   float* chain, int32_t* nan_flags, void* stream);

dl_status dl_sample_chain(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                          const float* xh, const int8_t* node_mask, const float* fragment_mask,
                          const float* linker_mask, const int8_t* edge_mask, const float* context,
                          const float* noise, const dl_step_coef* coef, const float* norm, float* chain,
                          int32_t* nan_flags, void* stream) {
  if (!noise) { set_err("null argument (noise): use dl_sample_chain_rng to draw on the device"); return DL_ERR_INVALID; }
  return sample_chain_impl(e, sampler, B, N, T, keep_frames, xh, node_mask, fragment_mask, linker_mask, edge_mask, context, noise,
                           nullptr, coef, norm, chain, nan_flags, stream);
}

dl_status dl_sample_chain_rng(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                              const float* xh, const int8_t* node_mask, const float* fragment_mask,
                              const float* linker_mask, const int8_t* edge_mask, const float* context, uint64_t seed,
                              uint64_t offset, uint64_t* offset_consumed, const dl_step_coef* coef, const float* norm,
                              float* chain, int32_t* nan_flags, void* stream) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (e->slice_B_full > 0 && e->slice_b0 + B > e->slice_B_full) { set_err("batch slice [%d, %d) exceeds the full batch %d", e->slice_b0, e->slice_b0 + B, e->slice_B_full); return DL_ERR_INVALID; }
  if (sampler != DL_SAMPLER_LINKER) { set_err("device-side noise is implemented for the linker sampler (the inpainting sampler takes prepared slabs)"); return DL_ERR_UNSUPPORTED; }
  if (offset % 4 != 0) { set_err("philox offset must be a multiple of 4 (torch.Generator.get_offset())"); return DL_ERR_INVALID; }
  const NoiseRng q = make_rng(e, B, N, seed, offset);
  if (offset_consumed) *offset_consumed = (uint64_t)(T + 2) * q.per_draw;
  return sample_chain_impl(e, sampler, B, N, T, keep_frames, xh, node_mask, fragment_mask, linker_mask, edge_mask, context, nullptr,
                           &q, coef, norm, chain, nan_flags, stream);
}

dl_status dl_diffusion_loss(dl_engine* e, int32_t B, int32_t N, const float* xh, const int8_t* node_mask,
                            const float* fragment_mask, const float* linker_mask, const int8_t* edge_mask,
                            const float* context, const float* coef, const float* eps, uint64_t seed, uint64_t offset,
                            uint64_t* offset_consumed, const float* norm, float* terms, int32_t* nan_flags, void* stream) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (e->cfg.centering) { set_err("dl_diffusion_loss: inpainting models (centering = 1) are not supported"); return DL_ERR_UNSUPPORTED; }
  if (!xh || !node_mask || !fragment_mask || !linker_mask || !coef || !norm || !terms) { set_err("null argument"); return DL_ERR_INVALID; }
  if (!e->cfg.condition_time) { set_err("dl_diffusion_loss needs a time-conditioned model (condition_time = 1)"); return DL_ERR_UNSUPPORTED; }
  if (e->cfg.context_node_nf > 0 && !context) { set_err("context required (context_node_nf=%d)", e->cfg.context_node_nf); return DL_ERR_INVALID; }
  if (!eps && offset % 4 != 0) { set_err("philox offset must be a multiple of 4 (torch.Generator.get_offset())"); return DL_ERR_INVALID; }
  if (!eps && e->slice_B_full > 0) { set_err("dl_diffusion_loss draws the whole batch: switch the noise slice off first"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if ((s = ensure_workspace(e, B, N)) != DL_OK) return s;
  Workspace& ws = e->ws;
  const int n = B * N, xd = 3 + e->cfg.in_node_nf;
  NoiseRng q{};
  if (!eps) q = make_rng(e, B, N, seed, offset);
  if (offset_consumed) *offset_consumed = eps ? 0 : (uint64_t)q.per_draw;
  CK(cudaEventRecord(e->ev_t0, st));
  if (nan_flags) CK(cudaMemsetAsync(nan_flags, 0, B * sizeof(int32_t), st));
  TIMED("k_qsample", st, (k_qsample<<<(n * xd + 255) / 256, 256, 0, st>>>(n, N, xd, xh, fragment_mask, linker_mask, eps, q, coef,
                                                                          ws.z, ws.eps)));
  LAUNCH_CHECK();
  e->launches += 1;
  if ((s = build_plan(e, B, N, node_mask, linker_mask, edge_mask, st)) != DL_OK) return s;
  FwdIO io;
  io.xh = ws.z; io.t = coef + DL_LOSS_T * B; io.t_numel = B; io.out = ws.eps_hat; io.node_mask = node_mask;
  io.linker_mask = linker_mask; io.edge_mask = edge_mask; io.context = context; io.nan_flags = nan_flags;
  if ((s = enqueue_forward(e, B, N, io, st)) != DL_OK) return s;
  LossArgs la{};
  la.N = N; la.F = e->cfg.in_node_nf; la.xh = xh; la.z = ws.z; la.eps = ws.eps; la.out = ws.eps_hat; la.lm = linker_mask;
  la.coef = coef; la.norm1 = norm[1]; la.bias1 = norm[2]; la.terms = terms;
  TIMED("k_diffusion_loss", st, (k_diffusion_loss<<<B, LOSS_THREADS, 0, st>>>(la)));
  LAUNCH_CHECK();
  e->launches += 1;
  CK(cudaEventRecord(e->ev_t1, st));
  g_times.collect(st);
  return DL_OK;
}

dl_status dl_set_noise_slice(dl_engine* e, int32_t B_full, int32_t b0) {
  if (!e) { set_err("null engine"); return DL_ERR_INVALID; }
  if (B_full < 0 || b0 < 0 || (B_full > 0 && b0 >= B_full)) { set_err("bad batch slice (%d of %d)", b0, B_full); return DL_ERR_INVALID; }
  e->slice_B_full = B_full; e->slice_b0 = B_full > 0 ? b0 : 0;
  return DL_OK;
}

dl_status dl_noise_fill(dl_engine* e, int32_t n_draws, int32_t B, int32_t N, uint64_t seed, uint64_t offset, float* out,
                        uint64_t* offset_consumed, void* stream) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (!out || n_draws < 1) { set_err("null argument"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  const NoiseRng q = make_rng(e, B, N, seed, offset);
  if (offset_consumed) *offset_consumed = (uint64_t)n_draws * q.per_draw;
  k_noise_fill<<<e->num_sms * 4, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(n_draws, B * N, 3 + e->cfg.in_node_nf, q, out);
  LAUNCH_CHECK();
  return DL_OK;
}

static dl_status sample_chain_impl(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                                   const float* xh, const int8_t* node_mask, const float* fragment_mask,
                                   const float* linker_mask, const int8_t* edge_mask, const float* context,
                                   const float* noise, const NoiseRng* rng, const dl_step_coef* coef, const float* norm,
                                   float* chain, int32_t* nan_flags, void* stream) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (sampler != DL_SAMPLER_LINKER && sampler != DL_SAMPLER_INPAINT) { set_err("unknown sampler %d", sampler); return DL_ERR_INVALID; }
  const bool inpaint = sampler == DL_SAMPLER_INPAINT;
  if (inpaint != (e->cfg.centering != 0)) { set_err("the inpainting sampler needs a model built with centering=1 (and vice versa)"); return DL_ERR_INVALID; }
  if (!xh || !node_mask || !fragment_mask || !linker_mask || (!noise && !rng) || !coef || !norm || !chain) {
    set_err("null argument"); return DL_ERR_INVALID;
  }
  if (T < 1 || keep_frames < 1 || keep_frames > T) { set_err("need 1 <= keep_frames <= T"); return DL_ERR_INVALID; }
  if (e->cfg.context_node_nf > 0 && !context) { set_err("context required"); return DL_ERR_INVALID; }
  static_assert(sizeof(dl_step_coef) == 32, "dl_step_coef layout");
  CK(cudaSetDevice(e->cfg.device));
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  cudaStream_t st = e->loop_stream;
  // DL_TIME_CHAIN=1: host-clock breakdown of one call to stderr (adds stream synchronisations: diagnostic only)
  static const bool time_chain = getenv("DL_TIME_CHAIN") != nullptr;
  auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
  const double tc0 = time_chain ? now_ms() : 0.0;
  double tc_plan = 0, tc_capture = 0, tc_inst = 0, tc_launch = 0;
  if ((s = ensure_workspace(e, B, N)) != DL_OK) return s;
  if (e->coef_cap < T + 1) {
    if (e->coef_dev) cudaFree(e->coef_dev);
    e->coef_dev = nullptr;
    CK(cudaMalloc((void**)&e->coef_dev, (size_t)(T + 1) * sizeof(dl_step_coef)));
    e->coef_cap = T + 1;
  }
  // order the private loop stream after the caller's stream (the legacy default stream cannot be captured)
  if (user != st) {
    CK(cudaEventRecord(e->ev_in, user));
    CK(cudaStreamWaitEvent(st, e->ev_in, 0));
  }
  CK(cudaMemcpyAsync(e->coef_dev, coef, (size_t)(T + 1) * sizeof(dl_step_coef), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(e->step_ctr, 0, 2 * sizeof(int), st));
  if (nan_flags) CK(cudaMemsetAsync(nan_flags, 0, B * sizeof(int32_t), st));
  const int n = B * N, xd = 3 + e->cfg.in_node_nf;
  // frames that no reverse step is the last writer of stay zero, as torch.zeros in edm.py:143
  CK(cudaMemsetAsync(chain, 0, (size_t)keep_frames * n * xd * sizeof(float), st));
  if (inpaint) {
    // z_T = COM-free masked noise on every atom (edm.py:565); the caller's slab 0 is already masked and projected
    CK(cudaMemcpyAsync(e->ws.z, noise, (size_t)n * xd * sizeof(float), cudaMemcpyDeviceToDevice, st));
  } else {
    k_init_z<<<(n * xd + 255) / 256, 256, 0, st>>>(n, xd, xh, fragment_mask, linker_mask, noise, rng ? *rng : NoiseRng{}, e->ws.z);
    LAUNCH_CHECK();
    e->launches += 1;
  }
  // inpainting: the dynamics see linker_mask=None (edm.py:632), so every live row gets a coordinate update
  if ((s = build_plan(e, B, N, node_mask, inpaint ? nullptr : linker_mask, edge_mask, st)) != DL_OK) return s;

  if (time_chain) { cudaStreamSynchronize(st); tc_plan = now_ms(); }
  FwdIO io;
  io.sampler = true; io.inpaint = inpaint; io.xh0 = xh; io.upd_linker_mask = linker_mask;
  io.node_mask = node_mask; io.linker_mask = inpaint ? nullptr : linker_mask; io.edge_mask = edge_mask;
  io.context = context; io.nan_flags = nan_flags; io.fragment_mask = fragment_mask; io.noise = noise;
  if (rng) io.rng = *rng;
  io.chain = chain; io.T = T; io.norm0 = norm[0]; io.norm1 = norm[1]; io.bias1 = norm[2];

  // capture ONE reverse step; the step index lives on the device, so the same graph serves all T+1 steps
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  const int64_t before = e->launches;
  CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  s = enqueue_forward(e, B, N, io, st);
  cudaError_t ce = cudaStreamEndCapture(st, &graph);
  if (s != DL_OK) { if (graph) cudaGraphDestroy(graph); return s; }
  if (ce != cudaSuccess) { set_err("cudaStreamEndCapture -> %s", cudaGetErrorString(ce)); return DL_ERR_CUDA; }
  const int64_t per_step = e->launches - before;
  // every exit below releases the captured graph and its executable (destruction is deferred by the runtime until the
  // launched work has finished)
  if (time_chain) tc_capture = now_ms();
  cudaError_t ge = cudaGraphInstantiate(&exec, graph, 0);
  if (time_chain) tc_inst = now_ms();
  if (ge == cudaSuccess) ge = cudaEventRecord(e->ev_t0, st);
  int failed_step = -1;
  for (int r = 0; ge == cudaSuccess && r <= T; ++r) {
    ge = cudaGraphLaunch(exec, st);
    if (ge != cudaSuccess) failed_step = r;
  }
  if (ge == cudaSuccess) ge = cudaEventRecord(e->ev_t1, st);
  if (time_chain) {
    tc_launch = now_ms();
    cudaStreamSynchronize(st);
    const double tc_done = now_ms();
    float loop = 0.f; cudaEventElapsedTime(&loop, e->ev_t0, e->ev_t1);
    fprintf(stderr, "[dl chain] setup+plan %.2f ms | capture %.2f | instantiate %.2f | %d graph launches enqueued in %.2f | wait for the GPU %.2f | device loop %.2f\n",
            tc_plan - tc0, tc_capture - tc_plan, tc_inst - tc_capture, T + 1, tc_launch - tc_inst, tc_done - tc_launch, loop);
  }
  if (ge == cudaSuccess && user != st) {
    ge = cudaEventRecord(e->ev_out, st);
    if (ge == cudaSuccess) ge = cudaStreamWaitEvent(user, e->ev_out, 0);
  }
  if (exec) cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  if (ge != cudaSuccess) {
    if (failed_step >= 0) set_err("cudaGraphLaunch step %d -> %s", failed_step, cudaGetErrorString(ge));
    else set_err("%s:%d reverse-loop graph -> %s", __FILE__, __LINE__, cudaGetErrorString(ge));
    return DL_ERR_CUDA;
  }
  e->launches = before + per_step * (T + 1);
  return DL_OK;
}

dl_status dl_sample_chain_host(dl_engine* e, int32_t sampler, int32_t B, int32_t N, int32_t T, int32_t keep_frames,
                               const float* xh, const int8_t* node_mask, const float* fragment_mask,
                               const float* linker_mask, const int8_t* edge_mask, const float* context,
                               const float* noise, const dl_step_coef* coef, const float* norm, float* chain,
                               int32_t* nan_flags) {
  dl_status s = check_shapes(e, B, N);
  if (s != DL_OK) return s;
  if (!xh || !node_mask || !fragment_mask || !linker_mask || !noise || !coef || !norm || !chain) {
    set_err("null argument"); return DL_ERR_INVALID;
  }
  if (T < 1 || keep_frames < 1 || keep_frames > T) { set_err("need 1 <= keep_frames <= T"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  const size_t n = (size_t)B * N;
  const int xd = 3 + e->cfg.in_node_nf, C = e->cfg.context_node_nf;
  const bool has_em = edge_mask && e->cfg.graph_type == DL_GRAPH_FC;
  const size_t n_slabs = sampler == DL_SAMPLER_INPAINT ? (size_t)2 * T + 3 : (size_t)T + 2;
  const size_t o_xh = 0, o_nm = o_xh + align256(n * xd * 4), o_fm = o_nm + align256(n), o_lm = o_fm + align256(n * 4),
               o_em = o_lm + align256(n * 4), o_ctx = o_em + align256(has_em ? n * N : 1),
               o_nz = o_ctx + align256(n * std::max(C, 1) * 4), o_ch = o_nz + align256((size_t)n_slabs * n * xd * 4),
               o_fl = o_ch + align256((size_t)keep_frames * n * xd * 4), total = o_fl + align256(B * 4);
  if ((s = stage_reserve(e, total)) != DL_OK) return s;
  char* d = e->stage.buf;
  cudaStream_t st = e->loop_stream;
  CK(cudaMemcpyAsync(d + o_xh, xh, n * xd * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_nm, node_mask, n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_fm, fragment_mask, n * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_lm, linker_mask, n * 4, cudaMemcpyHostToDevice, st));
  if (has_em) CK(cudaMemcpyAsync(d + o_em, edge_mask, n * N, cudaMemcpyHostToDevice, st));
  if (context) CK(cudaMemcpyAsync(d + o_ctx, context, n * C * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d + o_nz, noise, n_slabs * n * xd * 4, cudaMemcpyHostToDevice, st));
  s = dl_sample_chain(e, sampler, B, N, T, keep_frames, (const float*)(d + o_xh), (const int8_t*)(d + o_nm),
                      (const float*)(d + o_fm), (const float*)(d + o_lm), has_em ? (const int8_t*)(d + o_em) : nullptr,
                      context ? (const float*)(d + o_ctx) : nullptr, (const float*)(d + o_nz), coef, norm,
                      (float*)(d + o_ch), (int32_t*)(d + o_fl), st);
  if (s != DL_OK) return s;
  std::vector<int32_t> flags(B);
  CK(cudaMemcpyAsync(chain, d + o_ch, (size_t)keep_frames * n * xd * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(flags.data(), d + o_fl, B * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  bool any = false;
  for (int i = 0; i < B; ++i) { any |= flags[i] != 0; if (nan_flags) nan_flags[i] = flags[i]; }
  return any ? DL_NAN_DETECTED : DL_OK;
}

int64_t dl_launch_count(const dl_engine* e) { return e ? e->launches : 0; }

float dl_last_elapsed_ms(dl_engine* e) {
  if (!e) return -1.f;
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, e->ev_t0, e->ev_t1) != cudaSuccess) { cudaGetLastError(); return -1.f; }
  return ms;
}

dl_status dl_cut_graph_stats(dl_engine* e, int64_t* out) {
  if (!e || !out) return DL_ERR_INVALID;
  Workspace& ws = e->ws;
  out[0] = out[1] = out[2] = out[3] = 0;
  if (ws.recs == nullptr) return DL_OK;
  if (cudaSetDevice(e->cfg.device) != cudaSuccess) return DL_ERR_CUDA;
  CK(cudaDeviceSynchronize());
  int n[2] = {0, 0};
  CK(cudaMemcpy(n, ws.n_recs, sizeof(n), cudaMemcpyDeviceToHost));
  std::vector<int> recs((size_t)n[0] * CUT_REC);
  CK(cudaMemcpy(recs.data(), ws.recs, recs.size() * sizeof(int), cudaMemcpyDeviceToHost));
  out[0] = n[0]; out[3] = n[1];
  long long n_heavy = 0, e_heavy = 0, max_heavy = 0, rows_light = 0;
  for (int k = 0; k < n[0]; ++k) {
    const int* r = recs.data() + (size_t)k * CUT_REC;
    const bool heavy = (r[1] >> 8) & 1;
    out[1] += heavy ? (r[2] + tc::TN - 1) / tc::TN : 1;
    out[2] += r[2];
    if (heavy) { ++n_heavy; e_heavy += r[2]; max_heavy = std::max<long long>(max_heavy, r[2]); }
    else rows_light += r[1] & 0xff;
  }
  if (getenv("DL_DEBUG_CUT"))
    fprintf(stderr, "[dl cut] records %d (heavy %lld, deg sum %lld, max %lld; light rows %lld) tiles %lld edges %lld | coord records %d\n",
            n[0], n_heavy, e_heavy, max_heavy, rows_light, (long long)out[1], (long long)out[2], n[1]);
  return DL_OK;
}

float dl_time_edge_kernel(dl_engine* e, int32_t reps) {
  if (!e || !e->finalized || e->last_B == 0 || reps < 1) { set_err("dl_time_edge_kernel: no previous forward"); return -1.f; }
  if (cudaSetDevice(e->cfg.device) != cudaSuccess) return -1.f;
  Workspace& ws = e->ws;
  const Geom gm = make_geom(e, e->last_B, e->last_N);
  const GclW& w = e->gcl[0];
  EdgeArgs ea{};
  const float ksc = e->use_tc ? 1.4426950408889634f : 1.0f;
  ea.AB = ws.ABg; ea.ABmax = ws.ABgmax; ea.w2_descale = w.w2_descale; ea.wdmax = w.wdmax * ksc; ea.w0max = w.w0max * ksc;
  ea.x = ws.xa; ea.x0 = ws.x0; ea.x4 = ws.xa4; ea.x04 = ws.x04; ea.x4_out = nullptr; ea.edge_mask = e->last_edge_mask; ea.cls = ws.cls; ea.nm = ws.nm;
  ea.linker_mask = e->last_linker_mask; ea.W2_t = w.W2_t; ea.b2 = w.b2; ea.wd = e->use_tc ? w.wd_u : w.wd; ea.w0 = e->use_tc ? w.w0_u : w.w0; ea.w5 = nullptr;
  ea.plan = make_plan(ws); ea.agg = ws.agg; ea.x_out = nullptr; ea.nbr = ws.nbr; ea.recs = ws.recs; ea.n_recs = ws.n_recs;
  cudaStream_t st = e->loop_stream;
  if (e->use_tc && getenv("DL_PROFILE_EDGE")) {
    if (ws.v3) tc3::profile_edge_v3(gm, ea, w.W2_v3, ws.tm_abg, make_tile_tables(ws, false), e->num_sms, st, false);
    else tc::profile_edge_tc(gm, ea, w.W2_tc, e->num_sms, st);
  }
  if (e->use_tc && getenv("DL_PROFILE_NODE")) {
    for (int np = 1; np <= (e->cfg.n_layers > 1 ? 2 : 1); ++np) {
      tcn::NodeTcArgs ta{};
      ta.h = ws.h; ta.agg = ws.agg; ta.nm = ws.nm;
      ta.w3 = reinterpret_cast<const __half*>(w.W3_tc); ta.w4 = reinterpret_cast<const __half*>(w.W4_tc);
      ta.b3 = w.b3; ta.b4 = w.b4; ta.w3_descale = w.w3_descale; ta.w4_descale = w.w4_descale;
      const EqW& q = e->eq[0];
      ta.n_proj = np; ta.pw[0] = reinterpret_cast<const __half*>(q.W1_tc); ta.pb1[0] = q.b1_u;
      ta.p_descale[0] = q.w1_descale; ta.AB[0] = ws.ABc; ta.ABmax[0] = ws.ABcmax;
      const GclW& nx = e->gcl[e->cfg.n_layers > 1 ? e->cfg.inv_sublayers : 0];
      ta.pw[1] = reinterpret_cast<const __half*>(nx.W1_tc); ta.pb1[1] = nx.b1_u;
      ta.p_descale[1] = nx.w1_descale; ta.AB[1] = ws.ABg; ta.ABmax[1] = ws.ABgmax;
      tcn::profile_node(e->last_B * e->last_N, ta, st);
    }
  }
  for (int i = 0; i < 2; ++i) if (launch_edge(e, gm, ea, false, w.W2_tc, st, w.W2_v3) != DL_OK) return -1.f;
  if (cudaEventRecord(e->ev_t0, st) != cudaSuccess) return -1.f;
  for (int i = 0; i < reps; ++i) if (launch_edge(e, gm, ea, false, w.W2_tc, st, w.W2_v3) != DL_OK) return -1.f;
  if (cudaEventRecord(e->ev_t1, st) != cudaSuccess) return -1.f;
  if (cudaStreamSynchronize(st) != cudaSuccess) { set_err("dl_time_edge_kernel: %s", cudaGetErrorString(cudaGetLastError())); return -1.f; }
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, e->ev_t0, e->ev_t1) != cudaSuccess) return -1.f;
  return ms / reps;
}

dl_status dl_selftest_tc(dl_engine* e, float* max_abs_err, float* max_rel_err) {
  if (!e) { set_err("null engine"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  return tc::selftest(e->num_sms, max_abs_err, max_rel_err, false);
}

dl_status dl_selftest_tc_layout(dl_engine* e, int32_t b_mn_major, float* max_abs_err, float* max_rel_err) {
  if (!e) { set_err("null engine"); return DL_ERR_INVALID; }
  CK(cudaSetDevice(e->cfg.device));
  if (b_mn_major == 2) return tc3::selftest_ts(max_abs_err, max_rel_err);   // A operand in tensor memory (k_edge_v3)
  return tc::selftest(e->num_sms, max_abs_err, max_rel_err, b_mn_major != 0);
}

}  // extern "C"

#include "size_gnn.cuh"
